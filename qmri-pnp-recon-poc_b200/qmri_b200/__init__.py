"""qmri_b200 - host-side mirror of the reference's MATLAB operator surface over libqmri_b200.so.

Same names, argument meaning and error behaviour as ketanfatania/QMRI-PnP-Recon-POC for the
PnP-ADMM MRF reconstruction hot path; all arithmetic runs in hand-written sm_100a CUDA kernels
behind the C ABI of include/qmri.h.  There is no CPU fallback: a missing library or a missing
B200 raises.
"""
from ._capi import (QMRI_C128, QMRI_C64, QMRI_DEVICE, QMRI_F32, QMRI_F64, QMRI_HOST, Context, QmriError,
                    load_library)
from .admm import AdmmSession, PnP_ADMM
from .dictionary import fisp_dictionary, fisp_gram, fisp_signals, temporal_basis
from .denoiser import UNetRes, build_noise_map, denoiseImage_PnP_ADMM, load_checkpoint_state_dict, state_dict_keys
from .matching import Dictionary, mrf_dtm, mrf_dtm_cpu, synthesize_tsmis
from .sharding import allreduce_keys, atom_shard, mrf_dtm_sharded, pack_keys, slice_shard, unpack_keys
from .lrtv import FISTA_deep
from .metrics import getmask_fromPD, recon_metrics
from .onnx_import import load_onnx_state_dict, read_initializers
from .operators import (FOperator, SubsamplingPattern, awgn, fft_operator, setup_subsampling_epi,
                        setup_subsampling_explicit, setup_subsampling_spiralgrided)

__all__ = [
    "Context", "QmriError", "load_library", "PnP_ADMM", "AdmmSession", "UNetRes", "build_noise_map",
    "denoiseImage_PnP_ADMM", "state_dict_keys", "fisp_signals", "fisp_gram", "fisp_dictionary", "temporal_basis", "Dictionary", "mrf_dtm", "mrf_dtm_cpu", "synthesize_tsmis", "FOperator",
    "SubsamplingPattern", "fft_operator", "setup_subsampling_epi", "setup_subsampling_explicit",
    "setup_subsampling_spiralgrided", "slice_shard", "atom_shard", "pack_keys", "unpack_keys", "allreduce_keys",
    "mrf_dtm_sharded", "awgn", "FISTA_deep", "load_onnx_state_dict", "read_initializers", "load_checkpoint_state_dict", "getmask_fromPD", "recon_metrics", "QMRI_F32", "QMRI_F64", "QMRI_C64", "QMRI_C128", "QMRI_HOST", "QMRI_DEVICE",
]
