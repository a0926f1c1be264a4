"""ctypes binding of libqmri_b200.so (include/qmri.h).

This is the only way the Python host layer reaches the GPU: there is no CPU
fallback.  Importing the package without the built library, or creating a
context on a machine without a B200, raises immediately.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libqmri_b200.so")

QMRI_F32, QMRI_F64, QMRI_C64, QMRI_C128 = 0, 1, 2, 3
QMRI_HOST, QMRI_DEVICE = 0, 1
QMRI_OK, QMRI_EINVAL, QMRI_EUNSUPPORTED, QMRI_ECUDA, QMRI_ENOMEM, QMRI_ECALLBACK = 0, -1, -2, -3, -4, -5

_DTYPES = {np.dtype(np.float32): QMRI_F32, np.dtype(np.float64): QMRI_F64,
           np.dtype(np.complex64): QMRI_C64, np.dtype(np.complex128): QMRI_C128}


class QmriError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libqmri_b200 error {code}: {msg}")
        self.code = code


DENOISE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                         C.c_int, C.c_void_p)


class LrtvParams(C.Structure):
    _fields_ = [("K", C.c_double), ("iters", C.c_int), ("step", C.c_double), ("tol", C.c_double), ("backtrack", C.c_int),
                ("tv_tol", C.c_double), ("tv_maxit", C.c_int)]


class AdmmParams(C.Structure):
    _fields_ = [("iters", C.c_int), ("gamma", C.c_double), ("cg_tol", C.c_double), ("multi_level", C.c_int),
                ("noise_map", C.c_void_p), ("net", C.c_void_p), ("fn", DENOISE_FN), ("user", C.c_void_p),
                ("fn_space", C.c_int)]


# name -> (restype, argtypes); every symbol declared in include/qmri.h
_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_pp = C.POINTER(C.c_void_p)
SIGNATURES = {
    "qmri_version": (_i, []),
    "qmri_ctx_create": (_i, [_pp, _i]),
    "qmri_ctx_destroy": (_i, [_vp]),
    "qmri_ctx_set_stream": (_i, [_vp, _vp]),
    "qmri_ctx_synchronize": (_i, [_vp]),
    "qmri_ctx_launch_count": (_i64, [_vp]),
    "qmri_last_error": (C.c_char_p, []),
    "qmri_op_spiral": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _pp]),
    "qmri_op_epi": (_i, [_vp, _i, _i, _d, _vp, _i, _i, _pp]),
    "qmri_op_create": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _pp]),
    "qmri_op_destroy": (_i, [_vp]),
    "qmri_op_nmeas": (_i64, [_vp]),
    "qmri_op_indices": (_i, [_vp, _vp, _vp]),
    "qmri_forward": (_i, [_vp, _vp, _i, _i, _vp, _i]),
    "qmri_adjoint": (_i, [_vp, _vp, _i, _i, _vp, _i]),
    "qmri_xupdate": (_i, [_vp, _d, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _i, _vp, _i, _vp]),
    "qmri_unetres_load": (_i, [_vp, _i, _vp, _i, _pp]),
    "qmri_unetres_destroy": (_i, [_vp]),
    "qmri_unetres_set_precision": (_i, [_vp, _i]),
    "qmri_unetres_forward": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "qmri_unetres_denoise": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i]),
    "qmri_unetres_forward_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i]),
    "qmri_unetres_flops": (_d, [_vp, _i, _i, _i]),
    "qmri_pnp_admm": (_i, [_vp, _vp, _i, _vp, _i, _i, C.POINTER(AdmmParams), _vp, _i]),
    "qmri_admm_create": (_i, [_vp, _i, C.POINTER(AdmmParams), _pp]),
    "qmri_admm_upload": (_i, [_vp, _vp, _i, _vp, _i]),
    "qmri_admm_run": (_i, [_vp, _i]),
    "qmri_admm_download": (_i, [_vp, _vp, _i]),
    "qmri_admm_state_dev": (_i, [_vp, _pp, _pp]),
    "qmri_admm_destroy": (_i, [_vp]),
    "qmri_admm_xupdate_only": (_i, [_vp, _i]),
    "qmri_admm_xupdate_bytes": (_i, [_vp]),
    "qmri_admm_monitor": (_i, [_vp, _i, _vp, _i]),
    "qmri_admm_history": (_i, [_vp, _vp, _vp, C.POINTER(C.c_int)]),
    "qmri_dict_load": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i64, _i64, _pp]),
    "qmri_dict_load_shard": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i64, _i64, _pp]),
    "qmri_dict_destroy": (_i, [_vp]),
    "qmri_match": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _vp]),
    "qmri_match_dev": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "qmri_match_keys_dev": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "qmri_match_finish_dev": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "qmri_synthesize": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "qmri_op_for": (_i, [_vp, _vp, _i, _vp, _i]),
    "qmri_op_adj": (_i, [_vp, _vp, _i, _vp, _i]),
    "qmri_awgn": (_i, [_vp, _vp, _i, _i64, _i, _d, C.c_uint64]),
    "qmri_awgn_dev": (_i, [_vp, _vp, _i64, _i, _d, C.c_uint64, _vp]),
    "qmri_foreground_mask": (_i, [_vp, _vp, _i, _i, _i, _d, _vp]),
    "qmri_lrtv": (_i, [_vp, _vp, _i, C.POINTER(LrtvParams), _vp, _i, C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "qmri_recon_metrics": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _i, _vp]),
}

_lib = None


def load_library():
    """Load libqmri_b200.so; raise loudly if it was not built (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C qmri-pnp-recon-poc_b200`).  qmri_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library diverge
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        raise QmriError(code, load_library().qmri_last_error().decode(errors="replace"))


def dtype_code(arr):
    try:
        return _DTYPES[arr.dtype]
    except KeyError:
        raise TypeError(f"unsupported array dtype {arr.dtype}; use float32/float64/complex64/complex128") from None


def as_f(arr, dtype=None):
    """Column-major (MATLAB) contiguous view/copy of an array."""
    a = np.asarray(arr)
    if dtype is not None:
        a = a.astype(dtype, copy=False)
    if a.dtype not in _DTYPES:
        a = a.astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    return np.asfortranarray(a)


def ptr(arr):
    return None if arr is None else arr.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA context / stream on one B200 (qmri_ctx)."""

    _default = {}

    def __init__(self, device=0):
        lib = load_library()
        h = C.c_void_p()
        check(lib.qmri_ctx_create(C.byref(h), int(device)))
        self.handle = h
        self.device = int(device)
        self.lib = lib

    @classmethod
    def default(cls, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def set_stream(self, cuda_stream):
        check(self.lib.qmri_ctx_set_stream(self.handle, C.c_void_p(cuda_stream or 0)))

    def synchronize(self):
        check(self.lib.qmri_ctx_synchronize(self.handle))

    @property
    def launch_count(self):
        return int(self.lib.qmri_ctx_launch_count(self.handle))

    def close(self):
        if self.handle:
            self.lib.qmri_ctx_destroy(self.handle)
            self.handle = None
