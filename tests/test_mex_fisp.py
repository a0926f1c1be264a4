"""The MEX commands fisp_signals / fisp_gram / fisp_compress, and the steps of matlab/qmri_fisp_dictionary.m, driven through the
gateway compiled against the MEX mock: bit-identical to the ctypes path."""
import numpy as np
import pytest

from test_gpu_fisp import grid_lut
from test_oracle_epg import schedule

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("ti", [None, 0.02])
def test_mex_fisp_commands_match_ctypes(split, ti):
    import qmri_b200 as q
    from mexmock import MexMock
    q.Context.default()
    m = MexMock(split)
    lut = grid_lut()
    seq = dict(schedule(200, seed=8), ti=ti)
    mseq = {"flip_deg": seq["flip_deg"], "tr": seq["tr"], "te": seq["te"], "ti": np.zeros((0, 0)) if ti is None else ti}
    try:
        sig = m.call("fisp_signals", lut, mseq)
        assert sig.dtype == np.float32 and np.array_equal(sig, q.fisp_signals(lut, seq))
        # qmri_fisp_dictionary.m: G = fisp_gram; [U, L] = eig((G + G') / 2); descending order; sign rule; fisp_compress
        G = m.call("fisp_gram", lut, mseq)
        assert np.array_equal(G, q.fisp_gram(lut, seq)) and np.array_equal((G + G.T) / 2, G)
        V = q.temporal_basis(G, 10)
        D, normD = m.call("fisp_compress", lut, mseq, V, nlhs=2)
        ref = q.fisp_dictionary(lut, seq, V=V)
        assert np.array_equal(D, ref["D"]) and np.array_equal(normD.reshape(-1), ref["normD"])
        Ds, nds = m.call("fisp_compress", lut, mseq, V, 3.0, 20.0, nlhs=2)      # 0-based atom range [3, 20)
        assert np.array_equal(Ds, ref["D"][3:20]) and np.array_equal(nds.reshape(-1), ref["normD"][3:20])
    finally:
        m.call("shutdown", nlhs=0)
