"""PnP-ADMM convergence history on the GPU (PnP_ADMM.m:106-109): PnP_ADMM(..., history=True), AdmmSession.monitor / history and
the C entry points qmri_admm_monitor / qmri_admm_history, against the float64 oracle, against norms of the downloaded iterates, and
for bit-identical results with and without monitoring and with and without the CUDA graph."""
import ctypes

import numpy as np
import pytest

from test_monitor_oracle import oracle_history

pytestmark = pytest.mark.gpu

TOL_ORACLE = 1e-4


@pytest.fixture(scope="module")
def q():
    import qmri_b200
    qmri_b200.Context.default()  # raises without a B200: no fallback
    return qmri_b200


def box_denoiser(v):
    """The 5-point average of tests/test_gpu_parity.py: a cheap deterministic stand-in for param.net."""
    v = np.asarray(v, dtype=np.float64)[:, :, :10]
    return (v + np.roll(v, 1, 0) + np.roll(v, -1, 0) + np.roll(v, 1, 1) + np.roll(v, -1, 1)) / 5.0


def tsmi(N, seed, S=None, C=10):
    rng = np.random.default_rng(seed)
    shape = (N, N, C) + (() if S is None else (S,))
    n = np.arange(N)[:, None, None] / N
    m = np.arange(N)[None, :, None] / N
    c = np.arange(C)[None, None, :]
    base = np.exp(-((n - 0.5) ** 2 + (m - 0.45) ** 2) * 8) * np.cos(0.3 * c) + 0.2 * np.sin(7 * n + c) * np.cos(5 * m)
    x = base if S is None else np.repeat(base[..., None], S, axis=3)
    return x + 0.05 * rng.standard_normal(shape)


def make(q, kind, N, seed, S=None, V=None):
    from oracle import sampling
    from oracle.sampling import FOperator
    from oracle.synth import awgn_measured
    V = np.eye(10) if V is None else V
    if kind == "spiral":
        P, Po = q.setup_subsampling_spiralgrided(N, N, 771, V), sampling.setup_subsampling_spiralgrided(N, N, 771, V)
    else:
        P, Po = q.setup_subsampling_epi(N, N, 1 / 65, V), sampling.setup_subsampling_epi(N, N, 1 / 65, V)
    Fo = FOperator(Po)
    Xgt = tsmi(N, seed, S=S, C=V.shape[1])
    Y = awgn_measured(Fo.forward(Xgt), 30, seed)
    X0 = Fo.adjoint(Y)
    X0 = X0 + 0.02 * np.random.default_rng(seed + 1).standard_normal(X0.shape)  # k = 1 then has a residual to report
    return P, Fo, Xgt, Y, X0


def host_norms(Fo, Y, Xgt, x, S):
    """float64 |y - A x| / |y| and |gt - x| / |gt| per slice of a downloaded iterate."""
    Y = Y.reshape(-1, S, order="F")
    dc = np.array([np.linalg.norm(Y[:, s] - Fo.forward(x[..., s])) / np.linalg.norm(Y[:, s]) for s in range(S)])
    ge = np.array([np.linalg.norm((Xgt[..., s] - x[..., s]).ravel()) / np.linalg.norm(Xgt[..., s].ravel()) for s in range(S)])
    return dc, ge


# ---- 3. against the oracle --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,N,S", [("spiral", 224, 1), ("spiral", 224, 3), ("epi", 224, 1), ("epi", 224, 3), ("spiral", 256, 2)])
def test_history_matches_oracle(q, kind, N, S):
    P, Fo, Xgt, Y, X0 = make(q, kind, N, 31, S=None if S == 1 else S)
    param = {"iter": 6, "gamma": 0.05, "X0": X0, "gt_tsmi": Xgt, "denoiser_type": "single_level"}
    x, info = q.PnP_ADMM(Y, dict(param, F=q.fft_operator(P), net=box_denoiser), history=True)
    dc, ge = info["dc_residual"], info["gt_error"]
    assert dc.shape == ge.shape == ((6,) if S == 1 else (6, S))
    assert dc.dtype == ge.dtype == np.float64
    dc, ge = dc.reshape(6, S), ge.reshape(6, S)
    for s in range(S):
        sl = (lambda a: a) if S == 1 else (lambda a: a[..., s])
        ys = Y if S == 1 else Y[:, s]
        _, dco, geo = oracle_history(ys, dict(param, F=Fo, net=box_denoiser, X0=sl(X0), gt_tsmi=sl(Xgt)))
        assert np.max(np.abs(dc[:, s] - dco)) <= TOL_ORACLE
        assert np.max(np.abs(ge[:, s] - geo)) <= TOL_ORACLE
    # history=False is the plain call: same x, gt_tsmi ignored
    x_plain = q.PnP_ADMM(Y, dict(param, F=q.fft_operator(P), net=box_denoiser))
    assert x_plain.shape == x.shape


def general_V(L=12, C=10):
    return np.random.default_rng(3).standard_normal((L, C)) / np.sqrt(C)


@pytest.mark.parametrize("S", [1, 2])
def test_history_matches_oracle_general_V(q, S):
    """General V (12 x 10 spiral): the residual comes from the per-location solve, the ground-truth error from the adjoint pass
    that completes x."""
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 41, S=None if S == 1 else S, V=general_V())
    param = {"iter": 6, "gamma": 0.05, "X0": X0, "gt_tsmi": Xgt, "denoiser_type": "single_level"}
    x, info = q.PnP_ADMM(Y, dict(param, F=q.fft_operator(P), net=box_denoiser), history=True)
    dc, ge = info["dc_residual"].reshape(6, S), info["gt_error"].reshape(6, S)
    for s in range(S):
        sl = (lambda a: a) if S == 1 else (lambda a: a[..., s])
        ys = Y if S == 1 else Y[:, s]
        _, dco, geo = oracle_history(ys, dict(param, F=Fo, net=box_denoiser, X0=sl(X0), gt_tsmi=sl(Xgt)))
        assert np.max(np.abs(dc[:, s] - dco)) <= TOL_ORACLE
        assert np.max(np.abs(ge[:, s] - geo)) <= TOL_ORACLE


# ---- 4. self-consistency of the device reductions -----------------------------------------------------------------------------
@pytest.mark.parametrize("N,S", [(224, 3), (256, 2)])
def test_history_rows_equal_norms_of_the_iterates(q, N, S):
    P, Fo, Xgt, Y, X0 = make(q, "spiral", N, 32, S=S)
    K = 5
    sess = q.AdmmSession({"iter": K, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0}, S)
    sess.monitor(Xgt)
    sess.upload(Y, X0)
    sess.run(K)
    h = sess.history()
    assert h["dc_residual"].shape == (K, S)
    for k in (1, 2, K):
        sess.run(k)
        xk = sess.download()
        dc, ge = host_norms(Fo, Y, Xgt, xk, S)
        assert np.all(np.abs(h["dc_residual"][k - 1] - dc) <= 1e-6 + 1e-5 * dc)
        assert np.all(np.abs(h["gt_error"][k - 1] - ge) <= 1e-6 + 1e-5 * ge)
        hk = sess.history()  # the k-iteration run's own history is the first k rows
        assert np.array_equal(hk["dc_residual"], h["dc_residual"][:k])
        assert np.array_equal(hk["gt_error"], h["gt_error"][:k])
    sess.close()


# ---- 5. monitoring does not change x ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,S", [(224, 3), (256, 2), (224, 1)])
def test_monitoring_leaves_x_bit_identical(q, N, S, monkeypatch):
    if S == 1:
        monkeypatch.setenv("QMRI_K1_KERNEL", "stream")  # a monitored single slice runs the streaming kernels
    P, Fo, Xgt, Y, X0 = make(q, "spiral", N, 33, S=None if S == 1 else S)
    param = {"iter": 5, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0, "gt_tsmi": Xgt}
    x_plain = q.PnP_ADMM(Y, param)
    x_res, info_res = q.PnP_ADMM(Y, {k: v for k, v in param.items() if k != "gt_tsmi"}, history=True)
    x_gt, info_gt = q.PnP_ADMM(Y, param, history=True)
    assert np.array_equal(x_plain, x_res) and np.array_equal(x_plain, x_gt)
    assert info_res["gt_error"] is None
    assert np.array_equal(info_res["dc_residual"], info_gt["dc_residual"])


@pytest.mark.parametrize("L,S", [(12, 2), (200, 1)])
def test_monitoring_leaves_x_bit_identical_general_V(q, L, S):
    """General V with 12 and 200 frames: the union of the masks is processed in parts, x of the last iteration is completed by
    the in-place correction passes, and a monitored session writes and checks x on every iteration."""
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 42, S=None if S == 1 else S, V=general_V(L))
    param = {"iter": 4, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0, "gt_tsmi": Xgt}
    x_plain = q.PnP_ADMM(Y, param)
    x_res, info_res = q.PnP_ADMM(Y, {k: v for k, v in param.items() if k != "gt_tsmi"}, history=True)
    x_gt, info_gt = q.PnP_ADMM(Y, param, history=True)
    assert np.array_equal(x_plain, x_res) and np.array_equal(x_plain, x_gt)
    assert np.array_equal(info_res["dc_residual"], info_gt["dc_residual"])
    # the last row is the norm of the returned x
    xs = x_gt if S > 1 else x_gt[..., None]
    dc, ge = host_norms(Fo, Y, Xgt if S > 1 else Xgt[..., None], xs, S)
    assert np.all(np.abs(info_gt["dc_residual"].reshape(4, S)[-1] - dc) <= 1e-6 + 1e-5 * dc)
    assert np.all(np.abs(info_gt["gt_error"].reshape(4, S)[-1] - ge) <= 1e-6 + 1e-5 * ge)


def test_single_slice_224_monitored_runs_streaming_kernels(q):
    """At one slice the default x-update kernel is the cluster kernel; a monitored run takes the streaming kernels and still
    matches the unmonitored result to the x-update tolerance."""
    from conftest import rel_l2
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 34)
    param = {"iter": 4, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0, "gt_tsmi": Xgt}
    x_plain = q.PnP_ADMM(Y, param)
    x_mon, info = q.PnP_ADMM(Y, param, history=True)
    assert rel_l2(x_mon, x_plain) <= 1e-5
    assert info["dc_residual"].shape == (4,)


# ---- 6. CUDA-graph replay ----------------------------------------------------------------------------------------------------
def test_history_graph_replay_equals_direct_launches_and_recapture(q, monkeypatch):
    from oracle import unetres
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 35, S=2)
    net = q.UNetRes(unetres.make_state_dict(10, seed=0), in_nc=10)
    param = {"iter": 8, "gamma": 0.05, "X0": X0, "denoiser_type": "single_level", "F": q.fft_operator(P), "net": net,
             "gt_tsmi": Xgt}
    ctx = q.Context.default()
    l0 = ctx.launch_count
    x_graph, h_graph = q.PnP_ADMM(Y, param, history=True)
    n_graph = ctx.launch_count - l0
    monkeypatch.setenv("QMRI_NO_GRAPH", "1")
    l0 = ctx.launch_count
    x_direct, h_direct = q.PnP_ADMM(Y, param, history=True)
    n_direct = ctx.launch_count - l0
    monkeypatch.delenv("QMRI_NO_GRAPH")
    assert np.array_equal(x_graph, x_direct)
    assert np.array_equal(h_graph["dc_residual"], h_direct["dc_residual"])
    assert np.array_equal(h_graph["gt_error"], h_direct["gt_error"])
    assert n_graph == n_direct
    assert np.all(np.isfinite(h_graph["dc_residual"])) and np.all(np.isfinite(h_graph["gt_error"]))

    # monitored -> unmonitored -> monitored in one session: the graph is re-captured each time
    x_plain = q.PnP_ADMM(Y, param)
    sess = q.AdmmSession(param, 2)
    sess.upload(Y, X0)
    sess.monitor(Xgt)
    sess.run(8)
    ha = sess.history()
    xa = sess.download()
    sess.monitor(enable=False)
    sess.run(8)
    assert sess.history()["dc_residual"].shape == (0, 2)
    xb = sess.download()
    sess.monitor(None)  # residual only
    sess.run(8)
    hc = sess.history()
    xc = sess.download()
    sess.monitor(Xgt)
    sess.run(8)
    hd = sess.history()
    sess.close()
    for x in (xa, xb, xc):
        assert np.array_equal(x, x_plain)
    assert np.array_equal(ha["dc_residual"], h_graph["dc_residual"]) and np.array_equal(ha["gt_error"], h_graph["gt_error"])
    assert np.array_equal(hc["dc_residual"], h_graph["dc_residual"]) and hc["gt_error"] is None
    assert np.array_equal(hd["dc_residual"], h_graph["dc_residual"]) and np.array_equal(hd["gt_error"], h_graph["gt_error"])


def test_history_when_iters_change_between_graph_runs(q):
    """A monitored session run for 8, then 20, then 8 iterations: the graph's history row limit follows, each history equals
    a fresh session's."""
    from oracle import unetres
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 43, S=2)
    net = q.UNetRes(unetres.make_state_dict(10, seed=0), in_nc=10)
    param = {"iter": 8, "gamma": 0.05, "X0": X0, "denoiser_type": "single_level", "F": q.fft_operator(P), "net": net}

    def fresh(k):
        f = q.AdmmSession(param, 2)
        f.monitor(Xgt)
        f.upload(Y, X0)
        f.run(k)
        h = f.history()
        f.close()
        return h
    sess = q.AdmmSession(param, 2)
    sess.monitor(Xgt)
    sess.upload(Y, X0)
    for k in (8, 20, 8):
        sess.run(k)
        h, hf = sess.history(), fresh(k)
        assert h["dc_residual"].shape == (k, 2)
        assert np.array_equal(h["dc_residual"], hf["dc_residual"]) and np.array_equal(h["gt_error"], hf["gt_error"])
    sess.close()


# ---- 7. edge cases ---------------------------------------------------------------------------------------------------------------
def test_real_state_sessions_run_the_complex_loop_when_monitored(q, monkeypatch):
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 36, S=2)
    param = {"iter": 5, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0, "gt_tsmi": Xgt}
    xc, hc = q.PnP_ADMM(Y, param, history=True)
    monkeypatch.setenv("QMRI_K1_STATE", "real")
    xr, hr = q.PnP_ADMM(Y, param, history=True)
    assert np.array_equal(xc, xr)
    assert np.array_equal(hc["dc_residual"], hr["dc_residual"]) and np.array_equal(hc["gt_error"], hr["gt_error"])


def test_cluster_kernel_with_monitor_is_unsupported(q, monkeypatch):
    monkeypatch.setenv("QMRI_K1_KERNEL", "cluster")
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 37)
    with pytest.raises(q.QmriError, match="cluster") as e:
        q.PnP_ADMM(Y, {"iter": 2, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0}, history=True)
    assert e.value.code == q._capi.QMRI_EUNSUPPORTED


def test_monitor_argument_errors_and_zero_iterations(q):
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 39, S=2)
    sess = q.AdmmSession({"iter": 3, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0}, 2)
    with pytest.raises(q.QmriError) as e:
        sess.monitor(Xgt[:, :, :9])
    assert e.value.code == q._capi.QMRI_EINVAL
    with pytest.raises(q.QmriError) as e:
        sess.monitor(Xgt[..., 0])  # one slice of ground truth for a two-slice session
    assert e.value.code == q._capi.QMRI_EINVAL
    sess.upload(Y, X0)
    sess.monitor(None)
    sess.run(3)
    n = ctypes.c_int()
    dc = np.zeros((3, 2), order="F")
    ge = np.zeros((3, 2), order="F")
    assert sess.lib.qmri_admm_history(sess.handle, q._capi.ptr(dc), q._capi.ptr(ge), ctypes.byref(n)) == q._capi.QMRI_EINVAL
    assert sess.lib.qmri_admm_history(sess.handle, q._capi.ptr(dc), None, ctypes.byref(n)) == 0 and n.value == 3
    assert np.array_equal(dc, sess.history()["dc_residual"])
    sess.run(0)
    assert sess.lib.qmri_admm_history(sess.handle, q._capi.ptr(dc), q._capi.ptr(ge), ctypes.byref(n)) == q._capi.QMRI_EINVAL
    sess.monitor(Xgt.astype(np.complex64))  # complex ground truth, another dtype
    sess.run(0)
    h = sess.history()
    assert h["dc_residual"].shape == (0, 2) and h["gt_error"].shape == (0, 2)
    sess.run(2)
    h = sess.history()
    assert h["gt_error"].shape == (2, 2) and np.all(np.isfinite(h["gt_error"]))
    sess.close()
    x, info = q.PnP_ADMM(Y, {"iter": 0, "gamma": 0.05, "F": q.fft_operator(P), "net": box_denoiser, "X0": X0}, history=True)
    assert info["dc_residual"].shape == (0, 2) and info["gt_error"] is None


# ---- 8. the MEX gateway ---------------------------------------------------------------------------------------------------------
def mex_pnp_admm_with_info(m, *args):
    """[x, info] = qmri_b200_mex('pnp_admm', ...) through the MEX mock: x and the fields of the info struct."""
    L = m.lib
    L.mxGetField.restype = ctypes.c_void_p
    L.mxGetField.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p]
    prhs = [m.to_mx("pnp_admm")] + [m.to_mx(a) for a in args]
    rhs = (ctypes.c_void_p * len(prhs))(*prhs)
    lhs = (ctypes.c_void_p * 4)()
    rc = L.mock_call_mex(2, lhs, len(prhs), rhs)
    try:
        assert rc == 0, L.mock_last_error().decode()
        x = m.from_mx(lhs[0])
        info = {f: m.from_mx(L.mxGetField(lhs[1], 0, f.encode())) for f in ("dc_res", "gt_err")}
    finally:
        for p in prhs:
            L.mxDestroyArray(p)
        for i in range(2):
            if lhs[i]:
                L.mxDestroyArray(lhs[i])
    return x, info


@pytest.mark.parametrize("split", [False, True])
def test_mex_gateway_returns_the_history(q, split):
    from mexmock import FunctionHandle, MexMock
    m = MexMock(split)
    V = np.eye(10)
    h = m.call("op_spiral", 224, 224, 771, V)
    P, Fo, Xgt, Y, X0 = make(q, "spiral", 224, 44, S=2)
    prm = {"iter": 4, "gamma": 0.05, "cg_tol": 1e-4, "X0": X0, "denoiser_type": "single_level"}
    xq, iq = q.PnP_ADMM(Y, dict(prm, F=q.fft_operator(P), net=box_denoiser, gt_tsmi=Xgt), history=True)
    xm, im = mex_pnp_admm_with_info(m, h, Y, dict(prm, net=FunctionHandle(box_denoiser), gt_tsmi=Xgt))
    assert np.array_equal(xm, xq)
    assert im["dc_res"].shape == (4, 2) and np.array_equal(im["dc_res"], iq["dc_residual"])
    assert np.array_equal(im["gt_err"], iq["gt_error"])
    xm, im = mex_pnp_admm_with_info(m, h, Y, dict(prm, net=FunctionHandle(box_denoiser)))  # no ground truth: gt_err = []
    assert np.array_equal(xm, xq) and np.array_equal(im["dc_res"], iq["dc_residual"]) and im["gt_err"].size == 0
    assert np.array_equal(m.call("pnp_admm", h, Y, dict(prm, net=FunctionHandle(box_denoiser))), xq)  # nargout 1: as before
