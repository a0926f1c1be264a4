"""256 x 256 images on the GPU: masks, F.forward / F.adjoint, P.for / P.adj, the x-update (identity and general V), the PnP-ADMM
loop (direct and CUDA-graph replay), the denoiser, matching, LRTV, foreground mask and metrics - the CUDA path (through the C ABI)
against the CPU oracle, with the tolerances of tests/test_gpu_parity.py.  Sizes other than 224 and 256 stay unsupported."""
import numpy as np
import pytest

from conftest import rel_l2

pytestmark = pytest.mark.gpu

N = 256
TOL_XUPDATE = 1e-5
TOL_DENOISER = 1e-4
NEAR_TIE = 1e-6


@pytest.fixture(scope="module")
def q():
    import qmri_b200
    qmri_b200.Context.default()  # raises without a B200: no fallback
    return qmri_b200


def make_ops(q, kind, V):
    from oracle import sampling
    if kind == "spiral":
        return q.setup_subsampling_spiralgrided(N, N, 771, V), sampling.setup_subsampling_spiralgrided(N, N, 771, V)
    return q.setup_subsampling_epi(N, N, 1 / 65, V), sampling.setup_subsampling_epi(N, N, 1 / 65, V)


@pytest.fixture(scope="module")
def ops(q):
    return {kind: make_ops(q, kind, np.eye(10)) for kind in ("spiral", "epi")}


def tsmi(seed, S=None, cplx=False, C=10):
    """Smooth, brain-like-ish random TSMI (N x N x C [x S])."""
    rng = np.random.default_rng(seed)
    shape = (N, N, C) + (() if S is None else (S,))
    n = np.arange(N)[:, None, None] / N
    m = np.arange(N)[None, :, None] / N
    c = np.arange(C)[None, None, :]
    base = np.exp(-((n - 0.5) ** 2 + (m - 0.45) ** 2) * 8) * np.cos(0.3 * c) + 0.2 * np.sin(7 * n + c) * np.cos(5 * m)
    x = base if S is None else np.repeat(base[..., None], S, axis=3)
    x = x + 0.05 * rng.standard_normal(shape)
    if cplx:
        x = x + 1j * (0.3 * np.roll(x, 5, axis=0) + 0.05 * rng.standard_normal(shape))
    return x


def make_problem(Po, seed, S=None):
    from oracle.sampling import FOperator
    from oracle.synth import awgn_measured
    Fo = FOperator(Po)
    Xgt = tsmi(seed, S=S)
    Y = awgn_measured(Fo.forward(Xgt), 30, seed)
    return Fo, Xgt, Y, Fo.adjoint(Y)


# ---- operator -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["spiral", "epi"])
def test_mask_constructors_match_oracle_256(ops, kind):
    P, Po = ops[kind]
    idx, fp = P.indices()
    assert P.nmeas == Po.nmeas
    assert np.array_equal(fp, Po.frame_ptr) and np.array_equal(idx, Po.idx)


@pytest.mark.parametrize("kind", ["spiral", "epi"])
@pytest.mark.parametrize("dtype", [np.float64, np.complex128, np.float32, np.complex64])
@pytest.mark.parametrize("S", [1, 16])
def test_forward_adjoint_256(q, ops, kind, dtype, S):
    from oracle.sampling import FOperator
    P, Po = ops[kind]
    F, Fo = q.fft_operator(P), FOperator(Po)
    x = tsmi(1, S=None if S == 1 else S, cplx=np.issubdtype(dtype, np.complexfloating)).astype(dtype)
    y = F.forward(x)
    xs = x[..., None] if S == 1 else x
    ys = y.reshape(P.nmeas, S)
    for s in range(S):
        assert rel_l2(ys[:, s], Fo.forward(xs[..., s].astype(np.complex128))) <= TOL_XUPDATE
    rng = np.random.default_rng(2)
    b = rng.standard_normal((P.nmeas, S)) + 1j * rng.standard_normal((P.nmeas, S))
    xa = F.adjoint(b if S > 1 else b[:, 0]).reshape(N, N, 10, S)
    for s in range(S):
        assert rel_l2(xa[..., s], Fo.adjoint(b[:, s])) <= TOL_XUPDATE
    lhs, rhs = np.vdot(b, ys), np.vdot(xa, xs)             # <A x, b> == <x, A^H b>
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)


@pytest.mark.parametrize("kind", ["spiral", "epi"])
def test_p_for_adj_match_the_sparse_matrix_256(q, ops, kind):
    P, Po = ops[kind]
    rng = np.random.default_rng(3)
    n = N * N * 10
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    y = rng.standard_normal(Po.nmeas) + 1j * rng.standard_normal(Po.nmeas)
    assert np.array_equal(P.for_(x), Po.for_(x)) and np.array_equal(P["adj"](y), Po.adj(y))


# ---- x-update -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["spiral", "epi"])
@pytest.mark.parametrize("S", [1, 3])
def test_xupdate_matches_exact_solve_256(q, ops, kind, S):
    from oracle.sampling import FOperator
    from oracle.xupdate import xupdate_exact
    P, Po = ops[kind]
    F, Fo = q.fft_operator(P), FOperator(Po)
    rho = 0.05
    xt, v, u = tsmi(3, S=S), tsmi(4, S=S), 0.1 * tsmi(5, S=S, cplx=True)
    y = np.stack([Fo.forward(xt[..., s]) for s in range(S)], axis=1)
    x, w, mm = F.xupdate(y, v, u, rho, want_w=True)
    x2 = F.xupdate(y, v, None, rho)                          # u omitted = the scalar 0 of PnP_ADMM.m:78
    for s in range(S):
        xo = xupdate_exact(Fo, y[:, s], v[..., s] - u[..., s], rho)
        assert rel_l2(x[..., s], xo) <= TOL_XUPDATE
        wo = xo + u[..., s]
        assert rel_l2(w[..., s], wo) <= TOL_XUPDATE
        scale = abs(wo.real).max()
        mms = np.asarray(mm).reshape(S, 2)[s] if S > 1 else np.asarray(mm).ravel()
        assert abs(mms[0] - wo.real.min()) <= 1e-5 * scale and abs(mms[1] - wo.real.max()) <= 1e-5 * scale
        assert rel_l2(x2[..., s], xupdate_exact(Fo, y[:, s], v[..., s], rho)) <= TOL_XUPDATE


@pytest.mark.parametrize("L,C", [(12, 10), (40, 4)])
def test_general_V_operator_and_xupdate_256(q, L, C):
    from oracle.sampling import FOperator
    from oracle.xupdate import xupdate_exact
    rng = np.random.default_rng(60 + L)
    V = rng.standard_normal((L, C)) / np.sqrt(C)
    P, Po = make_ops(q, "spiral", V)
    F, Fo = q.fft_operator(P), FOperator(Po)
    assert P.nmeas == Po.nmeas
    x = tsmi(61, C=C, cplx=True)
    assert rel_l2(F.forward(x), Fo.forward(x)) <= TOL_XUPDATE
    b = rng.standard_normal(P.nmeas) + 1j * rng.standard_normal(P.nmeas)
    assert rel_l2(F.adjoint(b), Fo.adjoint(b)) <= TOL_XUPDATE
    yv = Fo.forward(tsmi(62, C=C))
    v, u = tsmi(63, C=C), 0.1 * tsmi(64, C=C, cplx=True)
    xs, w, mm = F.xupdate(yv, v, u, 0.05, want_w=True)
    xo = xupdate_exact(Fo, yv, v - u, 0.05)
    assert rel_l2(xs, xo) <= TOL_XUPDATE
    assert rel_l2(w, xo + u) <= TOL_XUPDATE


# ---- denoiser and loop ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("in_nc", [10, 11])
def test_denoiser_tensor_mode_256(q, in_nc):
    import torch
    from oracle import unetres
    sd = unetres.make_state_dict(in_nc, seed=0)
    net = q.UNetRes(sd, in_nc=in_nc)
    net.set_precision("tc")
    torch.manual_seed(11)
    x = torch.rand(2, in_nc, N, N)
    with torch.no_grad():
        ref = unetres.unetres_forward(sd, x).numpy()
    out = net.forward(x.numpy())
    assert out.shape == ref.shape
    err = rel_l2(out, ref)
    print(f"denoiser tc (2, {N}, {N}) in_nc {in_nc}: rel-L2 {err:.3e}")
    assert err <= TOL_DENOISER


@pytest.mark.parametrize("dtype", ["single_level", "multi_level"])
def test_admm_loop_with_builtin_unetres_256(q, ops, dtype):
    """10 iterations on a 2-slice batch, tensor-mode UNetRes, against the oracle loop with the CPU UNetRes (slice by slice)."""
    from oracle import unetres
    from oracle.admm import pnp_admm
    P, Po = ops["spiral"]
    Fo, Xgt, Y, X0 = make_problem(Po, 24, S=2)
    in_nc = 10 if dtype == "single_level" else 11
    sd = unetres.make_state_dict(in_nc, seed=0)
    net = q.UNetRes(sd, in_nc=in_nc)
    net.set_precision("tc")
    param = {"iter": 10, "gamma": 0.05, "denoiser_type": dtype}
    if dtype == "multi_level":
        param["noise_map"] = q.build_noise_map(0.01, N, N)
        assert param["noise_map"].shape == (N, N)
    x = q.PnP_ADMM(Y, dict(param, F=q.fft_operator(P), net=net, X0=X0))
    assert x.shape == (N, N, 10, 2)
    for s in range(2):
        xo = pnp_admm(Y[:, s], dict(param, F=Fo, X0=X0[..., s], net=lambda v: unetres.denoise_matlab_layout(sd, v)), solver="exact")
        err = rel_l2(x[..., s], xo)
        print(f"admm {dtype} 256 slice {s}: rel-L2 {err:.3e}")
        assert err <= 1e-4  # bounded by the denoiser tolerance


def test_admm_session_graph_replay_256(q, ops):
    """An AdmmSession run twice replays its captured CUDA graph: bit-identical to itself and to PnP_ADMM."""
    from oracle import unetres
    P, Po = ops["spiral"]
    Fo, Xgt, Y, X0 = make_problem(Po, 25, S=2)
    net = q.UNetRes(unetres.make_state_dict(10, seed=0), in_nc=10)
    param = {"iter": 8, "gamma": 0.05, "X0": X0, "denoiser_type": "single_level", "F": q.fft_operator(P), "net": net}
    x_ref = q.PnP_ADMM(Y, param)
    sess = q.AdmmSession(param, 2)
    try:
        runs = []
        for _ in range(2):
            sess.upload(Y, X0)
            sess.run()
            runs.append(sess.download())
    finally:
        sess.close()
    assert np.array_equal(runs[0], runs[1])
    assert np.array_equal(runs[0].reshape(x_ref.shape), x_ref)


# ---- downstream: matching, LRTV, mask and metrics --------------------------------------------------------------------------------
def test_matching_on_a_256_reconstruction(q, ops):
    from oracle import synth
    from oracle.matching import mrf_dtm_cpu as oracle_match
    P, Po = ops["spiral"]
    Fo, Xgt, Y, X0 = make_problem(Po, 27)
    x = q.PnP_ADMM(Y, {"iter": 3, "gamma": 0.05, "X0": X0, "denoiser_type": "single_level", "F": q.fft_operator(P),
                       "net": lambda v: v})
    d = synth.make_dictionary(K_target=4000, cut=3, seed=0)
    out = q.mrf_dtm_cpu(d, {"X": x}, {"f": {"qout": 1, "pdout": 1, "dmout": 1}})
    ref = oracle_match(d, {"X": x}, None, return_gap=True)
    assert out["qmap"].shape[:2] == (N, N) and out["pd"].shape == (N, N) and out["dm"].shape == (N, N)
    decided = ref["gap"] >= NEAR_TIE
    assert decided.any()
    assert np.array_equal(out["dm"].astype(np.int64)[decided], ref["dm"][decided])


def test_lrtv_256(q, ops):
    from oracle import lrtv
    P, Po = ops["spiral"]
    from oracle.sampling import FOperator
    F, Fo = q.fft_operator(P), FOperator(Po)
    X0 = tsmi(11)
    Y = q.awgn(Fo.forward(X0), 30.0, "measured", seed=3)
    step0 = X0.size / Y.size
    param = {"K": 4e-5, "iter": 4, "step": step0, "tol": 1e-4, "backtrack": 1}
    data = {"N": N, "M": N, "L": 10, "y": Y, "F": F, "D": []}
    x, info = q.FISTA_deep(data, param, return_info=True)
    xo, its = lrtv.fista_lrtv(Y, Fo, X0.shape, K=4e-5, max_iter=4, step=step0, tol=1e-4, backtrack=True)
    assert info["iter"] == its
    assert x.shape == (N, N, 10) and rel_l2(x, xo) < 1e-4


def test_foreground_mask_and_metrics_256(q):
    import benchdata
    from oracle import metrics
    qm0 = np.transpose(benchdata.make_qmaps(seed=2, S=1, N=N, M=N)[0], (1, 2, 0))       # N x N x (T1, T2, PD)
    mask = q.getmask_fromPD(qm0[:, :, 2], 0.15)
    assert mask.shape == (N, N) and np.array_equal(mask, metrics.getmask_fromPD(qm0[:, :, 2], 0.15))
    rng = np.random.default_rng(4)
    est = qm0 * (1 + 0.03 * rng.standard_normal(qm0.shape))
    X0 = rng.standard_normal((N, N, 10)) * mask[:, :, None] * 0.2
    X = X0 + 0.01 * (rng.standard_normal(X0.shape) + 1j * rng.standard_normal(X0.shape))
    got = q.recon_metrics(est, qm0, mask, X, X0)
    ref = metrics.recon_metrics(est, qm0, mask, X, X0)
    assert set(got) == set(ref)
    for k in ref:
        assert got[k] == pytest.approx(ref[k], rel=1e-9, abs=1e-12), k


# ---- what stays unsupported -----------------------------------------------------------------------------------------------------
def test_other_sizes_and_the_cluster_kernel_stay_unsupported(q, monkeypatch):
    with pytest.raises(q.QmriError, match="224"):
        q.setup_subsampling_spiralgrided(240, 240, 771, np.eye(10))
    with pytest.raises(q.QmriError, match="224"):
        q.setup_subsampling_epi(256, 224, 1 / 65, np.eye(10))
    with pytest.raises(q.QmriError, match="224"):
        q.setup_subsampling_spiralgrided(128, 128, 771, np.eye(10))
    monkeypatch.setenv("QMRI_K1_KERNEL", "cluster")                 # read when the operator is built
    P = q.setup_subsampling_spiralgrided(N, N, 771, np.eye(10))
    F = q.fft_operator(P)
    with pytest.raises(q.QmriError, match="cluster"):
        F.forward(tsmi(1))
