"""FISP-MRF dictionaries simulated on the B200 (qmri_fisp_signals / _gram / _compress through qmri_b200) against the float64
EPG oracle (oracle/epg.py), and the dictionary through the reference's flow: synthesis, matching and the general-V operator."""
import numpy as np
import pytest

from conftest import rel_l2
from test_oracle_epg import schedule

pytestmark = pytest.mark.gpu

TOL = 1e-5
NEAR_TIE = 1e-6


@pytest.fixture(scope="module")
def q():
    import qmri_b200
    qmri_b200.Context.default()  # raises without a B200: no fallback
    return qmri_b200


def grid_lut():
    """(T1, T2) grid with T2 from 10 ms and T1 up to 4 s, T2 < T1, plus the corners."""
    t1 = np.geomspace(0.1, 4.0, 9)
    t2 = np.geomspace(0.01, 2.0, 8)
    g1, g2 = np.meshgrid(t1, t2, indexing="ij")
    keep = g2 < g1
    lut = np.stack([g1[keep], g2[keep]], axis=1)
    return np.vstack([lut, [[4.0, 0.01], [4.0, 2.0], [0.1, 0.01]]]).astype(np.float32)


def oracle_signals(lut, seq):
    from oracle import epg
    lut = np.asarray(lut, np.float64)   # the float32 values the kernels simulate
    return epg.epg_fisp(lut[:, 0], lut[:, 1], seq).real


def rel_rows(a, b):
    return np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)


@pytest.mark.parametrize("T", [1000, 200, 100])
@pytest.mark.parametrize("ti", [None, 0.02])
def test_signals_match_oracle(q, T, ti):
    lut = grid_lut()
    seq = dict(schedule(T), ti=ti)
    sig = q.fisp_signals(lut, seq)
    ref = oracle_signals(lut, seq)
    err = rel_rows(sig.astype(np.float64), ref)
    print(f"T = {T} ti = {ti}: max per-atom rel-L2 {err.max():.2e} over {lut.shape[0]} atoms")
    assert sig.shape == (lut.shape[0], T) and sig.dtype == np.float32
    assert err.max() <= TOL


@pytest.mark.parametrize("T,K", [(1000, 600), (200, 3000), (100, 40000)])
def test_gram_matches_oracle_and_is_reproducible(q, T, K):
    """(100, 40000) spans two simulation chunks of 32 768 atoms."""
    from oracle import epg
    rng = np.random.default_rng(T)
    lut = np.stack([rng.uniform(0.1, 4.0, K), rng.uniform(0.01, 0.6, K)], axis=1).astype(np.float32)
    seq = dict(schedule(T, seed=3), ti=0.02)
    G = q.fisp_gram(lut, seq)
    lut64 = lut.astype(np.float64)
    Go = epg.gram(epg.epg_fisp_real(lut64[:, 0], lut64[:, 1], seq))
    err = np.linalg.norm(G - Go) / np.linalg.norm(Go)
    print(f"T = {T} K = {K}: Gram rel-Frobenius {err:.2e}")
    assert err <= TOL
    assert np.array_equal(G, G.T)
    assert np.array_equal(G, q.fisp_gram(lut, seq))


@pytest.mark.parametrize("T", [1000, 200, 100])
def test_compress_matches_oracle_and_shards(q, T):
    from oracle import epg
    lut = grid_lut()
    seq = dict(schedule(T, seed=4), ti=None)
    ref = oracle_signals(lut, seq)
    Vo, _ = epg.temporal_basis(epg.gram(ref), 10)
    Do, ndo = epg.compress(ref, Vo)
    d = q.fisp_dictionary(lut, seq, V=Vo)
    assert d["D"].dtype == np.float32 and d["normD"].dtype == np.float32 and d["D"].shape == (lut.shape[0], 10)
    eD = rel_rows(d["D"].astype(np.float64), Do).max()
    en = np.max(np.abs(d["normD"] - ndo) / ndo)
    print(f"T = {T}: D max per-atom rel-L2 {eD:.2e}, normD max rel {en:.2e}")
    assert eD <= TOL and en <= TOL
    np.testing.assert_array_equal(d["lut"], lut)
    # an atom range is bit-identical to the matching rows of the whole call, and loads as a resident shard
    a0, a1 = 7, 41
    s = q.fisp_dictionary(lut, seq, V=Vo, atoms=(a0, a1))
    assert np.array_equal(s["D"], d["D"][a0:a1]) and np.array_equal(s["normD"][a0:a1], d["normD"][a0:a1])
    assert np.all(np.isnan(s["normD"][:a0])) and np.all(np.isnan(s["normD"][a1:]))
    sh = q.Dictionary(s, shard=(a0, a1), shard_only=True)
    assert sh.K == lut.shape[0]
    sh.close()


@pytest.mark.parametrize("T", [200, 1000])
def test_temporal_basis_matches_oracle(q, T):
    from oracle import epg
    rng = np.random.default_rng(10 + T)
    K = 1500
    lut = np.stack([rng.uniform(0.1, 4.0, K), rng.uniform(0.01, 0.6, K)], axis=1).astype(np.float32)
    seq = dict(schedule(T, seed=5), ti=0.02)
    lut64 = lut.astype(np.float64)
    Go = epg.gram(epg.epg_fisp_real(lut64[:, 0], lut64[:, 1], seq))
    Vo, wo = epg.temporal_basis(Go, 10)
    G = q.fisp_gram(lut, seq)
    w = np.sort(np.linalg.eigvalsh(G))[::-1]
    assert np.max(np.abs(w[:10] - wo[:10])) <= TOL * wo[0]
    V = q.fisp_dictionary(lut, seq, C=10)["V"]
    np.testing.assert_allclose(V.T @ V, np.eye(10), atol=1e-12)
    # Davis-Kahan (Yu, Wang & Samworth 2015): |sin Theta|_F <= 2 |G - Go|_F / (lambda_10 - lambda_11)
    bound = np.sqrt(2) * 2 * np.linalg.norm(G - Go) / (wo[9] - wo[10])
    diff = np.linalg.norm(V @ V.T - Vo @ Vo.T)
    print(f"T = {T}: projector difference {diff:.2e}, Davis-Kahan bound {bound:.2e}")
    assert diff <= bound


def test_round_trip_synthesis_and_matching(q):
    """cut3 (T = 200) dictionary of ~20 000 atoms -> synthesize_tsmis on phantom slices at 224 -> noiseless mrf_dtm_cpu."""
    import benchdata
    from oracle.matching import mrf_dtm_cpu as oracle_match
    lut = benchdata.dictionary_grid(20000).astype(np.float32)
    d = q.fisp_dictionary(lut, schedule(200, seed=6), C=10)
    assert d["V"].shape == (200, 10)
    for qm in benchdata.volunteer_slices(0, 2):
        X, I = q.synthesize_tsmis(d, qm, return_index=True)
        out = q.mrf_dtm_cpu(d, {"X": X}, {"f": {"qout": 1, "pdout": 1, "dmout": 1}})
        ref = oracle_match(d, {"X": X}, None, return_gap=True)
        decided = (ref["gap"] >= NEAR_TIE).reshape(-1, order="F")
        dm = out["dm"].reshape(-1, order="F").astype(np.int64) - 1
        fg = (qm[2] > 0).reshape(-1, order="F")
        print(f"decided pixels {decided.sum()} of {fg.sum()} in the foreground")
        assert decided[fg].sum() > 0.5 * fg.sum()
        assert np.array_equal(dm[decided], I[decided])
        qmap = out["qmap"].reshape(-1, 2, order="F")
        np.testing.assert_array_equal(qmap[decided], lut[I[decided]])


def test_reference_flow_general_V(q):
    """main_recon_tsmis_FFT.m: V = dict.V (200 x 10) -> setup_subsampling_spiralgrided(224, 224, 771, V) -> F.forward, F.adjoint
    and one x-update against the oracle."""
    from oracle import sampling
    from oracle.xupdate import xupdate_exact
    rng = np.random.default_rng(7)
    lut = np.stack([rng.uniform(0.1, 4.0, 4000), rng.uniform(0.01, 0.6, 4000)], axis=1).astype(np.float32)
    V = q.fisp_dictionary(lut, schedule(200, seed=7), C=10)["V"]
    P, Po = q.setup_subsampling_spiralgrided(224, 224, 771, V), sampling.setup_subsampling_spiralgrided(224, 224, 771, V)
    F, Fo = q.fft_operator(P), sampling.FOperator(Po)
    n = np.arange(224)[:, None, None] / 224.0
    m = np.arange(224)[None, :, None] / 224.0
    c = np.arange(10)[None, None, :]
    x = np.exp(-((n - 0.5) ** 2 + (m - 0.4) ** 2) * 6) * np.cos(0.4 * c + 0.2) + 0.05 * rng.standard_normal((224, 224, 10))
    y = F.forward(x)
    yo = Fo.forward(x)
    assert rel_l2(y.reshape(-1), yo.reshape(-1)) <= TOL
    assert rel_l2(F.adjoint(yo), Fo.adjoint(yo)) <= TOL
    v = np.real(Fo.adjoint(yo)) + 0.02 * rng.standard_normal((224, 224, 10))
    assert rel_l2(F.xupdate(yo, v, None, 0.05), xupdate_exact(Fo, yo, v, 0.05)) <= TOL


def test_invalid_inputs(q):
    import ctypes
    from qmri_b200._capi import QMRI_EINVAL, QMRI_EUNSUPPORTED, Context, FispSeq, QmriError, check
    lut = grid_lut()
    base = schedule(100)

    def code(fn):
        with pytest.raises(QmriError) as e:
            fn()
        return e.value.code

    def with_(**kw):
        s = dict(base)
        s.update(kw)
        return s

    bad = [with_(flip_deg=np.r_[-1.0, base["flip_deg"][1:]]), with_(flip_deg=np.r_[np.nan, base["flip_deg"][1:]]),
           with_(flip_deg=np.r_[np.inf, base["flip_deg"][1:]]), with_(tr=np.r_[0.0, base["tr"][1:]]),
           with_(tr=np.r_[-0.01, base["tr"][1:]]), with_(te=-1e-3), with_(te=float(np.min(base["tr"])) + 1e-4),
           with_(te=np.nan), with_(ti=-0.01), with_(ti=np.nan), with_(flip_deg=np.zeros(0), tr=np.zeros(0))]
    for s in bad:
        assert code(lambda: q.fisp_signals(lut, s)) == QMRI_EINVAL
        assert code(lambda: q.fisp_gram(lut, s)) == QMRI_EINVAL
    for l2 in (np.r_[lut, [[0.0, 0.05]]], np.r_[lut, [[1.0, -0.05]]], np.r_[lut, [[np.nan, 0.05]]], np.r_[lut, [[1.0, np.inf]]]):
        assert code(lambda: q.fisp_signals(l2, base)) == QMRI_EINVAL
        assert code(lambda: q.fisp_dictionary(l2, base, V=np.eye(100)[:, :10])) == QMRI_EINVAL
    V = np.linalg.qr(np.random.default_rng(0).standard_normal((100, 10)))[0]
    K = lut.shape[0]
    for atoms in ((0, 0), (5, 3), (-1, 4), (0, K + 1)):
        assert code(lambda: q.fisp_dictionary(lut, base, V=V, atoms=atoms)) == QMRI_EINVAL
    assert code(lambda: q.fisp_dictionary(lut, base, V=np.ones((100, 17)))) == QMRI_EINVAL          # C <= 16
    assert code(lambda: q.fisp_dictionary(lut, schedule(8), V=np.ones((8, 10)))) == QMRI_EINVAL  # C <= T
    long = schedule(1100)
    assert code(lambda: q.fisp_signals(lut, long)) == QMRI_EUNSUPPORTED
    assert code(lambda: q.fisp_gram(lut, long)) == QMRI_EUNSUPPORTED
    assert q.fisp_signals(lut, schedule(1024)).shape == (K, 1024)
    # null pointers through the C ABI
    ctx = Context.default()
    flip, tr = np.ascontiguousarray(base["flip_deg"]), np.ascontiguousarray(base["tr"])
    s = FispSeq(T=100, flip_deg=flip.ctypes.data, tr=tr.ctypes.data, te=0.004, inversion=0, ti=0.0)
    lutf = np.asfortranarray(lut)
    out = np.empty((K, 100), np.float32, order="F")
    G = np.empty((100, 100))
    for call in (lambda: ctx.lib.qmri_fisp_signals(ctx.handle, None, lutf.ctypes.data, K, out.ctypes.data),
                 lambda: ctx.lib.qmri_fisp_signals(ctx.handle, ctypes.byref(s), None, K, out.ctypes.data),
                 lambda: ctx.lib.qmri_fisp_signals(ctx.handle, ctypes.byref(s), lutf.ctypes.data, K, None),
                 lambda: ctx.lib.qmri_fisp_gram(None, ctypes.byref(s), lutf.ctypes.data, K, G.ctypes.data),
                 lambda: ctx.lib.qmri_fisp_compress(ctx.handle, ctypes.byref(s), lutf.ctypes.data, K, None, 10, 0, K,
                                                    out.ctypes.data, G.ctypes.data)):
        assert code(lambda: check(call())) == QMRI_EINVAL
    s0 = FispSeq(T=100, flip_deg=None, tr=tr.ctypes.data, te=0.004, inversion=0, ti=0.0)
    assert code(lambda: check(ctx.lib.qmri_fisp_gram(ctx.handle, ctypes.byref(s0), lutf.ctypes.data, K, G.ctypes.data))) == QMRI_EINVAL
