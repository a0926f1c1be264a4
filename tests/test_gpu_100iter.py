"""The loop the benchmark times, against the oracle (VERDICT r1 parity item 1a / ADVICE): 100 PnP-ADMM iterations with the
built-in random-init UNetRes in tensor mode (split-bf16 tcgen05) through the CUDA-graph replay, spiral and EPI masks, one slice
and a 15-slice batch - relative L2 against ``oracle.admm.pnp_admm`` (float64 x-update + PyTorch-CPU fp32 UNetRes) recorded every
10 iterations.

Measured on B200 (profiles/r02_drift100.json): the loop does not amplify the per-forward difference - tensor mode stays at
1e-6 (EPI) / 2e-5 (spiral) relative L2 through all 100 iterations, the fp32 CUDA-core mode at 1e-7 ... 1e-5; asserted here:
<= 1e-4 at EVERY checkpoint (the north-star denoiser tolerance, which bounds the loop), both precision modes, and the curve is
printed as one JSON line per case (pytest -s shows it)."""
import json
import time

import numpy as np
import pytest

from conftest import rel_l2

pytestmark = pytest.mark.gpu

CHECKPOINTS = list(range(10, 101, 10))


def _problem(q, kind, S, seed):
    from oracle import sampling, synth
    import bench
    V = np.eye(10)
    if kind == "spiral":
        P, Po = q.setup_subsampling_spiralgrided(224, 224, 771, V), sampling.setup_subsampling_spiralgrided(224, 224, 771, V)
    else:
        P, Po = q.setup_subsampling_epi(224, 224, 1 / 65, V), sampling.setup_subsampling_epi(224, 224, 1 / 65, V)
    Fo = sampling.FOperator(Po)
    X = bench.synthetic_slices(S, seed)
    Y = np.stack([synth.awgn_measured(Fo.forward(X[..., s]), 30, seed + s) for s in range(S)], axis=1)
    X0 = np.stack([Fo.adjoint(Y[:, s]) for s in range(S)], axis=3)
    return P, Fo, Y, X0


def drift_curves(q, kind, S, picks, seed=31):
    """rel-L2 of the device loop vs the oracle loop at CHECKPOINTS, for the slices in `picks`, in tc and fp32 mode."""
    from oracle import unetres
    from oracle.admm import pnp_admm
    P, Fo, Y, X0 = _problem(q, kind, S, seed)
    sd = unetres.make_state_dict(10, seed=0)
    net = q.UNetRes(sd, in_nc=10)
    F = q.fft_operator(P)
    oracle_x = {}
    t0 = time.time()
    for s in picks:
        trace = []
        pnp_admm(Y[:, s], {"iter": 100, "gamma": 0.05, "F": Fo, "X0": X0[..., s],
                           "net": lambda v: unetres.denoise_matlab_layout(sd, v)}, solver="exact", trace=trace)
        oracle_x[s] = {k: trace[k - 1]["x"] for k in CHECKPOINTS}
    t_oracle = time.time() - t0
    out = {"mask": kind, "slices": S, "picks": list(picks), "oracle_seconds": t_oracle}
    for mode in ("tc", "fp32"):
        net.set_precision(mode)
        sess = q.AdmmSession({"iter": 100, "gamma": 0.05, "F": F, "X0": X0, "net": net, "denoiser_type": "single_level"}, S)
        sess.upload(Y, X0)
        curve = {s: [] for s in picks}
        for k in CHECKPOINTS:
            sess.run(k)                                     # restarts from X0: iterations 2 .. k-2 are graph replays
            x = sess.download()
            for s in picks:
                curve[s].append(rel_l2(x[..., s], oracle_x[s][k]))
        sess.close()
        out[mode] = {str(s): curve[s] for s in picks}
    net.close()
    return out


@pytest.mark.parametrize("kind,S,picks", [("spiral", 1, (0,)), ("epi", 1, (0,)), ("spiral", 15, (0, 14)), ("epi", 15, (7,))])
def test_100_iterations_against_the_oracle(kind, S, picks):
    import qmri_b200 as q
    q.Context.default()
    res = drift_curves(q, kind, S, picks)
    print(json.dumps({f"{kind}_S{S}": res}))
    for s in picks:
        tc, fp = res["tc"][str(s)], res["fp32"][str(s)]
        assert np.all(np.isfinite(tc)) and np.all(np.isfinite(fp))
        assert max(tc) <= 1e-4, f"{kind} S={S} slice {s}: tensor-mode drift {tc}"
        assert max(fp) <= 1e-4, f"{kind} S={S} slice {s}: fp32-mode drift {fp}"
