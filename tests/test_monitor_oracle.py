"""The PnP-ADMM convergence history (PnP_ADMM.m:106-109) on the CPU oracle.

The device computes the data-consistency residual from the solve's own residual: with x = z + A^H (y - A z) / (1 + rho) and
A A^H = I, |y - A x| = rho / (1 + rho) |y - A z|.  These tests check that identity on the exact float64 x-update, and define the
reference history the GPU tests compare with: |y - F.forward(x_k)| / |y| and |gt - x_k| / |gt|, computed directly from the iterate
x_k of the oracle loop (the x-update output of iteration k, before the denoiser).
"""
import numpy as np
import pytest

from oracle import sampling
from oracle.admm import pnp_admm
from oracle.sampling import FOperator
from oracle.xupdate import xupdate_exact


def oracle_history(y, param):
    """(x, dc_res, gt_err) of the oracle loop for one slice; dc_res / gt_err are float64 arrays of length param['iter']
    (gt_err None without param['gt_tsmi'])."""
    trace = []
    x = pnp_admm(y, param, solver="exact", trace=trace)
    F, gt = param["F"], param.get("gt_tsmi")
    y = np.asarray(y, dtype=np.complex128)
    dc = np.array([np.linalg.norm(y - F.forward(t["x"])) / np.linalg.norm(y) for t in trace])
    ge = None
    if gt is not None:
        gt = np.asarray(gt, dtype=np.complex128)
        ge = np.array([np.linalg.norm((gt - t["x"]).ravel()) / np.linalg.norm(gt.ravel()) for t in trace])
    return x, dc, ge


def box_denoiser(v):
    v = np.asarray(v, dtype=np.float64)[:, :, :10]
    return (v + np.roll(v, 1, 0) + np.roll(v, -1, 0) + np.roll(v, 1, 1) + np.roll(v, -1, 1)) / 5.0


def _problem(kind, N, seed):
    V = np.eye(10)
    Po = (sampling.setup_subsampling_spiralgrided(N, N, 771, V) if kind == "spiral"
          else sampling.setup_subsampling_epi(N, N, 1 / 65, V))
    F = FOperator(Po)
    rng = np.random.default_rng(seed)
    gt = rng.standard_normal((N, N, 10)) + 0.3j * rng.standard_normal((N, N, 10))
    y = F.forward(gt) + 0.05 * (rng.standard_normal(Po.nmeas) + 1j * rng.standard_normal(Po.nmeas))
    return F, gt, y


@pytest.mark.parametrize("kind,N", [("spiral", 224), ("epi", 224), ("spiral", 256)])
@pytest.mark.parametrize("rho", [0.05, 1.7])
def test_residual_identity_of_the_exact_xupdate(kind, N, rho):
    F, gt, y = _problem(kind, N, 3)
    rng = np.random.default_rng(4)
    z = rng.standard_normal((N, N, 10)) + 1j * rng.standard_normal((N, N, 10))
    x = xupdate_exact(F, y, z, rho)
    lhs = np.linalg.norm(y - F.forward(x))
    rhs = rho / (1.0 + rho) * np.linalg.norm(y - F.forward(z))
    assert abs(lhs - rhs) <= 1e-12 * rhs


def test_oracle_history_matches_the_iterates():
    F, gt, y = _problem("spiral", 224, 5)
    X0 = F.adjoint(y)
    rho = 0.05
    param = {"iter": 4, "gamma": rho, "F": F, "X0": X0, "net": box_denoiser, "gt_tsmi": gt}
    x, dc, ge = oracle_history(y, param)
    assert dc.shape == (4,) and ge.shape == (4,)
    # k = 1 is the solve from X0, computed independently of the loop
    x1 = xupdate_exact(F, y, X0, rho)
    assert abs(dc[0] - np.linalg.norm(y - F.forward(x1)) / np.linalg.norm(y)) <= 1e-12
    assert abs(ge[0] - np.linalg.norm((gt - x1).ravel()) / np.linalg.norm(gt.ravel())) <= 1e-12
    # row k is the norm of what a k-iteration run returns
    for k in (2, 4):
        xk = x if k == 4 else pnp_admm(y, dict(param, iter=k), solver="exact")
        assert dc[k - 1] == pytest.approx(np.linalg.norm(y - F.forward(xk)) / np.linalg.norm(y), rel=1e-12)
        assert ge[k - 1] == pytest.approx(np.linalg.norm((gt - xk).ravel()) / np.linalg.norm(gt.ravel()), rel=1e-12)
    assert np.all(np.isfinite(dc)) and np.all(dc > 0)
    _, dc0, ge0 = oracle_history(y, dict(param, iter=0))
    assert dc0.shape == (0,) and ge0.shape == (0,)
    _, _, none = oracle_history(y, {k: v for k, v in param.items() if k != "gt_tsmi"})
    assert none is None
