"""``x = PnP_ADMM(y, param)`` - the reference's ADMM loop, run on the GPU.

Mirrors ``main_files/algorithms/PnP_ADMM/PnP_ADMM.m:1-148`` with the ``param`` struct of
``main_recon_tsmis_FFT.m:164-170,285-292``:

    param['iter'], param['gamma'], param['cg_tol'], param['F'], param['gt_tsmi'],
    param['X0'], param['net'], param['denoiser_type'] ('single_level' | 'multi_level'),
    param['noise_map'] (multi_level only)

``param['net']`` is either the built-in on-device :class:`UNetRes` (whole loop stays on the
device) or any Python callable ``v_out = net(v_in)`` taking the ``N x M x Cin`` array in [0,1]
and returning ``N x M x 10`` (the pluggable proximal step of the reference; costs a D2H/H2D hop
per iteration).  A trailing slice axis (``y: nmeas x S``, ``X0: N x M x C x S``) runs S
independent reconstructions, each with its own min/max normalisation (``PnP_ADMM.m:121``).

The least-squares step is solved exactly instead of by ``lsqr`` to ``cg_tol`` (identical to
1e-15 when ``A A^H = I``, SURVEY.md A.5), a deliberate difference from the reference.

The per-iteration progress of ``:106-109`` is not printed (that would stop the device loop
once per iteration); ``x, info = PnP_ADMM(y, param, history=True)`` records it on the device
instead and returns it after the run: ``info["dc_residual"]`` holds
``|y - F.forward(x_k)| / |y|`` and ``info["gt_error"]`` ``|param.gt_tsmi - x_k| / |param.gt_tsmi|``
(None without ``gt_tsmi``) for every iteration k, ``(iter, S)`` arrays (``(iter,)`` unbatched),
with ``x_k`` the x-update output of iteration k, before the denoiser.  With ``history=False``
``gt_tsmi`` is ignored and nothing extra runs.  :meth:`AdmmSession.monitor` /
:meth:`AdmmSession.history` are the same on a resident session.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from ._capi import QMRI_EINVAL, AdmmParams, DENOISE_FN, QmriError, as_f, check, dtype_code, ptr
from .denoiser import UNetRes
from .operators import FOperator


def _make_params(param, keep):
    for k in ("iter", "gamma", "F", "X0", "net"):
        if k not in param:
            raise KeyError(f"param.{k} is required (PnP_ADMM.m:60-77)")
    F = param["F"]
    if not isinstance(F, FOperator):
        raise TypeError("param['F'] must come from qmri_b200.fft_operator(P)")
    dtype = param.get("denoiser_type", "single_level")
    if dtype not in ("single_level", "multi_level"):
        raise ValueError(f"denoiser_type must be 'single_level' or 'multi_level', got {dtype!r}")
    p = AdmmParams()
    p.iters = int(param["iter"])
    p.gamma = float(param["gamma"])
    p.cg_tol = float(param.get("cg_tol", 1e-4))
    p.multi_level = 1 if dtype == "multi_level" else 0
    if p.multi_level:
        if "noise_map" not in param:
            raise KeyError("param.noise_map is required for the multi_level denoiser (PnP_ADMM.m:70-72)")
        nm = np.asfortranarray(np.asarray(param["noise_map"], dtype=np.float32))
        if nm.shape != (F.N, F.M):
            raise ValueError(f"noise_map must be {F.N} x {F.M}")
        keep.append(nm)
        p.noise_map = nm.ctypes.data
    net = param["net"]
    if isinstance(net, UNetRes):
        p.net = net.handle
    elif callable(net):
        cin = 11 if p.multi_level else 10

        def _cb(user, v_in, v_out, H, W, Cin, Cout, S, space, stream):
            try:
                n_in, n_out = H * W * Cin, H * W * Cout
                a = np.ctypeslib.as_array((C.c_float * (n_in * S)).from_address(v_in))
                o = np.ctypeslib.as_array((C.c_float * (n_out * S)).from_address(v_out))
                for s in range(S):
                    vi = a[s * n_in:(s + 1) * n_in].reshape((H, W, Cin), order="F")
                    vo = np.asarray(net(vi))
                    if vo.shape != (H, W, Cout):
                        raise ValueError(f"denoiser returned shape {vo.shape}, expected {(H, W, Cout)}")
                    o[s * n_out:(s + 1) * n_out] = vo.astype(np.float32).reshape(-1, order="F")
                return 0
            except Exception as e:  # never let an exception cross the C ABI
                keep.append(e)
                return 1

        cb = DENOISE_FN(_cb)
        keep.append(cb)
        p.fn = cb
        p.fn_space = _capi.QMRI_HOST
        del cin
    else:
        raise TypeError("param['net'] must be a qmri_b200.UNetRes or a callable")
    return p, F


def _prep_inputs(F, y, X0):
    y = as_f(y)
    if not np.iscomplexobj(y):
        y = y.astype(np.complex128)
    X0 = as_f(X0)
    batched = X0.ndim == 4
    S = X0.shape[3] if batched else 1
    if X0.shape[:3] != (F.N, F.M, F.C):
        raise ValueError(f"param.X0 must be {F.N} x {F.M} x {F.C}, got {X0.shape}")
    if y.size != F.P.nmeas * S:
        raise ValueError(f"y has {y.size} entries, expected {F.P.nmeas} per slice x {S} slices")
    return y, X0, S, batched


def _prep_gt(F, gt, S):
    gt = as_f(gt)
    if gt.shape != (F.N, F.M, F.C, S) and not (S == 1 and gt.shape == (F.N, F.M, F.C)):
        raise QmriError(QMRI_EINVAL, f"param.gt_tsmi must be {F.N} x {F.M} x {F.C}" + (f" x {S}" if S > 1 else "") +
                        f", got {gt.shape}")
    return gt


def PnP_ADMM(y, param, history=False):
    if history:
        return _pnp_admm_history(y, param)
    keep = []
    p, F = _make_params(param, keep)
    y, X0, S, batched = _prep_inputs(F, y, param["X0"])
    x = np.zeros((F.N, F.M, F.C, S), np.complex128, order="F")
    rc = F.P.ctx.lib.qmri_pnp_admm(F.P.handle, ptr(y), dtype_code(y), ptr(X0), dtype_code(X0), S, C.byref(p), ptr(x),
                                   dtype_code(x))
    for k in keep:
        if isinstance(k, Exception):
            raise k
    check(rc)
    return x if batched else x[..., 0]


def _pnp_admm_history(y, param):
    X0 = param.get("X0")
    batched = X0 is not None and np.ndim(X0) == 4
    S = np.shape(X0)[3] if batched else 1
    sess = AdmmSession(param, S)
    try:
        sess.monitor(param.get("gt_tsmi"))
        sess.upload(y, X0)
        sess.run()
        x = sess.download()
        info = sess.history()
    finally:
        sess.close()
    if not batched:
        x = x[..., 0]
        info = {k: (None if v is None else v[:, 0]) for k, v in info.items()}
    return x, info


class AdmmSession:
    """Resident-state variant of :func:`PnP_ADMM` (create / upload / run / download), used to time
    the loop with its inputs already in HBM and to chain matching without a host round trip."""

    def __init__(self, param, S):
        self._keep = []
        self.p, self.F = _make_params(param, self._keep)
        self.S = int(S)
        self.lib = self.F.P.ctx.lib
        h = C.c_void_p()
        check(self.lib.qmri_admm_create(self.F.P.handle, self.S, C.byref(self.p), C.byref(h)))
        self.handle = h
        self._mon_gt = False     # a ground truth is attached (monitor)
        self._run_gt = False     # ... and was for the last run (history)

    def upload(self, y, X0):
        y, X0, S, _ = _prep_inputs(self.F, y, X0)
        if S != self.S:
            raise ValueError(f"session was created for {self.S} slices, got {S}")
        check(self.lib.qmri_admm_upload(self.handle, ptr(y), dtype_code(y), ptr(X0), dtype_code(X0)))

    def upload_raw(self, y, X0):
        """No host-side conversion: arrays must already be F-contiguous (pinned buffers welcome)."""
        check(self.lib.qmri_admm_upload(self.handle, ptr(y), dtype_code(y), ptr(X0), dtype_code(X0)))

    def monitor(self, gt=None, enable=True):
        """Record the convergence history of ``PnP_ADMM.m:106-109`` in every later run (see :meth:`history`).
        ``gt``: the ground truth, ``N x M x C [x S]``, or None for the data-consistency residual only."""
        if not enable:
            check(self.lib.qmri_admm_monitor(self.handle, 0, None, 0))
            self._mon_gt = False
            return
        g = None if gt is None else _prep_gt(self.F, gt, self.S)
        check(self.lib.qmri_admm_monitor(self.handle, 1, ptr(g), 0 if g is None else dtype_code(g)))
        self._mon_gt = g is not None

    def history(self):
        """History of the last run: ``{"dc_residual": (iters, S), "gt_error": (iters, S) or None}``, float64."""
        n = C.c_int()
        check(self.lib.qmri_admm_history(self.handle, None, None, C.byref(n)))
        dc = np.zeros((n.value, self.S), np.float64, order="F")
        gt = np.zeros((n.value, self.S), np.float64, order="F") if self._run_gt else None
        check(self.lib.qmri_admm_history(self.handle, ptr(dc), ptr(gt), C.byref(n)))
        return {"dc_residual": dc, "gt_error": gt}

    def run(self, iters=None):
        self._run_gt = self._mon_gt
        check(self.lib.qmri_admm_run(self.handle, int(self.p.iters if iters is None else iters)))
        for k in self._keep:
            if isinstance(k, Exception):
                raise k

    def xupdate_only(self, reps=1):
        check(self.lib.qmri_admm_xupdate_only(self.handle, int(reps)))

    def xupdate_bytes(self):
        """Algorithmic bytes per pixel-channel of one x-update in the state formulation this session runs (8 or 20)."""
        return int(self.lib.qmri_admm_xupdate_bytes(self.handle))

    def download(self, out=None):
        F = self.F
        x = out if out is not None else np.zeros((F.N, F.M, F.C, self.S), np.complex128, order="F")
        check(self.lib.qmri_admm_download(self.handle, ptr(x), dtype_code(x)))
        return x

    def state_dev(self):
        re, im = C.c_void_p(), C.c_void_p()
        check(self.lib.qmri_admm_state_dev(self.handle, C.byref(re), C.byref(im)))
        return re.value, im.value

    def close(self):
        if self.handle:
            self.lib.qmri_admm_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
