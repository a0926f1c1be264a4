"""FISP-MRF dictionaries simulated on the GPU: the ``dict`` struct the reference loads from
``dictionaries/real_fisp_cut*_dict/SVD_dict_FISP_cut*.mat`` (``main_recon_tsmis_FFT.m:127-129``,
``main_synthesize_tsmis.m:50-54``; fields as in ``mrf_dtm_cpu.m:8-12``).

    seq  : {'flip_deg': [T] degrees, 'tr': [T] seconds, 'te': seconds, 'ti': seconds or None (no inversion)}
    lut  : [K x 2] (T1, T2) in seconds; the atoms are simulated at exactly these float32 values

The signal model (EPG FISP, RF phase 0, one dephasing cycle per TR) is stated in ``include/qmri.h``.  ``cut`` = the first T
pulses of a schedule (``main_recon_tsmis_FFT.m:42``).
"""
from __future__ import annotations

from ctypes import byref

import numpy as np

from ._capi import Context, FispSeq, check, ptr


def _seq(seq):
    flip = np.ascontiguousarray(np.asarray(seq["flip_deg"], dtype=np.float64).reshape(-1))
    tr = np.ascontiguousarray(np.asarray(seq["tr"], dtype=np.float64).reshape(-1))
    if tr.size != flip.size:
        raise ValueError(f"seq: {flip.size} flip angles but {tr.size} repetition times")
    ti = seq.get("ti")
    s = FispSeq(T=flip.size, flip_deg=ptr(flip), tr=ptr(tr), te=float(seq["te"]), inversion=0 if ti is None else 1,
                ti=0.0 if ti is None else float(ti))
    return s, (flip, tr)  # the arrays must outlive the call


def _lut(lut):
    a = np.asfortranarray(np.asarray(lut, dtype=np.float32))
    if a.ndim != 2 or a.shape[1] != 2:
        raise ValueError("lut must be K x 2 (T1, T2)")
    return a


def fisp_signals(lut, seq, ctx=None):
    """Raw fingerprints: [K x T] float32 (row k = the atom lut[k])."""
    ctx = ctx or Context.default()
    s, keep = _seq(seq)
    lut = _lut(lut)
    sig = np.empty((lut.shape[0], s.T), np.float32, order="F")
    check(ctx.lib.qmri_fisp_signals(ctx.handle, byref(s), ptr(lut), lut.shape[0], ptr(sig)))
    return sig


def fisp_gram(lut, seq, ctx=None):
    """Temporal Gram matrix sum_k d_k d_k^T: [T x T] float64, exactly symmetric, the same bits on every call."""
    ctx = ctx or Context.default()
    s, keep = _seq(seq)
    lut = _lut(lut)
    G = np.empty((s.T, s.T), np.float64, order="F")
    check(ctx.lib.qmri_fisp_gram(ctx.handle, byref(s), ptr(lut), lut.shape[0], ptr(G)))
    return G


def temporal_basis(G, C=10):
    """dict.V from a Gram matrix: the top-C eigenvectors in descending eigenvalue order (float64, on the host), each column
    signed so that its entry of largest magnitude is positive (the lowest index wins a tie)."""
    w, U = np.linalg.eigh(np.asarray(G, dtype=np.float64))
    V = U[:, np.argsort(w)[::-1][:C]]
    peak = np.argmax(np.abs(V), axis=0)
    V = V * np.where(V[peak, np.arange(V.shape[1])] < 0, -1.0, 1.0)
    return np.asfortranarray(V)


def fisp_dictionary(lut, seq, C=10, V=None, atoms=None, gram_lut=None, ctx=None):
    """``dict`` = {'D', 'normD', 'lut', 'V'} with the conventions of ``benchdata.make_dictionary``: D [K x C] unit-norm float32
    rows d V / |d V|, normD [K] float32 = |d V|, lut [K x 2] float32, V [T x C] float64.  ``V=None``: V =
    ``temporal_basis(fisp_gram(gram_lut or lut))``.  ``atoms=(a0, a1)``: D holds rows a0..a1-1 only (the shard an atom-sharded
    rank loads with ``Dictionary(..., shard=atoms, shard_only=True)``); normD is NaN outside the range."""
    ctx = ctx or Context.default()
    lut = _lut(lut)
    K = lut.shape[0]
    if V is None:
        V = temporal_basis(fisp_gram(lut if gram_lut is None else gram_lut, seq, ctx), C)
    V = np.asfortranarray(np.asarray(V, dtype=np.float64))
    s, keep = _seq(seq)
    if V.ndim != 2 or V.shape[0] != s.T:
        raise ValueError(f"V must be T x C with T = {s.T}")
    C = V.shape[1]
    a0, a1 = (0, K) if atoms is None else (int(atoms[0]), int(atoms[1]))
    D = np.empty((max(a1 - a0, 0), C), np.float32, order="F")
    nd = np.empty(max(a1 - a0, 0), np.float32)
    check(ctx.lib.qmri_fisp_compress(ctx.handle, byref(s), ptr(lut), K, ptr(V), C, a0, a1, ptr(D), ptr(nd)))
    normD = np.full(K, np.nan, np.float32)
    normD[a0:a1] = nd
    return {"D": D, "normD": normD, "lut": lut, "V": V}

