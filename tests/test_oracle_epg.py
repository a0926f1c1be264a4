"""The FISP-MRF dictionary oracle (oracle/epg.py) against itself and the signal model, and the qmri_fisp_seq binding (CPU only)."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import epg


def schedule(T, seed=0):
    """Seeded FISP schedule: sinusoidal flip-angle lobes of 100 pulses between 10 degrees and a peak in [10, 60], TR 10-14 ms,
    TE 4 ms."""
    rng = np.random.default_rng(seed)
    i = np.arange(T)
    peaks = rng.uniform(10.0, 60.0, T // 100 + 2)
    flip = 10.0 + (peaks[i // 100] - 10.0) * np.abs(np.sin(np.pi * (i % 100) / 100))
    return {"flip_deg": flip, "tr": rng.uniform(0.010, 0.014, T), "te": 0.004, "ti": None}


T1 = np.array([0.3, 1.0, 4.0, 2.0, 0.8])
T2 = np.array([0.01, 0.1, 0.3, 1.5, 0.05])


def rel_rows(a, b):
    return np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)


@pytest.mark.parametrize("T", [100, 200])
@pytest.mark.parametrize("ti", [None, 0.02])
def test_epg_matches_isochromats(T, ti):
    s = dict(schedule(T), ti=ti)
    c = epg.epg_fisp(T1, T2, s)
    b = epg.bloch_fisp(T1, T2, s)
    assert np.abs(c.imag).max() == 0.0          # the sample i F+_0 is real
    # the isochromat mean is F+_0 (rotation about +x); the EPG sample is i F+_0: the fixed factor 1j
    assert rel_rows(c, 1j * b).max() <= 1e-12


@pytest.mark.parametrize("T", [100, 200, 1000])
def test_real_recursion_and_order_window(T):
    s = dict(schedule(T, seed=1), ti=0.015)
    c = epg.epg_fisp(T1, T2, s).real
    full = epg.epg_fisp_real(T1, T2, s, window=False)
    win = epg.epg_fisp_real(T1, T2, s, window=True)
    assert rel_rows(full, c).max() <= 1e-13
    assert rel_rows(win, c).max() <= 1e-13
    assert np.array_equal(win, full)            # dropping the orders outside the window changes nothing


@pytest.mark.parametrize("ti", [None, 0.02])
def test_first_sample(ti):
    s = dict(schedule(100), ti=ti)
    d = epg.epg_fisp(T1, T2, s)[:, 0].real
    z0 = 1.0 if ti is None else 1.0 - 2.0 * np.exp(-ti / T1)
    want = np.sin(np.deg2rad(s["flip_deg"][0])) * z0 * np.exp(-s["te"] / T2)
    np.testing.assert_allclose(d, want, rtol=1e-14, atol=0)


def test_cut_is_a_prefix():
    s = dict(schedule(500, seed=2), ti=0.02)
    full = epg.epg_fisp_real(T1, T2, s)
    for Tc in (100, 200, 300):
        short = epg.epg_fisp_real(T1, T2, s, T=Tc)
        np.testing.assert_allclose(full[:, :Tc], short, rtol=0, atol=1e-15)


def test_live_order_count():
    # about T^2/4 order-updates per atom, and never more than (T - 1) / 2 + 1 live orders (16 slots of 32 at T = 1024)
    for T in (100, 200, 1000, 1024):
        w = [epg.live_orders(i, T) + 1 for i in range(T)]
        assert max(w) == (T - 1) // 2 + 1
        assert abs(sum(w) - T * T / 4) <= T


def test_temporal_basis_sign_rule():
    rng = np.random.default_rng(0)
    sig = epg.epg_fisp_real(rng.uniform(0.2, 3, 40), rng.uniform(0.02, 0.3, 40), schedule(100))
    V, w = epg.temporal_basis(epg.gram(sig), 10)
    assert np.all(np.diff(w) <= 0)
    np.testing.assert_allclose(V.T @ V, np.eye(10), atol=1e-12)
    for c in range(10):
        p = np.argmax(np.abs(V[:, c]))
        assert V[p, c] > 0
    D, nd = epg.compress(sig, V)
    np.testing.assert_allclose(np.linalg.norm(D, axis=1), 1.0, atol=1e-14)


def test_fisp_seq_layout_matches_header(tmp_path):
    from qmri_b200._capi import FispSeq
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "qmri.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(qmri_fisp_seq), offsetof(qmri_fisp_seq, T),\n'
                   '         offsetof(qmri_fisp_seq, flip_deg), offsetof(qmri_fisp_seq, tr), offsetof(qmri_fisp_seq, te),\n'
                   '         offsetof(qmri_fisp_seq, inversion), offsetof(qmri_fisp_seq, ti));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(FispSeq)] + [getattr(FispSeq, f).offset for f, _ in FispSeq._fields_]
    assert got == want
