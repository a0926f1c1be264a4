"""160 x 160 and 192 x 192 images on the CPU: the mask constructors, the streaming kernels' work-item tables and the streaming
kernels' arithmetic (csrc/xupdate_stream.cu, N = 16 R instances with R = 10 and 12: a radix-R register stage and a radix-16 stage,
R-column slabs, one thread per k-space row), thread by thread through csrc/k1_emulate.cpp, against the float64 oracle.
tests/test_gpu_sizes.py repeats the comparison on the device."""
import ctypes
import os

import numpy as np
import pytest

from conftest import PKG, rel_l2
from oracle import sampling
from oracle.xupdate import xupdate_exact

LIB = os.path.join(PKG, "lib", "libk1emu.so")
fp = ctypes.POINTER(ctypes.c_float)
SIDES = [160, 192]
MASKS = [(0, 771.0), (1, 1 / 65)]   # pattern 0: spiral with S = 771, pattern 1: EPI with 1/65 of the rows


def P(a):
    return a.ctypes.data_as(fp) if a is not None else None


@pytest.fixture(scope="module")
def emu():
    if not os.path.exists(LIB):
        pytest.skip("libk1emu.so not built (run __graft_entry__.build())")
    lib = ctypes.CDLL(LIB)
    lib.k1emu_masks.restype = ctypes.c_int
    lib.k1emu_masks.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.k1emu_run_n.restype = ctypes.c_int
    lib.k1emu_run_n.argtypes = [ctypes.c_int] * 3 + [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [fp] * 4 + [ctypes.c_float] + [fp] * 4
    lib.k1emu_stream_tables.restype = ctypes.c_int
    lib.k1emu_stream_tables.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int] + [ctypes.c_void_p] * 4
    return lib


def oracle_op(N, pat, L):
    return (sampling.setup_subsampling_spiralgrided(N, N, 771, np.eye(L)) if pat == 0
            else sampling.setup_subsampling_epi(N, N, 1 / 65, np.eye(L)))


def planar(a):
    a = np.transpose(a, (2, 1, 0))
    return np.ascontiguousarray(a.real.astype(np.float32)), np.ascontiguousarray(a.imag.astype(np.float32))


def unplanar(re, im):
    return np.transpose(re.astype(np.float64) + 1j * im.astype(np.float64), (2, 1, 0))


@pytest.mark.parametrize("N", SIDES)
@pytest.mark.parametrize("pat,arg", MASKS)
def test_cxx_mask_constructors_equal_oracle_sizes(emu, N, pat, arg):
    for L in (10, 50):
        Po = oracle_op(N, pat, L)
        n = emu.k1emu_masks(pat, N, arg, L, None, None)
        idx = np.zeros(n, np.int32)
        fptr = np.zeros(L + 1, np.int64)
        emu.k1emu_masks(pat, N, arg, L, idx.ctypes.data, fptr.ctypes.data)
        assert np.array_equal(idx, Po.idx) and np.array_equal(fptr, Po.frame_ptr)


@pytest.mark.parametrize("N", SIDES)
@pytest.mark.parametrize("qmin", ["1", "8"])
@pytest.mark.parametrize("pat,arg", MASKS)
def test_stream_tables_cover_every_sample_once_sizes(emu, N, pat, arg, qmin, monkeypatch):
    """Every sample of every frame sits in exactly one work item of its own k-space row, the N threads hold at most one item each,
    items carry at least one sample (cnt == 0 is the only "no item" mark), and the row mask names exactly the rows with samples:
    bit a of entry b is row R a + b, R = N / 16."""
    monkeypatch.setenv("QMRI_K1_QMIN", qmin)
    C, R = 10, N // 16
    Po = oracle_op(N, pat, C)
    itA = np.zeros((C, N), np.uint32)
    itB = np.zeros((C, N), np.uint32)
    ent = np.zeros(max(Po.nmeas, 1), np.uint32)
    rowmask = np.zeros((C, 16), np.uint16)
    assert emu.k1emu_stream_tables(N, pat, arg, C, itA.ctypes.data, itB.ctypes.data, ent.ctypes.data, rowmask.ctypes.data) == Po.nmeas
    for c in range(C):
        f0, f1 = int(Po.frame_ptr[c]), int(Po.frame_ptr[c + 1])
        k = np.asarray(Po.idx[f0:f1])
        seen = np.zeros(f1 - f0, np.int64)
        primaries = {}
        for tid in range(N):
            A, B = int(itA[c, tid]), int(itB[c, tid])
            k1, cnt, start = A & 0xff, (A >> 8) & 0xff, A >> 16
            if cnt == 0:
                assert A == 255 and B == 0
                continue
            assert cnt <= 64 and k1 < N
            slot = B & 0xff
            if slot == 0:
                assert k1 not in primaries
                primaries[k1] = tid
            for e in ent[f0 + start: f0 + start + cnt]:
                j, k2 = int(e) & 0xffff, int(e) >> 16
                assert k[j] == k1 + N * k2
                seen[j] += 1
        assert np.all(seen == 1)
        rows = np.unique(k % N)
        assert sorted(primaries) == list(rows)
        want = np.zeros(16, np.uint16)
        for r in rows:
            want[r % R] |= 1 << (r // R)
        assert np.array_equal(rowmask[c], want)


@pytest.mark.parametrize("N", SIDES)
@pytest.mark.parametrize("pat,arg,qmin", [(0, 771.0, "8"), (1, 1 / 65, "8"), (0, 771.0, "1")])  # qmin 1: many overflow partials
def test_k1_stream_arithmetic_all_modes_sizes(emu, N, pat, arg, qmin, monkeypatch):
    monkeypatch.setenv("QMRI_K1_QMIN", qmin)
    C = 3
    F = sampling.FOperator(oracle_op(N, pat, C))
    n = F.P.nmeas
    rng = np.random.default_rng(N)
    z = rng.standard_normal((N, N, C)) + 1j * rng.standard_normal((N, N, C))
    zr, zi = planar(z)
    yout = np.zeros((n, 2), np.float32)
    assert emu.k1emu_run_n(N, 2, pat, arg, C, 1, P(zr), P(zi), None, None, 0.05, None, None, P(yout), None) == n
    assert rel_l2(yout[:, 0] + 1j * yout[:, 1], F.forward(z)) < 1e-6
    y = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    y32 = np.stack([y.real, y.imag], 1).astype(np.float32)
    ore, oim = np.zeros_like(zr), np.zeros_like(zr)
    emu.k1emu_run_n(N, 3, pat, arg, C, 1, None, None, None, P(y32), 0.05, P(ore), P(oim), None, None)
    assert rel_l2(unplanar(ore, oim), F.adjoint(y)) < 1e-6
    mm = np.zeros(2, np.float32)
    emu.k1emu_run_n(N, 1, pat, arg, C, 1, P(zr), P(zi), None, P(y32), 0.05, P(ore), P(oim), None, P(mm))
    xe = xupdate_exact(F, y, z, 0.05)
    assert rel_l2(unplanar(ore, oim), xe) < 1e-6
    assert abs(mm[0] - xe.real.min()) < 1e-5 and abs(mm[1] - xe.real.max()) < 1e-5
    v = rng.standard_normal((N, N, C))
    vr, _ = planar(v + 0j)
    emu.k1emu_run_n(N, 0, pat, arg, C, 1, P(zr), P(zi), P(vr), P(y32), 0.05, P(ore), P(oim), None, P(mm))
    x = xupdate_exact(F, y, 2 * v - z, 0.05)
    assert rel_l2(unplanar(ore, oim), x + (z - v)) < 1e-6   # w' = x + u, u = w - v


@pytest.mark.parametrize("N", [128, 144, 176, 208, 240])
def test_other_sides_stay_unsupported(emu, N):
    """128 and the odd-R sides (144, 176, 208, 240) have no streaming-kernel instance."""
    z = np.zeros((1, N, N), np.float32)
    assert emu.k1emu_run_n(N, 3, 0, 771.0, 1, 1, None, None, None, None, 0.05, P(z), P(z), None, None) == -2
