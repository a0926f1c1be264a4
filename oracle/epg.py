"""FISP-MRF dictionary oracle (test infrastructure): float64 restatements of the signal model of include/qmri.h.

    epg_fisp        complex128 extended phase graph with the whole state vector (orders 0..T) and Weigel's operators
    epg_fisp_real   the same recursion in three real numbers per order (F = i f), optionally on the live order window only
    bloch_fisp      isochromat Bloch simulation: 2T + 2 spins spread evenly over one dephasing cycle
    gram / temporal_basis / compress   the SVD compression of the dict struct, with the sign rule of the V columns

seq = {'flip_deg': [T], 'tr': [T], 'te': s, 'ti': s or None}.  T1, T2: arrays of atoms (any shape, flattened).
"""
import numpy as np


def _schedule(seq, T=None):
    flip = np.asarray(seq["flip_deg"], np.float64).reshape(-1)
    tr = np.asarray(seq["tr"], np.float64).reshape(-1)
    T = flip.size if T is None else int(T)
    return np.deg2rad(flip[:T]), tr[:T], float(seq["te"]), seq.get("ti")


def _z0(T1, ti):
    return np.ones_like(T1) if ti is None else 1.0 - 2.0 * np.exp(-float(ti) / T1)


def epg_fisp(T1, T2, seq, T=None):
    """Complex fingerprints i F+_0 e^{-te/T2}, [n x T] complex128 (the imaginary part is zero by the model)."""
    T1 = np.asarray(T1, np.float64).reshape(-1)
    T2 = np.asarray(T2, np.float64).reshape(-1)
    a, tr, te, ti = _schedule(seq, T)
    n, T = T1.size, a.size
    Fp = np.zeros((n, T + 1), np.complex128)
    Fm = np.zeros_like(Fp)
    Z = np.zeros_like(Fp)
    Z[:, 0] = _z0(T1, ti)
    out = np.empty((n, T), np.complex128)
    ete = np.exp(-te / T2)
    for i in range(T):
        c2, s2, sa, ca = np.cos(a[i] / 2) ** 2, np.sin(a[i] / 2) ** 2, np.sin(a[i]), np.cos(a[i])
        # T(alpha, phi = 0), Weigel (2015) eq. 15
        Fp, Fm, Z = (c2 * Fp + s2 * Fm - 1j * sa * Z,
                     s2 * Fp + c2 * Fm + 1j * sa * Z,
                     -0.5j * sa * Fp + 0.5j * sa * Fm + ca * Z)
        out[:, i] = 1j * Fp[:, 0] * ete
        E1, E2 = np.exp(-tr[i] / T1), np.exp(-tr[i] / T2)
        Fp = Fp * E2[:, None]
        Fm = Fm * E2[:, None]
        Z = Z * E1[:, None]
        Z[:, 0] += 1.0 - E1
        Fp = np.concatenate([np.zeros((n, 1)), Fp[:, :-1]], axis=1)
        Fm = np.concatenate([Fm[:, 1:], np.zeros((n, 1))], axis=1)
        Fp[:, 0] = np.conj(Fm[:, 0])
    return out


def live_orders(i, T):
    """Highest order that can still reach order 0 before the last readout, around pulse i: before the pulse min(i, T-1-i),
    after its shift min(i+1, T-2-i).  Work count of the simulation: sum_i (live_orders(i, T) + 1)."""
    return max(min(i, T - 1 - i), min(i + 1, T - 2 - i))


def epg_fisp_real(T1, T2, seq, T=None, window=True):
    """Real fingerprints [n x T] float64 from the substitution F = i f: f+' = c2 f+ + s2 f- - sin(a) Z,
    f-' = s2 f+ + c2 f- + sin(a) Z, Z' = sin(a)/2 (f+ - f-) + cos(a) Z, sample -f+_0 e^{-te/T2}, f+_0 = -f-_0 after the shift.
    window=True: orders above the live window are dropped (set to zero) after every pulse."""
    T1 = np.asarray(T1, np.float64).reshape(-1)
    T2 = np.asarray(T2, np.float64).reshape(-1)
    a, tr, te, ti = _schedule(seq, T)
    n, T = T1.size, a.size
    fp = np.zeros((n, T + 1))
    fm = np.zeros_like(fp)
    z = np.zeros_like(fp)
    z[:, 0] = _z0(T1, ti)
    out = np.empty((n, T))
    ete = np.exp(-te / T2)
    for i in range(T):
        c2, s2, sa, ca = np.cos(a[i] / 2) ** 2, np.sin(a[i] / 2) ** 2, np.sin(a[i]), np.cos(a[i])
        fp, fm, z = c2 * fp + s2 * fm - sa * z, s2 * fp + c2 * fm + sa * z, 0.5 * sa * (fp - fm) + ca * z
        out[:, i] = -fp[:, 0] * ete
        E1, E2 = np.exp(-tr[i] / T1), np.exp(-tr[i] / T2)
        fp *= E2[:, None]
        fm *= E2[:, None]
        z *= E1[:, None]
        z[:, 0] += 1.0 - E1
        fp = np.concatenate([np.zeros((n, 1)), fp[:, :-1]], axis=1)
        fm = np.concatenate([fm[:, 1:], np.zeros((n, 1))], axis=1)
        fp[:, 0] = -fm[:, 0]
        if window:
            w = min(i + 1, T - 2 - i)
            fp[:, w + 1:] = 0.0
            fm[:, w + 1:] = 0.0
            z[:, w + 1:] = 0.0
    return out


def bloch_fisp(T1, T2, seq, T=None):
    """Isochromat simulation, [n x T] complex128: mean transverse magnetisation M_x + i M_y of 2T + 2 spins whose dephasing
    angles per TR are spread evenly over [0, 2 pi), sampled after each pulse and multiplied by e^{-te/T2}.  The RF pulse is a
    rotation by alpha about +x (M_y' = M_y cos a - M_z sin a), so the mean is F+_0 of the EPG: the EPG sample i F+_0 is
    1j times this (no fitted factor)."""
    T1 = np.asarray(T1, np.float64).reshape(-1)
    T2 = np.asarray(T2, np.float64).reshape(-1)
    a, tr, te, ti = _schedule(seq, T)
    n, T = T1.size, a.size
    N = 2 * T + 2
    phi = 2 * np.pi * np.arange(N) / N
    cph, sph = np.cos(phi)[None, :], np.sin(phi)[None, :]
    Mx = np.zeros((n, N))
    My = np.zeros((n, N))
    Mz = np.repeat(_z0(T1, ti)[:, None], N, axis=1)
    out = np.empty((n, T), np.complex128)
    ete = np.exp(-te / T2)
    for i in range(T):
        ca, sa = np.cos(a[i]), np.sin(a[i])
        My, Mz = My * ca - Mz * sa, My * sa + Mz * ca
        out[:, i] = (Mx.mean(axis=1) + 1j * My.mean(axis=1)) * ete
        E1, E2 = np.exp(-tr[i] / T1)[:, None], np.exp(-tr[i] / T2)[:, None]
        Mx, My = Mx * E2, My * E2
        Mz = Mz * E1 + (1.0 - E1)
        Mx, My = Mx * cph - My * sph, Mx * sph + My * cph
    return out


def gram(sig):
    s = np.asarray(sig, np.float64)
    return s.T @ s


def temporal_basis(G, C):
    """Top-C eigenvectors of G, descending eigenvalues; each column's entry of largest magnitude positive (lowest index on a
    tie).  Returns (V [T x C], eigenvalues [T] descending)."""
    w, U = np.linalg.eigh(np.asarray(G, np.float64))
    order = np.argsort(w)[::-1]
    V = U[:, order[:C]].copy()
    for c in range(C):
        p = int(np.argmax(np.abs(V[:, c])))
        if V[p, c] < 0:
            V[:, c] = -V[:, c]
    return V, w[order]


def compress(sig, V):
    """D = d V / |d V|, normD = |d V| in float64 (the conventions of benchdata.make_dictionary / oracle/synth.py)."""
    Dc = np.asarray(sig, np.float64) @ np.asarray(V, np.float64)
    nd = np.linalg.norm(Dc, axis=1)
    return Dc / nd[:, None], nd
