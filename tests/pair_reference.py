"""Test-side per-ion reference of the all-pairs loop, with the error scales that the per-ion bound of the pair kernels needs.

The pair kernels (k_pairs_items, k_pairs) sum, for every ion row i over all j, the force F_i = sum_j d f(r), the potential
phi_i = sum_j exp(-kappa r)/r and the tensor T_i,ab = sum_j d_a d_b f(r), with d the minimum image of r_i - r_j, only 0 < r < rcut,
f(r) = (1/r + kappa) exp(-kappa r)/r^2. Every observable of the loop is a fixed function of these row sums: the forces, the
potential energy 1/(2 n) sum_i phi_i, the virial W = 1/2 sum_i T_i and the pair parts of the heat current (1/2 sum_i phi_i v_i,
1/2 sum_i T_i v_i, 1/2 sum_i phi_i, 1/2 sum_i tr T_i). tests/stress_reference.py and tests/heat_reference.py state those per
trajectory; this module keeps them per ion, and next to every sum it keeps
    S = the sum of |terms|, which scales the rounding of any summation order, and
    Q = sum over terms of sum_b |dt/dd_b| delta, what a per-component error delta of the separation d moves it by.
The minimum image of positions in [0, L] is exact until its final rounding: x_i - x_j by TwoSum (head and exact tail), the image
shift by Sterbenz' lemma, then one rounding of head + tail -- relative, not L 2^-53 as for a plain difference across the boundary.
Row blocks keep the memory at O(block x n); the blocks are spread over threads (numpy releases the GIL in the array operations).

bound() is the first-order worst-case error of the device against these sums. mp_pair() is the 50-digit pair function."""
import math
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

U = 2.0 ** -53                # unit roundoff of binary64
CP = 16                       # rounding of one pair term on the device, in units of U (DESIGN section 3: the pair arithmetic)
CR = 3                        # relative error of the device's r, in units of U: exp(-kappa r) multiplies it by kappa r
AB = ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))


def conversion_delta(L):
    """Largest error of one component of the separation the pair kernels use, against the exact minimum image of the double
    positions: each to_fixed (mdqt_fixed.cuh) rounds x/L to the 2^-62 grid twice (high and low part, 1/2 unit each), so a difference
    of two conversions is off by at most 2 L 2^-62."""
    return 2.0 * L * 2.0 ** -62


def ion_sums(R, L, kappa, rcut, rows=None, delta=None, block=48, workers=None):
    """Row sums of one trajectory (R: [3][n]) for the ions `rows` (default: all), each with its S and Q:
    F, SF, QF [3][m]; T, ST, QT [6][m] (ab = xx yy zz xy xz yz); phi, Qphi [m] (phi's S is phi itself).
    delta: per-component separation error for Q (default conversion_delta(L))."""
    R = np.ascontiguousarray(R, dtype=np.float64)
    if not (R.min() >= 0.0 and R.max() <= L):
        raise ValueError("ion_sums takes wrapped positions, in [0, L]")
    n = R.shape[1]
    rows = np.arange(n) if rows is None else np.asarray(rows)
    m = len(rows)
    delta = conversion_delta(L) if delta is None else delta
    out = {k: np.zeros((c, m)) for k, c in (("F", 3), ("SF", 3), ("QF", 3), ("T", 6), ("ST", 6), ("QT", 6))}
    out["phi"], out["Qphi"] = np.zeros(m), np.zeros(m)

    def one(k0):
        k1 = min(m, k0 + block)
        a, b = R[:, rows[k0:k1], None], -R[:, None, :]
        h = a + b                                   # TwoSum: h + t = x_i - x_j exactly
        a1 = h - b
        t = (a - a1) + (b - (h - a1))
        h -= L * np.rint(h / L)                     # exact: |h| in [L/2, L] when shifted
        d = h + t
        r = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
        inside = (r > 0) & (r < rcut)
        rs = np.where(inside, r, 1.0)
        ir = 1.0 / rs
        ex = np.where(inside, np.exp(-kappa * rs), 0.0)
        phi = ex * ir
        f = (ir + kappa) * ex * ir * ir
        dphi_r = ex * (ir + kappa) * ir * ir                                # |phi'| / r
        df_r = ex * (3 * ir * ir + 3 * kappa * ir + kappa * kappa) * ir ** 3  # |f'| / r
        ad = np.abs(d)
        l1 = ad[0] + ad[1] + ad[2]
        for a in range(3):
            t = f * d[a]
            out["F"][a, k0:k1] = t.sum(axis=1)
            out["SF"][a, k0:k1] = np.abs(t).sum(axis=1)
            out["QF"][a, k0:k1] = delta * (f + df_r * ad[a] * l1).sum(axis=1)
        for q, (a, b) in enumerate(AB):
            t = f * d[a] * d[b]
            out["T"][q, k0:k1] = t.sum(axis=1)
            out["ST"][q, k0:k1] = np.abs(t).sum(axis=1)
            out["QT"][q, k0:k1] = delta * (f * (ad[a] + ad[b]) + df_r * ad[a] * ad[b] * l1).sum(axis=1)
        out["phi"][k0:k1] = phi.sum(axis=1)
        out["Qphi"][k0:k1] = delta * (dphi_r * l1).sum(axis=1)

    with ThreadPoolExecutor(max_workers=workers or min(16, os.cpu_count() or 1)) as ex:
        list(ex.map(one, range(0, m, block)))
    return out


def records(s, V):
    """The pair-loop observables of one trajectory from its ion_sums over ALL its ions and its velocities V [3][n], each as
    (value, S, Q) arrays: epot (per ion), stress [12] (K, W of mdqt_stress_download) and heat [15] (mdqt_heat_download)."""
    V = np.asarray(V, dtype=np.float64)
    n = V.shape[1]
    av = np.abs(V)
    zero = np.zeros
    ep = (np.array([0.5 * s["phi"].sum() / n]), np.array([0.5 * s["phi"].sum() / n]), np.array([0.5 * s["Qphi"].sum() / n]))
    st = [zero(12), zero(12), zero(12)]
    for q, (a, b) in enumerate(AB):
        t = V[a] * V[b]
        st[0][q], st[1][q] = t.sum(), np.abs(t).sum()
        st[0][6 + q], st[1][6 + q], st[2][6 + q] = 0.5 * s["T"][q].sum(), 0.5 * s["ST"][q].sum(), 0.5 * s["QT"][q].sum()
    he = [zero(15), zero(15), zero(15)]
    e = 0.5 * (V * V).sum(axis=0)
    full = lambda M, q_of: np.array([M[q_of[a][b]] for a in range(3) for b in range(3)]).reshape(3, 3, -1)
    qi = ((0, 3, 4), (3, 1, 5), (4, 5, 2))
    Tm, STm, QTm = full(s["T"], qi), full(s["ST"], qi), full(s["QT"], qi)
    for a in range(3):
        he[0][a], he[1][a] = (e * V[a]).sum(), np.abs(e * V[a]).sum()
        he[0][3 + a], he[1][3 + a], he[2][3 + a] = (0.5 * (s["phi"] * V[a]).sum(), 0.5 * (s["phi"] * av[a]).sum(),
                                                    0.5 * (s["Qphi"] * av[a]).sum())
        he[0][6 + a] = 0.5 * sum((Tm[a, b] * V[b]).sum() for b in range(3))
        he[1][6 + a] = 0.5 * sum((STm[a, b] * av[b]).sum() for b in range(3))
        he[2][6 + a] = 0.5 * sum((QTm[a, b] * av[b]).sum() for b in range(3))
        he[0][9 + a], he[1][9 + a] = V[a].sum(), av[a].sum()
    he[0][12] = he[1][12] = e.sum()
    he[0][13] = he[1][13] = 0.5 * s["phi"].sum()
    he[2][13] = 0.5 * s["Qphi"].sum()
    he[0][14] = 0.5 * (s["T"][0] + s["T"][1] + s["T"][2]).sum()
    he[1][14] = 0.5 * (s["ST"][0] + s["ST"][1] + s["ST"][2]).sum()
    he[2][14] = 0.5 * (s["QT"][0] + s["QT"][1] + s["QT"][2]).sum()
    return {"epot": ep, "stress": tuple(st), "heat": tuple(he)}


def chain(jlen, nsplit, n, final=False):
    """m of the bound: the longest chain of additions a term meets on the device -- its row's j chunk, the chunk partials and, for
    the per-trajectory records (final=True), the row groups, the warp shuffle and the 256-thread trees (gcap + 13)."""
    return jlen + nsplit + (((n + 31) // 32) + 13 if final else 0)


def bound(S, Q, m, n, kappa_rcut, cp=CP):
    """|device - reference| <= (2 (cp + CR kappa rcut) + m + ceil(log2 n) + 4) u S + Q: cp u per term and the exp's condition kappa r
    times the relative error of r, once for the device and once for this module's float64 pair function (which rounds about as
    often), one u per addition of the device's chain m, numpy's pairwise sum (log2 n) and the final products (4 u)."""
    return (2 * (cp + CR * kappa_rcut) + m + math.ceil(math.log2(max(n, 2))) + 4) * U * np.asarray(S) + np.asarray(Q)


# ---- the 50-digit pair function ----------------------------------------------------------------------------------------------
def mp_pair(xi, xj, L, kappa, digits=50):
    """Exact minimum image d = (xi - xj) - L round((xi - xj)/L) of the double inputs (3-vectors) and, at `digits` digits,
    r, f(r) = (1/r + kappa) exp(-kappa r)/r^2 and phi(r) = exp(-kappa r)/r (f = phi = 0 at r = 0). Returns mpf values
    (d, r, f, phi, |f'(r)|, |phi'(r)|)."""
    import mpmath
    with mpmath.workdps(digits):
        Lm, km = mpmath.mpf(L), mpmath.mpf(kappa)
        d = []
        for a in range(3):
            x = mpmath.mpf(xi[a]) - mpmath.mpf(xj[a])
            q = x / Lm
            k = mpmath.floor(q + mpmath.mpf(0.5)) if q >= 0 else -mpmath.floor(-q + mpmath.mpf(0.5))
            d.append(x - Lm * k)
        r = mpmath.sqrt(d[0] ** 2 + d[1] ** 2 + d[2] ** 2)
        if r == 0:
            z = mpmath.mpf(0)
            return d, r, z, z, z, z
        e = mpmath.exp(-km * r)
        phi = e / r
        f = (1 / r + km) * e / r ** 2
        dphi = e * (1 / r ** 2 + km / r)
        df = e * (3 / r ** 4 + 3 * km / r ** 3 + km ** 2 / r ** 2)
        return d, r, f, phi, df, dphi


def probe_positions(L, rcut, B, grid, seed=0):
    """B two-ion trajectories [B][3][2], one pair each, for probing the pair function: the coincident pair; log-spaced r from
    1e-7 L to rcut along random directions; axis-aligned pairs; pairs across the periodic boundary and several box lengths apart
    (unwrapped); |d_a| = L/2 exactly; and (not on the grid) the cut-off band r = rcut (1 +- k 2^-52), k = 1..8, 16, 64.
    grid=True puts every coordinate on x = L m / 2^40, where the fixed-point separation is exact (L a power of two)."""
    rng = np.random.default_rng(seed)
    X = np.zeros((B, 3, 2))
    base = rng.uniform(0, L, size=(B, 3))
    dirs = rng.normal(size=(B, 3))
    dirs /= np.linalg.norm(dirs, axis=1)[:, None]
    r = np.exp(rng.uniform(np.log(1e-7 * L), np.log(rcut), size=B))
    k = 1
    X[0, :, :] = base[0][:, None]                                   # coincident pair
    # cut-off band: ion 0 at a random point, random direction; on the grid r = rcut exactly, along the axes
    band = [0] * 6 if grid else [s * kk for kk in (1, 2, 3, 4, 5, 6, 7, 8, 16, 64) for s in (1, -1)]
    for j, kk in enumerate(band):
        r[k + j] = rcut * (1 + kk * 2.0 ** -52)
        if grid:
            dirs[k + j] = np.eye(3)[j % 3] * (1 if j % 2 else -1)
    k_axis = k + len(band)
    for j in range(k_axis, k_axis + 96):                            # axis-aligned
        dirs[j] = np.eye(3)[j % 3] * (1 if j % 2 else -1)
    k_half = k_axis + 96
    for j in range(k_half, k_half + 24):                            # |d_a| = L/2 exactly, other components small or zero
        dirs[j] = 0.0
        r[j] = 0.0
    for j in range(1, B):
        X[j, :, 0] = base[j]
        X[j, :, 1] = base[j] + r[j] * dirs[j]
    for j in range(k_half, k_half + 24):
        a = j % 3
        X[j, a, 1] = X[j, a, 0] + (L / 2 if j % 2 else -L / 2)
        if j % 4 >= 2:
            X[j, (a + 1) % 3, 1] += rng.uniform(-0.3, 0.3) * L
    k_wrap = k_half + 24
    for j in range(k_wrap, k_wrap + 256):                           # unwrapped: shift one ion by -3 .. 3 box lengths per axis
        X[j, :, 1] += rng.integers(-3, 4, size=3) * L
    for j in range(k_wrap + 256, k_wrap + 384):                     # across the boundary: ion 0 near 0, ion 1 near L
        X[j, :, 0] = rng.uniform(0, 1e-3 * L, size=3)
        X[j, :, 1] = L - rng.uniform(0, 1e-3 * L, size=3) + rng.uniform(-1, 1, size=3) * r[j] / 2
    if grid:
        X = np.round(X * (2.0 ** 40 / L)) * (L / 2.0 ** 40)
    return X


PROBE_COLUMNS = {"forces": slice(0, 6), "epot": slice(6, 7), "stress": slice(7, 13), "heat": slice(13, 21)}


def mp_probe(X, V, L, kappa, rcuts, delta, digits=50):
    """The 50-digit values of what the device reports for the two-ion trajectories X [B][3][2] with velocities V [B][3][2]:
    columns F_0 (3), F_1 (3), Epotential() = phi/2, W (6), J_pot (3), J_vir (3), E_pot = phi, tr W = f r^2 (PROBE_COLUMNS).
    Returns hi, lo (the value as a double-double), S (sum of |terms|), Q (delta times the separation sensitivity), each [B][21],
    the exact r as a double, and per cut-off in `rcuts` the class of each pair: 1 inside (r <= rcut (1 - 8 2^-52)), 0 outside
    (r >= rcut (1 + 8 2^-52), r = rcut or r = 0), -1 in the band between."""
    import mpmath
    B = X.shape[0]
    hi, lo, S, Q = (np.zeros((B, 21)) for _ in range(4))
    rr = np.zeros(B)
    cls = {rc: np.zeros(B, dtype=int) for rc in rcuts}
    with mpmath.workdps(digits):
        eps = mpmath.mpf(2) ** -52 * 8
        for b in range(B):
            d, r, f, phi, df, dphi = mp_pair(X[b, :, 0], X[b, :, 1], L, kappa, digits)
            rr[b] = float(r)
            for rc in rcuts:
                rcm = mpmath.mpf(rc)
                cls[rc][b] = 0 if (r == 0 or r >= rcm * (1 + eps) or r == rcm) else (1 if r <= rcm * (1 - eps) else -1)
            v0, v1 = [mpmath.mpf(x) for x in V[b, :, 0]], [mpmath.mpf(x) for x in V[b, :, 1]]
            W = [d[a] * d[c] * f for a, c in AB]
            Wm = [[W[q] for q in row] for row in ((0, 3, 4), (3, 1, 5), (4, 5, 2))]
            vals = [f * d[a] for a in range(3)] + [-f * d[a] for a in range(3)] + [phi / 2] + W
            vals += [phi * (v0[a] + v1[a]) / 2 for a in range(3)]
            vals += [sum(Wm[a][c] * (v0[c] + v1[c]) for c in range(3)) / 2 for a in range(3)]
            vals += [phi, f * r * r]
            ad = [abs(x) for x in d]
            l1 = ad[0] + ad[1] + ad[2]
            rinv = 1 / r if r != 0 else mpmath.mpf(0)
            qF = [delta * (f + df * ad[a] * l1 * rinv) for a in range(3)]
            qphi = delta * dphi * l1 * rinv
            qW = [delta * (f * (ad[a] + ad[c]) + df * ad[a] * ad[c] * l1 * rinv) for a, c in AB]
            qWm = [[qW[q] for q in row] for row in ((0, 3, 4), (3, 1, 5), (4, 5, 2))]
            sv = [abs(v0[a]) + abs(v1[a]) for a in range(3)]
            scal = [abs(x) for x in vals[:13]] + [phi * sv[a] / 2 for a in range(3)]
            scal += [sum(abs(Wm[a][c]) * sv[c] for c in range(3)) / 2 for a in range(3)] + [phi, f * r * r]
            qs = qF + qF + [qphi / 2] + qW + [qphi * sv[a] / 2 for a in range(3)]
            qs += [sum(qWm[a][c] * sv[c] for c in range(3)) / 2 for a in range(3)] + [qphi, qW[0] + qW[1] + qW[2]]
            for k in range(21):
                h = float(vals[k])
                hi[b, k], lo[b, k] = h, float(vals[k] - h)
                S[b, k], Q[b, k] = float(scal[k]), float(qs[k])
    return hi, lo, S, Q, rr, cls
