"""Test-side reference for the heat (energy) current, the checker of the GPU recorder mdqt_heat_*.

A plain restatement of the definitions with numpy, written long-hand and independent of the engine's formulation: ordered pairs
i != j, the reference's minimum image d = r_i - r_j, d -= L round(d / L) (C's round: halves away from zero), r = sqrt(d.d), only
0 < r < rcut, phi(r) = exp(-kappa r) / r and the pair scalar of the forces f(r) = (1/r + kappa) exp(-kappa r) / r^2 (F_i = sum_j d f).
In engine units (unit mass), with phi_i = sum_{j != i} phi(r_ij):
    J_kin,a = 1/2 sum_i |v_i|^2 v_ia      J_pot,a = 1/2 sum_i phi_i v_ia      J_vir,a = 1/2 sum_i sum_{j != i} d_a f (d.v_i)
    P_a = sum_i v_ia      E_kin = 1/2 sum_i |v_i|^2      E_pot = 1/2 sum_i phi_i      tr W = 1/2 sum_i sum_{j != i} f r^2
Row blocks keep the memory at O(block x N), so N = 20000 (4e8 ordered pairs) takes some seconds."""
import numpy as np


def _round_half_away(x):
    return np.sign(x) * np.floor(np.abs(x) + 0.5)


def heat(R, V, L, kappa, rcut, block=128):
    """(values, scales): values = the 15 numbers of a record (J_kin, J_pot, J_vir, P, E_kin, E_pot, tr W); scales = the sums of
    |terms| of each (for tolerances; for J_vir the terms d_a d_b f v_ib that the contraction d (d.v) f adds). R and V are [3][n]."""
    R = np.asarray(R, dtype=np.float64)
    V = np.asarray(V, dtype=np.float64)
    n = R.shape[1]
    vals, scales = np.zeros(15), np.zeros(15)
    e = 0.5 * (V * V).sum(axis=0)
    for a in range(3):
        vals[a], scales[a] = (e * V[a]).sum(), np.abs(e * V[a]).sum()
        vals[9 + a], scales[9 + a] = V[a].sum(), np.abs(V[a]).sum()
    vals[12] = scales[12] = e.sum()
    phi = np.zeros(n)
    for i0 in range(0, n, block):
        i1 = min(n, i0 + block)
        d = R[:, i0:i1, None] - R[:, None, :]  # rows i of this block against all columns j
        d -= L * _round_half_away(d / L)
        r = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
        inside = (r > 0) & (r < rcut)  # also drops the self pair j = i
        rs = np.where(inside, r, 1.0)
        ex = np.exp(-kappa * rs)
        ph = np.where(inside, ex / rs, 0.0)
        f = np.where(inside, (1.0 / rs + kappa) * ex / (rs * rs), 0.0)
        phi[i0:i1] = ph.sum(axis=1)
        v = V[:, i0:i1, None]
        dv = d[0] * v[0] + d[1] * v[1] + d[2] * v[2]
        dv_abs = np.abs(d[0] * v[0]) + np.abs(d[1] * v[1]) + np.abs(d[2] * v[2])
        for a in range(3):
            vals[6 + a] += 0.5 * (d[a] * f * dv).sum()
            scales[6 + a] += 0.5 * (np.abs(d[a]) * f * dv_abs).sum()
        t = 0.5 * f * (r * r)
        vals[14] += t.sum()
        scales[14] += t.sum()
    for a in range(3):
        vals[3 + a] = 0.5 * (phi * V[a]).sum()
        scales[3 + a] = 0.5 * np.abs(phi * V[a]).sum()
    vals[13] = scales[13] = 0.5 * phi.sum()
    return vals, scales


def heat_flux(rec, n):
    """J_q = J_kin + J_pot + J_vir - hbar P of records [..][15][T] of n ions, hbar the records' mean enthalpy per ion: [..][3][T]."""
    rec = np.asarray(rec)
    h = rec[..., 12, :] + rec[..., 13, :] + (2 * rec[..., 12, :] + rec[..., 14, :]) / 3.0
    hbar = h.mean(axis=-1) / n
    return rec[..., 0:3, :] + rec[..., 3:6, :] + rec[..., 6:9, :] - np.asarray(hbar)[..., None, None] * rec[..., 9:12, :]


def autocorr(J):
    """C(t) = 1/(3 (T - t)) sum_a sum_{j < T - t} J_a(j) J_a(j + t) of series [3][T], and its scale (the same sums of |products|)."""
    T = J.shape[-1]
    c = np.array([(J[:, :T - t] * J[:, t:]).sum() / (3 * (T - t)) for t in range(T)])
    s = np.array([np.abs(J[:, :T - t] * J[:, t:]).sum() / (3 * (T - t)) for t in range(T)])
    return c, s
