"""Test-side reference for the pressure (stress) tensor, the checker of the GPU recorder mdqt_stress_*.

A plain restatement of the definitions with numpy, written long-hand and independent of the engine's formulation: unordered pairs
i < j, the reference's minimum image d -= L round(d / L) (C's round: halves away from zero), r = sqrt(d.d), and the pair scalar of the
forces f(r) = (1/r + kappa) exp(-kappa r) / r^2, so that F_i = sum_j d f. In engine units (unit mass), not divided by the volume:
    K_ab = sum_i v_a v_b,   W_ab = sum_{i<j, 0<r<rcut} d_a d_b f(r),   ab = xx, yy, zz, xy, xz, yz.
Row blocks keep the memory at O(block x N), so N = 20000 (2e8 pairs) takes a few seconds."""
import numpy as np

AB = ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))


def _round_half_away(x):
    return np.sign(x) * np.floor(np.abs(x) + 0.5)


def stress(R, V, L, kappa, rcut, block=256):
    """(values, scales): values = [K_xx .. K_yz, W_xx .. W_yz]; scales = the sums of |terms| of each component (for tolerances).
    R and V are [3][n]."""
    R = np.asarray(R, dtype=np.float64)
    V = np.asarray(V, dtype=np.float64)
    n = R.shape[1]
    vals, scales = np.zeros(12), np.zeros(12)
    for q, (a, b) in enumerate(AB):
        t = V[a] * V[b]
        vals[q], scales[q] = t.sum(), np.abs(t).sum()
    for i0 in range(0, n - 1, block):
        i1 = min(n - 1, i0 + block)
        d = R[:, i0:i1, None] - R[:, None, i0:]  # rows i of this block against columns j >= i0
        upper = np.arange(i0, i1)[:, None] < np.arange(i0, n)[None, :]  # pairs i < j only
        d -= L * _round_half_away(d / L)
        r = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
        inside = upper & (r > 0) & (r < rcut)
        d, r = d[:, inside], r[inside]
        f = (1.0 / r + kappa) * np.exp(-kappa * r) / (r * r)
        for q, (a, b) in enumerate(AB):
            t = d[a] * d[b] * f
            vals[6 + q] += t.sum()
            scales[6 + q] += np.abs(t).sum()
    return vals, scales
