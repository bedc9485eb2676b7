"""Test-side reference for the density and current Fourier modes, the checker of the GPU recorder mdqt_modes_*.

A plain restatement of the definitions with numpy, written long-hand and independent of the engine's fixed-point phase: for the
integer vector n and k = 2 pi n / L,
    rho_k = sum_i exp(i k.r_i),    j_k = sum_i v_i exp(i k.r_i),
with the phase taken as 2 pi ((n.r / L) mod 1) in np.longdouble, and cos, sin and the sums in np.longdouble. A record of one vector is
the 8 reals Re rho, Im rho, Re j_x, Im j_x, Re j_y, Im j_y, Re j_z, Im j_z. The correlations over T records, with khat = n / |n|,
j_L = khat.j and j_T = j - khat j_L, are
    F(k, t)   = 1/(N (T - t))   sum_{s < T - t} Re[rho(s) rho*(s + t)]
    C_L(k, t) = 1/(N (T - t))   sum_{s < T - t} Re[j_L(s) j_L*(s + t)]
    C_T(k, t) = 1/(2 N (T - t)) sum_{s < T - t} Re[j_T(s).j_T*(s + t)]"""
import numpy as np

LD = np.longdouble
TWO_PI = 2 * np.arccos(LD(-1))


def modes(R, V, L, nvec):
    """(values, scales), each [K][8]: the record of the vectors nvec [K][3] for positions R and velocities V [3][n]; scales = the
    sums of |w_i| of each component (w_i = 1 for rho, v_ia for j_a), for tolerances."""
    R = np.asarray(R, dtype=np.float64)
    V = np.asarray(V, dtype=np.float64)
    nvec = np.asarray(nvec, dtype=np.int64)
    frac = R.astype(LD) / LD(L)                       # [3][n]
    vals = np.zeros((len(nvec), 8))
    scales = np.zeros((len(nvec), 8))
    absV = np.abs(V).sum(axis=1)
    for q, n in enumerate(nvec):
        x = (LD(int(n[0])) * frac[0] + LD(int(n[1])) * frac[1] + LD(int(n[2])) * frac[2]) % LD(1)
        phase = TWO_PI * x
        c, s = np.cos(phase), np.sin(phase)
        vals[q, 0], vals[q, 1] = c.sum(), s.sum()
        scales[q, 0:2] = R.shape[1]
        for a in range(3):
            v = V[a].astype(LD)
            vals[q, 2 + 2 * a], vals[q, 3 + 2 * a] = (v * c).sum(), (v * s).sum()
            scales[q, 2 + 2 * a:4 + 2 * a] = absV[a]
    return vals, scales


def complex_modes(rec):
    """rho [..][T] and j [..][3][T] as complex arrays from records [..][8][T]."""
    rec = np.asarray(rec)
    rho = rec[..., 0, :] + 1j * rec[..., 1, :]
    j = rec[..., 2::2, :] + 1j * rec[..., 3::2, :]
    return rho, j


def _corr(a, n):
    """1/(n (T - t)) sum_{s < T - t} Re[a(s) . a*(s + t)] of complex series a [c][T], summed over the c components."""
    T = a.shape[-1]
    out = np.zeros(T)
    for t in range(T):
        out[t] = (a[:, :T - t] * np.conj(a[:, t:])).real.sum() / (n * (T - t))
    return out


def correlations(rec, n, nvec):
    """(F, C_L, C_T), each [K][T], of the records [K][8][T] of one trajectory of n ions."""
    rho, j = complex_modes(rec)
    nvec = np.asarray(nvec, dtype=np.float64)
    K = len(nvec)
    F, CL, CT = (np.zeros((K, rec.shape[-1])) for _ in range(3))
    for q in range(K):
        khat = nvec[q] / np.sqrt((nvec[q] ** 2).sum())
        jl = (khat[:, None] * j[q]).sum(axis=0)
        jt = j[q] - khat[:, None] * jl[None, :]
        F[q] = _corr(rho[q][None, :], n)
        CL[q] = _corr(jl[None, :], n)
        CT[q] = _corr(jt, n) / 2
    return F, CL, CT
