"""CPU suite: the test-side heat-current reference (tests/heat_reference.py), the checker of the GPU heat recorder, against a scalar
loop over ordered pairs, a two-ion case in closed form, the identities for uniform velocities (with tests/stress_reference.py), and
energy continuity along a velocity-Verlet trajectory of an isolated cluster, which pins the sign and the factors of 1/2."""
import math

import numpy as np
import pytest

import heat_reference
import stress_reference

KAPPA = 0.5


def _md_box(n):
    """L of the MD program: n ions in units of the Wigner-Seitz radius (mdqt_params_md, MD:73)."""
    return (n * 4.0 * math.pi / 3.0) ** (1.0 / 3.0)


def _scalar_heat(R, V, L, kappa, rcut):
    """The definitions as a scalar Python loop over ordered pairs (math.* only, correctly rounded sums)."""
    n = R.shape[1]
    phi = [0.0] * n
    jvir = [[] for _ in range(3)]
    trw = []
    for i in range(n):
        terms = []
        for j in range(n):
            if j == i:
                continue
            d = [R[c][i] - R[c][j] for c in range(3)]
            d = [x - L * math.copysign(math.floor(abs(x / L) + 0.5), x) for x in d]
            r = math.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
            if 0 < r < rcut:
                terms.append(math.exp(-kappa * r) / r)
                f = (1.0 / r + kappa) * math.exp(-kappa * r) / (r * r)
                dv = d[0] * V[0][i] + d[1] * V[1][i] + d[2] * V[2][i]
                for a in range(3):
                    jvir[a].append(0.5 * d[a] * f * dv)
                trw.append(0.5 * f * r * r)
        phi[i] = math.fsum(terms)
    e = [0.5 * (V[0][i] ** 2 + V[1][i] ** 2 + V[2][i] ** 2) for i in range(n)]
    out = [math.fsum(e[i] * V[a][i] for i in range(n)) for a in range(3)]
    out += [0.5 * math.fsum(phi[i] * V[a][i] for i in range(n)) for a in range(3)]
    out += [math.fsum(jvir[a]) for a in range(3)]
    out += [math.fsum(V[a][i] for i in range(n)) for a in range(3)]
    out += [math.fsum(e), 0.5 * math.fsum(phi), math.fsum(trw)]
    return np.array(out)


def test_reference_matches_a_scalar_loop_at_120_random_ions():
    rng = np.random.default_rng(12)
    n = 120
    L = _md_box(n)
    R = rng.uniform(-0.3 * L, 1.3 * L, size=(3, n))  # unwrapped coordinates too: the minimum image handles them
    V = rng.normal(size=(3, n)) * 0.6
    got, scale = heat_reference.heat(R, V, L, KAPPA, L / 2, block=37)  # a block size that does not divide n
    want = _scalar_heat(R, V, L, KAPPA, L / 2)
    assert np.all(np.abs(got - want) <= 1e-13 * scale), np.abs(got - want) / scale
    assert np.all(scale > 0)


def test_two_ions_in_closed_form():
    L = 10.0
    R = np.array([[1.0, 2.5], [1.0, 1.75], [1.0, 0.5]])  # d = r_0 - r_1 = (-1.5, -0.75, 0.5): exact in binary
    V = np.array([[0.5, -0.25], [0.125, 1.0], [-2.0, 0.75]])
    got, _ = heat_reference.heat(R, V, L, KAPPA, L / 2)
    d = R[:, 0] - R[:, 1]
    r = math.sqrt(d @ d)
    phi = math.exp(-KAPPA * r) / r
    f = (1.0 / r + KAPPA) * math.exp(-KAPPA * r) / (r * r)
    v0, v1 = V[:, 0], V[:, 1]
    want = np.concatenate([0.5 * (v0 @ v0) * v0 + 0.5 * (v1 @ v1) * v1,  # J_kin
                           0.5 * phi * (v0 + v1),                        # J_pot: phi_0 = phi_1 = phi
                           0.5 * d * f * (d @ (v0 + v1)),                 # J_vir: the pair (1, 0) has -d, so d f (d.v_1) again
                           v0 + v1,                                      # P
                           [0.5 * (v0 @ v0 + v1 @ v1), phi, f * r * r]])
    np.testing.assert_allclose(got, want, rtol=1e-15, atol=0)


def test_pair_beyond_the_cutoff_contributes_nothing():
    L = 10.0
    R = np.array([[0.0, 0.45 * L], [0.0, 0.45 * L], [0.0, 0.0]])  # r = 0.64 L > rcut = L/2
    V = np.array([[0.5, -0.25], [0.0, 1.0], [2.0, 0.0]])
    got, _ = heat_reference.heat(R, V, L, KAPPA, L / 2)
    assert np.all(got[3:9] == 0.0) and got[13] == 0.0 and got[14] == 0.0


def test_uniform_velocities():
    """V = c for every ion: J_pot = E_pot c, J_vir = W c with W the virial tensor of stress_reference, J_kin = |c|^2/2 N c, P = N c."""
    rng = np.random.default_rng(5)
    n = 300
    L = _md_box(n)
    R = rng.uniform(0, L, size=(3, n))
    c = np.array([0.3, -0.7, 1.1])
    V = np.repeat(c[:, None], n, axis=1)
    got, scale = heat_reference.heat(R, V, L, KAPPA, L / 2)
    W6 = stress_reference.stress(R, V, L, KAPPA, L / 2)[0][6:]
    W = np.array([[W6[0], W6[3], W6[4]], [W6[3], W6[1], W6[5]], [W6[4], W6[5], W6[2]]])
    assert np.allclose(got[3:6], got[13] * c, rtol=1e-13, atol=0)
    assert np.all(np.abs(got[6:9] - W @ c) <= 1e-12 * scale[6:9])
    assert got[14] == pytest.approx(np.trace(W), rel=1e-13)
    assert np.allclose(got[0:3], 0.5 * (c @ c) * n * c, rtol=1e-13, atol=0)
    assert np.allclose(got[9:12], n * c, rtol=1e-13, atol=0)


def _phi_and_forces(R, kappa):
    """Per-ion phi_i and F_i of an isolated cluster (all pairs, no images)."""
    d = R[:, :, None] - R[:, None, :]
    r = np.sqrt((d * d).sum(axis=0))
    np.fill_diagonal(r, 1.0)
    ph = np.exp(-kappa * r) / r
    f = (1.0 / r + kappa) * np.exp(-kappa * r) / (r * r)
    np.fill_diagonal(ph, 0.0)
    np.fill_diagonal(f, 0.0)
    return ph.sum(axis=1), (d * f).sum(axis=2)


def _energy_moment(R, V, kappa):
    """sum_i r_i e_i with e_i = |v_i|^2 / 2 + phi_i / 2."""
    phi, _ = _phi_and_forces(R, kappa)
    return (R * (0.5 * (V * V).sum(axis=0) + 0.5 * phi)).sum(axis=1)


def _verlet(R, V, kappa, h, nsteps):
    R, V = R.copy(), V.copy()
    F = _phi_and_forces(R, kappa)[1]
    for _ in range(nsteps):
        V += 0.5 * h * F
        R += h * V
        F = _phi_and_forces(R, kappa)[1]
        V += 0.5 * h * F
    return R, V


def test_energy_continuity():
    """d/dt sum_i r_i e_i = J_E for an isolated cluster: [sum r e](t + delta) - [sum r e](t), over delta, equals J_kin + J_pot + J_vir
    at t + delta/2 to O(delta^2). A box so large that no minimum image wraps, rcut = L/2 covering every pair; the trajectory is a
    velocity-Verlet one with steps of delta/64."""
    rng = np.random.default_rng(8)
    side = 5  # 125 ions on a jittered cubic lattice of spacing 1.6 (no close encounters)
    g = np.arange(side) * 1.6
    R0 = np.array(np.meshgrid(g, g, g, indexing="ij")).reshape(3, -1) + rng.uniform(-0.2, 0.2, size=(3, side ** 3))
    V0 = rng.normal(size=R0.shape) * 0.5
    L = 1000.0
    errs = []
    for delta in (0.04, 0.02):
        sub = 64
        Rm, Vm = _verlet(R0, V0, KAPPA, delta / sub, sub // 2)
        Re, Ve = _verlet(Rm, Vm, KAPPA, delta / sub, sub // 2)
        fd = (_energy_moment(Re, Ve, KAPPA) - _energy_moment(R0, V0, KAPPA)) / delta
        J = heat_reference.heat(Rm, Vm, L, KAPPA, L / 2)[0]
        JE = J[0:3] + J[3:6] + J[6:9]
        errs.append(np.abs(fd - JE).max() / np.abs(JE).max())
    assert errs[0] < 1e-4 and errs[1] < 3e-5, errs
    assert 3.0 < errs[0] / errs[1] < 5.0, errs  # second order in delta
