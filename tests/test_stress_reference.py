"""CPU suite: the test-side pressure-tensor reference (tests/stress_reference.py, K_ab = sum_i v_a v_b, W_ab = sum_{i<j, 0<r<rcut}
d_a d_b f(r)), the checker of the GPU stress recorder, against a scalar pair loop, hand-made pairs, the virial scaling identity with
the oracle's potential energy, and the symmetry of a cubic lattice."""
import math

import numpy as np
import pytest

import stress_reference

KAPPA = 0.5


def _md_box(n):
    """L of the MD program: n ions in units of the Wigner-Seitz radius (mdqt_params_md, MD:73)."""
    return (n * 4.0 * math.pi / 3.0) ** (1.0 / 3.0)


def _scalar_stress(R, V, L, kappa, rcut):
    """The definitions as a scalar Python loop over unordered pairs (math.* only)."""
    n = R.shape[1]
    ab = ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))
    out = [0.0] * 12
    for q, (a, b) in enumerate(ab):
        out[q] = math.fsum(V[a][i] * V[b][i] for i in range(n))
    terms = [[] for _ in range(6)]
    for i in range(n):
        for j in range(i + 1, n):
            d = [R[c][i] - R[c][j] for c in range(3)]
            d = [x - L * math.copysign(math.floor(abs(x / L) + 0.5), x) for x in d]
            r = math.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
            if 0 < r < rcut:
                f = (1.0 / r + kappa) * math.exp(-kappa * r) / (r * r)
                for q, (a, b) in enumerate(ab):
                    terms[q].append(d[a] * d[b] * f)
    for q in range(6):
        out[6 + q] = math.fsum(terms[q])  # correctly rounded sums
    return np.array(out)


def test_reference_matches_a_scalar_loop_at_200_random_ions():
    rng = np.random.default_rng(11)
    n = 200
    L = _md_box(n)
    R = rng.uniform(-0.3 * L, 1.3 * L, size=(3, n))  # unwrapped coordinates too: the minimum image handles them
    V = rng.normal(size=(3, n)) * 0.6
    got, scale = stress_reference.stress(R, V, L, KAPPA, L / 2, block=37)  # a block size that does not divide n
    want = _scalar_stress(R, V, L, KAPPA, L / 2)
    assert np.all(np.abs(got - want) <= 1e-13 * scale), np.abs(got - want) / scale
    assert np.all(scale[6:] > 0)


def test_stress_of_one_pair_is_d_d_f():
    L = 10.0
    R = np.array([[1.0, 2.5], [1.0, 1.75], [1.0, 0.5]])  # d = r_0 - r_1 = (-1.5, -0.75, 0.5): exact in binary
    got, _ = stress_reference.stress(R, np.zeros((3, 2)), L, KAPPA, L / 2)
    dx, dy, dz = -1.5, -0.75, 0.5
    dr = math.sqrt(dx * dx + dy * dy + dz * dz)
    f = (1. / dr + KAPPA) * np.exp(np.array([-KAPPA * dr]))[0] / (dr * dr)
    assert list(got[:6]) == [0.0] * 6
    assert list(got[6:]) == [dx * dx * f, dy * dy * f, dz * dz * f, dx * dy * f, dx * dz * f, dy * dz * f]


def test_pair_beyond_the_cutoff_contributes_nothing():
    L = 10.0
    # minimum image (0.45 L, 0.45 L, 0): r = 0.64 L > rcut = L/2, although every component is below L/2
    R = np.array([[0.0, 0.45 * L], [0.0, 0.45 * L], [0.0, 0.0]])
    V = np.array([[0.5, -0.25], [0.0, 1.0], [2.0, 0.0]])
    got, _ = stress_reference.stress(R, V, L, KAPPA, L / 2)
    assert np.all(got[6:] == 0.0)
    assert list(got[:6]) == [0.5 * 0.5 + 0.25 * 0.25, 1.0, 4.0, -0.25, 1.0, 0.0]


def test_virial_scaling_identity(oracle):
    """Scaling positions, L and rcut = L/2 together by s keeps the pair set: tr W = -d(N Epot)/ds at s = 1, with the potential
    energy of the oracle (orc_epot_su)."""
    rng = np.random.default_rng(3)
    n = 300
    L = _md_box(n)
    R = rng.uniform(0, L, size=(3, n))
    trW = stress_reference.stress(R, np.zeros((3, n)), L, KAPPA, L / 2)[0][6:9].sum()
    h = 1e-4
    e = [n * oracle.epot_su(np.ascontiguousarray(R * s), L * s, 1.0 / KAPPA) for s in (1 + h, 1 - h)]
    dEds = (e[0] - e[1]) / (2 * h)
    assert abs(trW + dEds) <= 1e-7 * abs(trW), (trW, -dEds)


def test_cubic_lattice_is_isotropic():
    """The MD program's start (init(), MD:174-205): a simple cubic lattice filling the box, N = 512."""
    n = 512
    L = _md_box(n)
    side = round(n ** (1 / 3))
    R = np.zeros((3, n))
    k = 0
    for a in range(side):
        for b in range(side):
            for c in range(side):
                R[:, k] = [a * L / n ** (1 / 3.) + 0.5, b * L / n ** (1 / 3.) + 0.5, c * L / n ** (1 / 3.) + 0.5]
                k += 1
    W = stress_reference.stress(R, np.zeros((3, n)), L, KAPPA, L / 2)[0][6:]
    assert W[0] > 0
    assert W[1] == pytest.approx(W[0], rel=1e-12) and W[2] == pytest.approx(W[0], rel=1e-12)
    assert np.all(np.abs(W[3:]) <= 1e-12 * W[0]), W
