"""CPU suite: pins the test-side mode reference (tests/modes_reference.py) that checks the GPU recorder mdqt_modes_*.

A single ion gives rho = exp(i k.r) and j = v rho; a simple cubic lattice gives rho_k = N when the lattice side divides every n_a and
zero otherwise; free streaming obeys continuity, d rho_k / dt = i k.j_k, to second order in the step of a central difference; and the
correlations satisfy C_L(k, 0) + 2 C_T(k, 0) = 1/(N T) sum_s sum_a |j_a(s)|^2."""
import numpy as np
import pytest

import modes_reference as mr


@pytest.mark.parametrize("eighths", range(8))
def test_single_ion_on_exact_phases(eighths):
    """r / L = (eighths / 8 + 2, -1, 3), outside the box: n.r / L = 3 eighths / 8 mod 1 with no rounding in r / L."""
    L = 16.0
    n = np.array([[3, -5, 7]])
    r = np.array([[L * (eighths / 8.0 + 2.0)], [-L], [3 * L]])
    v = np.array([[0.25], [-1.5], [2.0]])
    got, scale = mr.modes(r, v, L, n)
    ph = np.pi * ((3 * eighths) % 8) / 4
    want_rho = np.exp(1j * ph)
    assert abs(got[0, 0] - want_rho.real) <= 2 ** -52 and abs(got[0, 1] - want_rho.imag) <= 2 ** -52
    for a in range(3):
        assert abs(got[0, 2 + 2 * a] - v[a, 0] * want_rho.real) <= 2 ** -52 * abs(v[a, 0])
        assert abs(got[0, 3 + 2 * a] - v[a, 0] * want_rho.imag) <= 2 ** -52 * abs(v[a, 0])
    assert np.array_equal(scale[0], [1, 1, 0.25, 0.25, 1.5, 1.5, 2, 2])


def test_single_ion_at_random_positions():
    rng = np.random.default_rng(1)
    L = 11.3
    nvec = rng.integers(-200, 201, size=(20, 3))
    for _ in range(10):
        r = rng.uniform(-3 * L, 4 * L, size=(3, 1))
        v = rng.normal(size=(3, 1))
        got, _ = mr.modes(r, v, L, nvec)
        ph = 2 * np.pi * (nvec @ r[:, 0]) / L  # double: loses about |n.r| / L ulps of a turn
        rho = np.exp(1j * ph)
        tol = 1e-15 * np.abs(nvec @ r[:, 0] / L).max() * 8 + 1e-15
        assert np.allclose(got[:, 0] + 1j * got[:, 1], rho, rtol=0, atol=tol)
        for a in range(3):
            assert np.allclose(got[:, 2 + 2 * a] + 1j * got[:, 3 + 2 * a], v[a, 0] * rho, rtol=0, atol=tol * abs(v[a, 0]))


@pytest.mark.parametrize("side", [4, 6])
def test_simple_cubic_lattice(side):
    L = 9.7
    g = np.arange(side) * (L / side)
    R = np.array(np.meshgrid(g, g, g, indexing="ij")).reshape(3, -1)
    N = R.shape[1]
    V = np.ones_like(R)
    nvec = np.array([(a, b, c) for a in range(-7, 8) for b in range(-7, 8) for c in (-12, -3, 0, 1, side, 2 * side)
                     if (a, b, c) != (0, 0, 0)])
    got, _ = mr.modes(R, V, L, nvec)
    on = np.all(nvec % side == 0, axis=1)
    assert on.any() and (~on).any()
    rho = got[:, 0] + 1j * got[:, 1]
    assert np.all(np.abs(rho[on] - N) <= 1e-12 * N)
    assert np.all(np.abs(rho[~on]) <= 1e-12 * N)
    # unit velocities: every j_a equals rho
    for a in range(3):
        assert np.allclose(got[:, 2 + 2 * a] + 1j * got[:, 3 + 2 * a], rho, rtol=0, atol=1e-12 * N)
    # a shifted lattice: rho_k = N exp(i k.r0) on the reciprocal lattice
    r0 = np.array([0.37, -1.1, 2.9])
    got, _ = mr.modes(R + r0[:, None], V, L, nvec[on])
    want = N * np.exp(2j * np.pi * (nvec[on] @ r0) / L)
    assert np.allclose(got[:, 0] + 1j * got[:, 1], want, rtol=0, atol=1e-12 * N)


def test_free_streaming_obeys_continuity():
    """r(t) = r0 + v t: [rho(t + h) - rho(t - h)] / (2 h) = i k.j(t) + O(h^2)."""
    rng = np.random.default_rng(2)
    L, n = 10.0, 50
    r0 = rng.uniform(0, L, size=(3, n))
    v = rng.normal(size=(3, n))
    nvec = np.array([[1, 0, 0], [0, 2, 0], [1, -1, 3], [4, 0, -2]])
    kv = 2 * np.pi * nvec / L
    t = 0.7
    rec0, _ = mr.modes(r0 + v * t, v, L, nvec)
    rho0, j0 = mr.complex_modes(rec0[:, :, None])
    want = 1j * np.einsum("qa,qa->q", kv, j0[:, :, 0])
    errs = []
    for h in (0.02, 0.01, 0.005):
        rp, _ = mr.modes(r0 + v * (t + h), v, L, nvec)
        rm, _ = mr.modes(r0 + v * (t - h), v, L, nvec)
        d = ((rp[:, 0] + 1j * rp[:, 1]) - (rm[:, 0] + 1j * rm[:, 1])) / (2 * h)
        errs.append(np.abs(d - want).max() / np.abs(want).max())
    assert errs[0] < 1e-2
    for a, b in zip(errs, errs[1:]):
        assert 3.5 < a / b < 4.5, errs


def test_current_identity_at_zero_lag():
    rng = np.random.default_rng(3)
    K, T, n = 5, 30, 77
    rec = rng.normal(size=(K, 8, T)) * 10
    nvec = rng.integers(-9, 10, size=(K, 3))
    nvec[np.all(nvec == 0, axis=1)] = [1, 0, 0]
    F, CL, CT = mr.correlations(rec, n, nvec)
    rho, j = mr.complex_modes(rec)
    assert np.allclose(CL[:, 0] + 2 * CT[:, 0], (np.abs(j) ** 2).sum(axis=(1, 2)) / (n * T), rtol=1e-13, atol=0)
    assert np.allclose(F[:, 0], (np.abs(rho) ** 2).sum(axis=1) / (n * T), rtol=1e-13, atol=0)
    # one lag written out: C_T(k, 2) from the transverse vectors
    q, t = 2, 2
    khat = nvec[q] / np.linalg.norm(nvec[q])
    jt = j[q] - np.outer(khat, khat @ j[q])
    want = sum(np.vdot(jt[:, s + t], jt[:, s]).real for s in range(T - t)) / (2 * n * (T - t))
    assert CT[q, t] == pytest.approx(want, rel=1e-13)
