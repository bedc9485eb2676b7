"""The per-ion bound of tests/test_gpu_pair_plans.py and tests/test_gpu_pair_probe.py, on the CPU: it accepts a legitimate
different summation order and rejects the mistakes a pair kernel makes.

  * the oracle's float64 sequential sums (forces_su, forces_md) pass the bound of the plan the device uses at that size, and its
    energy (epot_su) the bound of its own summation chain;
  * a reference with one pair dropped, one pair counted twice, two trajectories swapped or one chunk's partial added twice fails it;
  * a pair term scaled by 1 + 32 u fails the probe's bound;
  * tests/pair_reference.py agrees with tests/stress_reference.py and tests/heat_reference.py, and with the 50-digit pair function
    within the device's per-term allowance on the probe set."""
import numpy as np
import pytest

import heat_reference
import pair_reference as pr
import stress_reference
from mdqtplasmasims_b200 import synthetic

# (n, jlen, nsplit) of the item plan the device takes for one trajectory of n ions (Engine.force_plan(); plan_items_jlen)
PLANS = [(600, 16, 38), (1001, 24, 42), (3529, 176, 21)]
LDEB = 1.0 / np.sqrt(0.3)  # kappa of the SU family (su_params: 0.5477)


def _system(n, seed):
    L = (n * 4.0 * np.pi / 3.0) ** (1.0 / 3.0)
    return synthetic.random_positions(n, L, seed=seed), L


def _violations(got, s, jlen, nsplit, n, kr):
    return int((np.abs(got - s["F"]) > pr.bound(s["SF"], s["QF"], pr.chain(jlen, nsplit, n), n, kr)).sum())


def _nearest(R, L, i):
    d = R[:, i:i + 1] - R
    d -= L * np.rint(d / L)
    r = np.sqrt((d * d).sum(axis=0))
    r[i] = np.inf
    j = int(np.argmin(r))
    return j, d[:, j], r[j]


def _f(r, kappa):
    return (1.0 / r + kappa) * np.exp(-kappa * r) / (r * r)


@pytest.mark.parametrize("n,jlen,nsplit", PLANS)
def test_oracle_passes_the_bound(oracle, n, jlen, nsplit):
    R, L = _system(n, n)
    kappa = 1.0 / LDEB
    s = pr.ion_sums(R, L, kappa, L / 2)
    assert _violations(oracle.forces_su(R, L, LDEB), s, jlen, nsplit, n, kappa * L / 2) == 0
    rc = 0.41 * L
    s_md = pr.ion_sums(R, L, 0.5, rc)
    assert _violations(oracle.forces_md(R, L, 0.5, rc), s_md, jlen, nsplit, n, 0.5 * rc) == 0
    rec = pr.records(s, np.zeros((3, n)))
    want, S, Q = rec["epot"]
    # epot_su is the per-ion energy that Epotential() returns, summed in ONE sequential accumulator over the n (n - 1) / 2
    # unordered pairs: that chain, not the device's, is the longest a term of the oracle meets
    m = pr.chain(jlen, nsplit, n, final=True) + n * (n - 1) // 2
    assert abs(oracle.epot_su(R, L, LDEB) - want[0]) <= pr.bound(S, Q, m, n, kappa * L / 2)[0]


@pytest.mark.parametrize("n,jlen,nsplit", PLANS)
def test_pair_and_chunk_mistakes_fail_the_bound(n, jlen, nsplit):
    R, L = _system(n, n + 1)
    kappa, rc = 1.0 / LDEB, L / 2
    kr = kappa * rc
    s = pr.ion_sums(R, L, kappa, rc)
    F = s["F"].copy()
    assert _violations(F, s, jlen, nsplit, n, kr) == 0
    i = n // 3
    j, d, r = _nearest(R, L, i)
    term = _f(r, kappa) * d
    dropped = F.copy()
    dropped[:, i] -= term
    assert _violations(dropped, s, jlen, nsplit, n, kr) > 0, "one pair dropped from one ion"
    doubled = F.copy()
    doubled[:, i] += term
    assert _violations(doubled, s, jlen, nsplit, n, kr) > 0, "one pair counted twice"
    # the chunk of ion i's j range that holds its nearest neighbour, added twice
    c0 = (j // jlen) * jlen
    Rc = np.concatenate([R[:, i:i + 1], R[:, c0:c0 + jlen]], axis=1)
    chunk = pr.ion_sums(Rc, L, kappa, rc, rows=[0])["F"][:, 0]
    twice = F.copy()
    twice[:, i] += chunk
    assert _violations(twice, s, jlen, nsplit, n, kr) > 0, "one chunk's partial added twice"


def test_swapped_trajectories_fail_the_bound():
    n, jlen, nsplit = PLANS[1]
    L = (n * 4.0 * np.pi / 3.0) ** (1.0 / 3.0)
    kappa = 1.0 / LDEB
    sums = [pr.ion_sums(synthetic.random_positions(n, L, seed=20 + b), L, kappa, L / 2) for b in range(2)]
    for b in range(2):
        assert _violations(sums[b]["F"], sums[b], jlen, nsplit, n, kappa * L / 2) == 0
        assert _violations(sums[1 - b]["F"], sums[b], jlen, nsplit, n, kappa * L / 2) > n  # trajectories b and b + 1 swapped
    recs = [pr.records(s, np.zeros((3, n))) for s in sums]
    want, S, Q = recs[0]["epot"]
    assert abs(recs[1]["epot"][0][0] - want[0]) > pr.bound(S, Q, pr.chain(jlen, nsplit, n, final=True), n, kappa * L / 2)[0]


def test_probe_term_scaled_by_32u_fails_the_bound():
    L, kappa = 2.0, 1.0
    X = pr.probe_positions(L, L / 2, 640, True, seed=3)
    V = np.random.default_rng(4).normal(size=X.shape)
    hi, lo, S, Q, r, cls = pr.mp_probe(X, V, L, kappa, (L / 2,), 0.0)
    inside = cls[L / 2] == 1
    lim = (pr.CP + pr.CR * kappa * r[:, None]) * pr.U * S + Q
    assert np.all(np.abs(lo) <= lim)  # the reference itself (its double head) is inside
    scaled = hi * (1 + 32 * pr.U)
    err = np.abs((scaled - hi) - lo)
    # every nonzero single term (all but the heat contractions, whose S adds two) of every pair inside the cut-off is caught
    # (kappa r <= 1 here: 16 + 3 < 32)
    single = np.zeros(21, dtype=bool)
    single[:13] = single[19:] = True
    nonzero = inside[:, None] & (hi != 0) & single
    assert nonzero.sum() > 1000
    assert np.all(err[nonzero] > lim[nonzero])


def test_records_agree_with_the_stress_and_heat_references():
    n = 700
    R, L = _system(n, 5)
    V = np.random.default_rng(6).normal(size=(3, n))
    for kappa, rc in ((1.0 / LDEB, L / 2), (0.5, 0.41 * L)):
        rec = pr.records(pr.ion_sums(R, L, kappa, rc), V)
        w, ws = stress_reference.stress(R, V, L, kappa, rc)
        h, hs = heat_reference.heat(R, V, L, kappa, rc)
        assert np.all(np.abs(rec["stress"][0] - w) <= 64 * pr.U * ws)
        assert np.all(np.abs(rec["heat"][0] - h) <= 64 * pr.U * hs)
        assert np.allclose(rec["stress"][1][6:], ws[6:], rtol=1e-12)


@pytest.mark.parametrize("rc", [1.0, 0.74])
def test_numpy_reference_agrees_with_50_digits_per_term(rc):
    """ion_sums of a two-ion trajectory is one pair term: within the device's per-term allowance (c_p + 3 kappa r) u of the 50-digit
    value -- numpy's float64 pair function rounds about as often as the kernel's (measured: up to 9 u at kappa r <= 1)."""
    L, kappa = 2.0, 1.0
    X = pr.probe_positions(L, rc, 640, False, seed=11)
    Xw = np.mod(X, L)  # ion_sums takes wrapped positions: both references start from these doubles
    V = np.zeros(X.shape)
    hi, lo, S, Q, r, cls = pr.mp_probe(Xw, V, L, kappa, (rc,), 0.0)
    inside = cls[rc] == 1
    for b in np.flatnonzero(inside):
        s = pr.ion_sums(Xw[b], L, kappa, rc, workers=1)
        got = np.concatenate([s["F"][:, 0], s["F"][:, 1], [s["phi"][0] / 2], s["T"][:, 0]])
        want_hi, want_lo = hi[b, :13], lo[b, :13]
        lim = (pr.CP + pr.CR * kappa * r[b]) * pr.U * S[b, :13]
        assert np.all(np.abs((got - want_hi) - want_lo) <= lim), (b, r[b], got, want_hi)
