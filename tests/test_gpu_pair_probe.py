"""GPU suite: the pair function of the all-pairs loop against a 50-digit reference, one pair at a time.

One handle holds B = 4096 trajectories of two ions, so every force, energy, stress and heat entry the device reports is one pair
term (or, for the heat current, one term contracted with two velocities): no summation error hides what the kernel computes per pair
-- the fixed-point minimum image, rsqrt, the table-plus-cubic exp and the prefactors. Both cut-off settings (rcut = L/2, the HL
instantiations, and rcut = 0.37 L), both plans (item walk and CTA tiles, MDQT_K1_ITEMS=0 read per handle) and two position sets:
one on the grid x = L m / 2^40 (L a power of two), where the fixed-point separation is exact, and random doubles, where the
conversion rounds. Every pair term t must satisfy
    |device - t| <= (c_p + 3 kappa r) u S + Q,    c_p = 16
(pair_reference: S = |t|, or the sum of |terms| of the heat contraction; Q = the conversion error times the separation sensitivity,
0 on the grid). Pairs with r <= rcut (1 - 8 2^-52) must contribute, pairs with r >= rcut (1 + 8 2^-52), r = rcut or r = 0 must give
exactly 0, and the band between may do either. The measured max |device - t| / (u S) per mode is printed."""
import numpy as np
import pytest

import pair_reference as pr
from mdqtplasmasims_b200 import Engine, md_params

pytestmark = pytest.mark.gpu
B, L, KAPPA = 4096, 2.0, 1.0
RCUTS = {"hl": L / 2, "rc037": L * round(0.37 * 2 ** 40) / 2 ** 40}  # on the grid: r = rcut exactly is representable


@pytest.fixture(scope="module")
def probe():
    """Positions, velocities and the 50-digit reference per (cut-off, position set), shared by both plans."""
    out = {}
    for rk, rc in RCUTS.items():
        for grid in (True, False):
            X = pr.probe_positions(L, rc, B, grid, seed=7 if grid else 8)
            V = np.random.default_rng(9).normal(size=X.shape)
            out[rk, grid] = (X, V) + pr.mp_probe(X, V, L, KAPPA, (rc,), 0.0 if grid else pr.conversion_delta(L))
    return out


def _device(X, V, rc):
    p = md_params(n_ions=2, n_traj=B, kappa=KAPPA)
    p.L, p.rcut = L, rc
    e = Engine(p)
    e.upload(R=X, V=V)
    got = np.zeros((B, 21))
    e.forces()
    F = e.download_forces()
    got[:, 0:3], got[:, 3:6] = F[:, :, 0], F[:, :, 1]
    got[:, 6] = e.Epotential()
    e.stress_begin(1)
    e.stress_record(0)
    got[:, 7:13] = e.stress_download(1)[:, 6:12, 0]
    e.heat_begin(1)
    e.heat_record(0)
    h = e.heat_download(1)[..., 0]
    got[:, 13:19], got[:, 19:21] = h[:, 3:9], h[:, 13:15]
    e.close()
    return got


@pytest.mark.parametrize("plan", ["items", "tiles"])
@pytest.mark.parametrize("rk", list(RCUTS))
@pytest.mark.parametrize("grid", [True, False], ids=["grid", "random"])
def test_pair_terms_within_the_bound(probe, plan, rk, grid, monkeypatch):
    if plan == "tiles":
        monkeypatch.setenv("MDQT_K1_ITEMS", "0")
    rc = RCUTS[rk]
    X, V, hi, lo, S, Q, r, cls = probe[rk, grid]
    cls = cls[rc]
    got = _device(X, V, rc)
    err = np.abs((got - hi) - lo)
    lim = (pr.CP + pr.CR * KAPPA * r[:, None]) * pr.U * S + Q
    inside, outside, band = cls == 1, cls == 0, cls == -1
    assert outside.sum() >= 1 and inside.sum() > B // 2
    # outside the cut-off (and the coincident pair): exactly 0 in every mode
    nz = outside[:, None] & (got != 0)
    assert not nz.any(), "pairs outside the cut-off contribute: %s, r = %s" % (np.argwhere(nz)[:4].tolist(), r[nz.any(axis=1)][:4])
    # inside: within the bound (and really there: the bound is far below |t|)
    bad = inside[:, None] & ~(err <= lim)
    assert not bad.any(), "pair terms outside the bound: %s, error/bound %s, r %s" % (
        np.argwhere(bad)[:6].tolist(), (err / lim)[bad][:6], r[bad.any(axis=1)][:6])
    assert np.all(got[inside][:, 6] > 0)
    # the band: either exactly 0 or within the bound, for every entry of a pair alike
    for b in np.flatnonzero(band):
        assert np.all(got[b] == 0) or np.all(err[b] <= lim[b]), (b, r[b], got[b], hi[b])
    meas = {m: float(((err - Q) / (pr.U * np.where(S > 0, S, 1)))[inside][:, cols].max()) for m, cols in pr.PROBE_COLUMNS.items()}
    print("pair probe %-5s %-5s %-6s max |error| / (u S) per mode: %s   (%d inside, %d outside, %d in the band)" % (
        plan, rk, "grid" if grid else "random", " ".join("%s %.2f" % kv for kv in meas.items()), inside.sum(), outside.sum(),
        band.sum()))
