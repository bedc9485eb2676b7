"""GPU suite: the pair-once force tiles of k_pairs_items (N <= 8192) -- 64-ion blocks, each unordered pair evaluated once, one partial
per partner block.

Forces are checked per ion against tests/pair_reference.py with the bound of the plan's addition chain (jlen + nsplit from
Engine.force_plan()), at block-count edges (N = 1, 2, 63, 64, 65, 129) and at the sizes the benchmark and the ensembles run. A batch of
unequal ion counts, a row split that is not a multiple of 64 and a repeated run must give the same bits as the single whole-system
run: the summation order of a row depends on its trajectory's own ion count alone."""
import numpy as np
import pytest

import pair_reference as pr
from mdqtplasmasims_b200 import Engine, su_params

pytestmark = pytest.mark.gpu


def _positions(n, L, seed):
    return np.random.default_rng(seed).uniform(0, L, size=(3, n))


def _forces(p, R, counts=None):
    e = Engine(p)
    if counts is not None:
        e.set_ion_counts(counts)
    e.upload(R=R)
    e.forces()
    F = e.download_forces()
    plan = e.force_plan()
    e.close()
    return F, plan


@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 129, 3500, 4096, 8192])
def test_forces_within_the_bound(n):
    p = su_params(n_ions=n, N0=n)
    R = _positions(n, p.L, n)
    F, (nsplit, jlen) = _forces(p, R)
    assert (nsplit, jlen) == ((n + 63) // 64, 64)
    s = pr.ion_sums(R, p.L, p.kappa, p.rcut)
    lim = pr.bound(s["SF"], s["QF"], pr.chain(jlen, nsplit, n), n, p.kappa * p.rcut)
    err = np.abs(F - s["F"])
    assert (err <= lim).all(), "worst error / bound %.3g" % float((err / np.where(lim > 0, lim, 1)).max())


def test_unequal_batch_equals_single_trajectories_bitwise():
    n, B = 700, 5
    counts = np.array([700, 641, 64, 129, 1])
    p = su_params(n_ions=n, N0=n, n_traj=B)
    R = np.stack([_positions(n, p.L, 50 + b) for b in range(B)])
    F, _ = _forces(p, R, counts)
    F = F.reshape(B, 3, n)
    for b in range(B):
        nb = int(counts[b])
        Fs, _ = _forces(su_params(n_ions=nb, N0=n), R[b][:, :nb])  # the same box (N0) as the batch
        assert np.array_equal(F[b][:, :nb], Fs.reshape(3, nb)), "trajectory %d (%d ions)" % (b, nb)


def test_row_split_equals_whole_system_bitwise():
    n, row0 = 3500, 37
    R = _positions(n, su_params(n_ions=n, N0=n).L, 9)
    F, _ = _forces(su_params(n_ions=n, N0=n), R)
    for r0, rows in ((0, row0), (row0, 1000), (row0 + 1000, n - row0 - 1000)):
        Fg, _ = _forces(su_params(n_ions=n, N0=n, row0=r0, n_rows=rows), R)
        assert np.array_equal(Fg[:, r0:r0 + rows], F[:, r0:r0 + rows]), "rows [%d, %d)" % (r0, r0 + rows)


def test_two_runs_bitwise_equal():
    n = 3500
    p = su_params(n_ions=n, N0=n)
    R = _positions(n, p.L, 3)
    F1, _ = _forces(p, R)
    F2, _ = _forces(p, R)
    assert np.array_equal(F1, F2)
