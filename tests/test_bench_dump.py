"""CPU suite: bench.py --dump-outputs on a stand-in engine (no GPU): every array a caller of the timed path receives, as float64
.npy; above the byte limit the same seeded sample of ions in every array and every run, within the limit."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


class FakeEngine:
    def __init__(self, B, N, S=12):
        lead = (B,) if B > 1 else ()
        rng = np.random.default_rng(B * 1000 + N)
        self.N = N
        self.state = dict(R=rng.random(lead + (3, N)), V=rng.random(lead + (3, N)), psi=rng.random(lead + (N, S, 2)),
                          tPart=rng.random(lead + (N,)), t=1.25, substep=1000)
        self.F = rng.random(lead + (3, N))

    def download(self):
        return dict(self.state)

    def download_forces(self):
        return self.F


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_writes_every_output_in_full_below_the_limit(tmp_path):
    e = FakeEngine(1, 500)
    bench.dump_outputs(str(tmp_path), e)
    got = _load(str(tmp_path))
    assert sorted(got) == ["F", "R", "V", "psi", "t", "tPart"]
    assert all(a.dtype == np.float64 for a in got.values())
    for k in ("R", "V", "psi", "tPart"):
        assert np.array_equal(got[k], e.state[k]), k
    assert np.array_equal(got["F"], e.F) and float(got["t"]) == 1.25


def test_dump_above_the_limit_keeps_one_seeded_ion_sample(tmp_path):
    B, N, limit = 4, 2000, 1 << 20               # 4 x 2000 ions x 34 doubles = 2.2 MB > 1 MiB
    e = FakeEngine(B, N)
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    bench.dump_outputs(a, e, "_rank1", limit)
    bench.dump_outputs(b, e, "_rank1", limit)
    ga, gb = _load(a), _load(b)
    assert sorted(ga) == ["F_rank1", "R_rank1", "V_rank1", "psi_rank1", "tPart_rank1", "t_rank1"]
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= limit + 6 * 128   # + the .npy headers
    assert all(np.array_equal(ga[k], gb[k]) for k in ga)                                        # same sample every run
    n = ga["tPart_rank1"].shape[1]
    assert 0 < n < N and ga["psi_rank1"].shape == (B, n, 12, 2)
    # one ion subset for every array: recover it from tPart and check the others against the full state
    keep = np.array([np.flatnonzero(e.state["tPart"][0] == x)[0] for x in ga["tPart_rank1"][0]])
    assert np.all(np.diff(keep) > 0)
    assert np.array_equal(ga["R_rank1"], e.state["R"][..., keep]) and np.array_equal(ga["V_rank1"], e.state["V"][..., keep])
    assert np.array_equal(ga["F_rank1"], e.F[..., keep]) and np.array_equal(ga["psi_rank1"], e.state["psi"][:, keep])
    assert np.array_equal(ga["tPart_rank1"], e.state["tPart"][:, keep])


def test_dump_outputs_is_refused_for_the_cpu_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not os.path.exists(str(tmp_path / "d"))
