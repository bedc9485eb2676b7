"""GPU suite, part 3: the opt-in kernel mappings (environment knobs read once per process) stay parity-green:
MDQT_QT_LANES=4|2 (four / two lanes per ion in the fused substep kernel; the default picks by system size), MDQT_K1_ITEMS=0
(the CTA-tile force kernel where the item-walking kernel is the default), MDQT_ITEMS_IPT=2 (two rows per lane in the item kernel), MDQT_GRAPH=0
(stream launches instead of the replayed CUDA graph), MDQT_PDL=1 (programmatic dependent launch) and the force-kernel plan
overrides. Each runs __graft_entry__.smoke() -- one MD step with jumps against the oracle -- plus the
no-jump and jump-table goldens in a fresh interpreter."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


T = {"MDQT_K1_ITEMS": "0"}  # the CTA-tile force kernel (default for N > 8192) instead of the item-walking kernel


@pytest.mark.parametrize("env", [{"MDQT_QT_LANES": "4"}, {"MDQT_QT_LANES": "2"}, {"MDQT_GRAPH": "0"}, {"MDQT_PDL": "1"},
                                 {"MDQT_ITEMS_IPT": "2"}, T, dict(T, MDQT_PDL="1"),
                                 dict(T, MDQT_FORCE_IPT="2", MDQT_FORCE_JSUB="4"), dict(T, MDQT_FORCE_IPT="2", MDQT_FORCE_NSPLIT="3"),
                                 dict(T, MDQT_FORCE_JSUB="1", MDQT_FORCE_NSPLIT="7")])
def test_variant_parity(env):
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=ROOT, env=e, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", "tests/test_gpu_parity.py", "-k",
                        "nojump_golden or jump_table or forces_golden or trajectory_golden"], cwd=ROOT, env=e, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


_MD5 = r"""
import hashlib, sys
import numpy as np
from mdqtplasmasims_b200 import Engine, su_params, synthetic
n = 1500
p = su_params(n_ions=n, N0=n, seed=5, renormalize=int(sys.argv[1]))
e = Engine(p)
e.upload(R=synthetic.random_positions(n, p.L, seed=1), V=synthetic.maxwellian(n, 0.05, seed=2), psi=synthetic.random_full_state(n, 12, seed=3),
         tPart=np.zeros(n), t=0.0, substep=0)
e.md_steps(40)
s = e.download()
print(hashlib.md5(b"".join(s[k].tobytes() for k in ("R", "V", "psi", "tPart"))).hexdigest(), int((s["tPart"] < 25 * p.dtq).sum()))
"""


@pytest.mark.parametrize("renorm", [0, 1])
def test_two_and_four_lane_mappings_give_identical_bits(renorm):
    """The substep kernel's lane mapping is chosen from (N, n_traj) for speed; a job must not notice: 40 MD steps with quantum
    jumps (and with reNormalizewvFns) end in the same bits under MDQT_QT_LANES=2 and MDQT_QT_LANES=4."""
    out = []
    for lanes in ("2", "4"):
        r = subprocess.run([sys.executable, "-c", _MD5, str(renorm)], cwd=ROOT, env=dict(os.environ, MDQT_QT_LANES=lanes), capture_output=True,
                           text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-1500:]
        out.append(r.stdout.split())
    assert out[0][0] == out[1][0], out
    assert int(out[0][1]) > 0  # jumps happened within the last MD step
