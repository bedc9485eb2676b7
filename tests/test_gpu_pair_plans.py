"""GPU suite: every instantiation of the all-pairs loop against a per-ion error bound.

The force planner picks one of 58 instantiations of k_pairs_items / k_pairs from (n_ions, n_traj, ion counts, rcut) and the
developer knobs. Each case below is one such plan, run in all four modes -- forces(), Epotential(), a stress record and a heat
record -- in both cut-off settings: SU parameters (rcut = L/2, the HL instantiations, with one coincident pair) and MD parameters
with rcut = 0.41 L. Every ion's force component and every record entry is compared with tests/pair_reference.py against
    |device - reference| <= (2 (c_p + 3 kappa rcut) + m + ceil(log2 n) + 4) u S + Q
(pair_reference.bound: S the sum of |terms|, Q the position-conversion term, m the plan's addition chain from Engine.force_plan()).
The bound is a first-order worst case, about 1e-13 of S here; a dropped, doubled or misrouted pair, chunk, row or trajectory moves a
result by orders of magnitude more. Ions beyond a job's count sit 1e-3 a from ion 0 and carry V = NaN: counting one shows.

Each case records the kernels it launched (torch.profiler, CUDA activities, in memory), and the last test requires the union to
be every k_pairs* symbol of the loaded library, so an instantiation added without a case here fails the suite.
MDQT_K1_ITEMS and MDQT_FORCE_* are read per handle (set in-process)."""
import re
import shutil
import subprocess
from collections import namedtuple

import numpy as np
import pytest

import pair_reference as pr
from mdqtplasmasims_b200 import Engine, md_params, su_params
from mdqtplasmasims_b200.engine import LIB_PATH

pytestmark = pytest.mark.gpu
MODES = ("forces", "epot", "stress", "heat")
OBSERVED = set()   # normalised k_pairs* names launched by the cases of this module
RAN = set()

Case = namedtuple("Case", "name n B counts plan_n env modes rows")


def case(name, n, B=1, counts=None, plan_n=0, env=None, modes=MODES, rows=None):
    return Case(name, n, B, counts, plan_n, env or {}, modes, rows)


def _tiles(**kw):
    return dict({"MDQT_K1_ITEMS": "0"}, **{"MDQT_FORCE_" + k: str(v) for k, v in kw.items()})


# jlen / nsplit of the item plans (plan_items_jlen): N = 1, 33 -> 8 / 1, 5; 1001 -> 24 / 42; 3529 -> 176 / 21; 4353 -> 136 / 33;
# 6945 -> 224 / 32; 600 -> 16 / 38; 128 -> 8 / 16. The ragged ones (N mod jlen = 1) leave one ion in the last chunk.
CASES = [
    # item walk, one trajectory: the one-CTA-per-SM kernel <8, 2, 0, HL, 8> up to N ~ 4100
    case("b1_n1", 1), case("b1_n2", 2), case("b1_n33", 33), case("b1_n1001", 1001), case("b1_n3529", 3529),
    case("b1_n4353", 4353),                                   # <8, 1, 0, HL, 16>, ragged
    case("b3_n1001", 1001, 3),                                # <8, 1, 0, HL, 16> for a batch
    case("b3_n4353", 4353, 3),                                # <16, 2, 0, HL, 16>, ragged
    case("b2_n6945", 6945, 2),                                # <8, 2, 0, HL, 16>: jlen 224 > 216 leaves no room for 16 warps; ragged
    case("b64_n600", 600, 64),                                # slot walk, equal counts
    case("b64_n600_unequal", 600, 64, counts=(400, 600)),     # packed list of non-empty items
    case("b600_n128_unequal", 128, 600, counts=(90, 128)),    # B > 512: ion counts and chunk lengths read from global memory
    case("b8_plan_n500", 1000, 8, counts=(400, 1000), plan_n=500),  # one nominal chunk length for n_ions up to 2 plan_n
    # CTA tiles: the default plans beyond the item walk, and a large ragged N on sampled rows
    case("tiles_b1_n8193", 8193), case("tiles_b2_n8193", 8193, 2),
    case("tiles_b1_n30011", 30011, modes=("forces",), rows=256),
]
# every (rows per thread, in-CTA split, row group) of each mode, with one chunk (direct store) and several (partials + last CTA)
for _n, _ns in ((1001, (1, 3, 7, 1, 3, 1, 3)), (3001, (5, 2, 1, 7, 1, 3, 1))):
    for _k, (_kn, _s) in enumerate(zip((dict(RG=128, IPT=2, JSUB=4), dict(RG=128, IPT=2, JSUB=2), dict(RG=128, IPT=2, JSUB=1),
                                        dict(RG=128, IPT=1, JSUB=2), dict(RG=128, IPT=1, JSUB=1), dict(RG=32, JSUB=8),
                                        dict(RG=32, JSUB=4)), _ns)):
        CASES.append(case("knob_n%d_%s" % (_n, "_".join("%s%s" % kv for kv in _kn.items())), _n, env=_tiles(NSPLIT=_s, **_kn)))
ALL_CASES = {c.name: c for c in CASES}


def _params(kind, c):
    if kind == "su":  # rcut = L/2
        p = su_params(n_ions=c.n, N0=c.n, n_traj=c.B)
    else:
        p = md_params(n_ions=c.n, n_traj=c.B)
        p.rcut = 0.41 * p.L
    p.plan_n = c.plan_n
    return p


def _counts(c):
    if c.counts is None:
        return None
    return np.random.default_rng(c.n + c.B).integers(c.counts[0], c.counts[1] + 1, size=c.B)


def _traj(kind, n, L, b, nb):
    """Positions in [0, L) and velocities of trajectory b (the same for every case of this n), ions >= nb padded."""
    rng = np.random.default_rng(1000 * n + b)
    R, V = rng.uniform(0, L, size=(3, n)), rng.normal(size=(3, n)) * 0.3
    if kind == "su" and nb >= 2:
        R[:, 1] = R[:, 0]  # a coincident pair: 0 in every mode
    a = L / max(nb, 1) ** (1.0 / 3.0)
    R[:, nb:] = ((R[:, 0] + np.array([1e-3 * a, 0.0, 0.0])) % L)[:, None]
    V[:, nb:] = np.nan
    return R, V


def _rows(c):
    if c.rows is None:
        return None
    rng = np.random.default_rng(c.n)
    edges = [0, 1, 31, 32, 127, 128, c.n // 2, c.n - 2, c.n - 1]
    return np.unique(np.concatenate([edges, rng.choice(c.n, c.rows - len(edges), replace=False)]))


def _names(prof):
    return {_norm(e.name) for e in prof.events() if "k_pairs" in e.name}


def _norm(name):
    """'void mdqt::k_pairs<1, 8, 0, 8, true, 32>(...)' (or cu++filt's '(int)1, (bool)1') -> 'k_pairs<1,8,0,8,true,32>'."""
    if name.startswith("_Z"):
        name = subprocess.run(["c++filt"], input=name, capture_output=True, text=True, check=True).stdout
    m = re.search(r"(k_pairs(?:_items)?)<([^>]*)>", name)
    args = [a.strip().replace("(int)", "") for a in m.group(2).split(",")]
    args = [{"(bool)0": "false", "(bool)1": "true"}.get(a, a) for a in args]
    return "%s<%s>" % (m.group(1), ",".join(args))


def run_case(kind, c):
    """Run case c on the device: (results per mode, (nsplit, jlen), normalised kernel names launched)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    p = _params(kind, c)
    counts = _counts(c)
    R, V = np.zeros((c.B, 3, c.n)), np.zeros((c.B, 3, c.n))
    for b in range(c.B):
        R[b], V[b] = _traj(kind, c.n, p.L, b, c.n if counts is None else int(counts[b]))
    out = {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e = Engine(p)
        if counts is not None:
            e.set_ion_counts(counts)
        e.upload(R=R if c.B > 1 else R[0], V=V if c.B > 1 else V[0])
        if "forces" in c.modes:
            e.forces()
            out["forces"] = e.download_forces().reshape(c.B, 3, c.n)
        if "epot" in c.modes:
            out["epot"] = np.atleast_1d(e.Epotential())
        if "stress" in c.modes:
            e.stress_begin(1)
            e.stress_record(0)
            out["stress"] = e.stress_download(1)[..., 0].reshape(c.B, 12)
        if "heat" in c.modes:
            e.heat_begin(1)
            e.heat_record(0)
            out["heat"] = e.heat_download(1)[..., 0].reshape(c.B, 15)
        e.sync()
        plan = e.force_plan()
        e.close()
        torch.cuda.synchronize()
    return out, plan, _names(prof)


_REF = {}


def _reference(kind, c, p, b, nb, rows):
    """ion_sums of trajectory b's first nb ions, shared by every case and mode that holds the same positions."""
    key = (kind, c.n, p.L, b, nb, None if rows is None else rows.tobytes())
    if key not in _REF:
        R, V = _traj(kind, c.n, p.L, b, nb)
        s = pr.ion_sums(R[:, :nb], p.L, p.kappa, p.rcut, rows=rows)
        _REF[key] = (s, None if rows is not None else pr.records(s, V[:, :nb]))
    return _REF[key]


def check_case(kind, c, out, plan):
    """Compare every result of case c with the reference; returns {mode: max error / bound}."""
    p = _params(kind, c)
    counts = _counts(c)
    nsplit, jlen = plan
    rows = _rows(c)
    kr = p.kappa * p.rcut
    worst = {}
    for b in range(c.B):
        nb = c.n if counts is None else int(counts[b])
        s, rec = _reference(kind, c, p, b, nb, rows)
        for mode in c.modes:
            if mode == "forces":
                got = out["forces"][b][:, :nb] if rows is None else out["forces"][b][:, rows]
                err = np.abs(got - s["F"])
                lim = pr.bound(s["SF"], s["QF"], pr.chain(jlen, nsplit, nb), nb, kr)
            else:
                want, S, Q = rec[mode]
                err = np.abs(out[mode][b] - want)
                lim = pr.bound(S, Q, pr.chain(jlen, nsplit, nb, final=True), nb, kr)
            bad = ~(err <= lim)
            assert not bad.any(), "%s %s %s b=%d: %d entries outside the bound, worst error/bound %.3g at %s" % (
                kind, c.name, mode, b, bad.sum(), np.nanmax(np.where(lim > 0, err / np.where(lim > 0, lim, 1), np.inf)),
                np.argwhere(bad)[:4].tolist())
            ratio = np.where(lim > 0, err / np.where(lim > 0, lim, 1.0), 0.0)
            worst[mode] = max(worst.get(mode, 0.0), float(ratio.max()) if ratio.size else 0.0)
    return worst


def _report(kind, c, plan, worst, names):
    print("pair plans %-3s %-26s nsplit/jlen %4d/%-5d max error/bound %s   kernels %s" % (
        kind, c.name, plan[0], plan[1], " ".join("%s %.2e" % kv for kv in worst.items()), " ".join(sorted(names))))


@pytest.mark.parametrize("kind", ["su", "md"])
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_plan_against_reference(name, kind, monkeypatch):
    c = ALL_CASES[name]
    for k, v in c.env.items():
        monkeypatch.setenv(k, v)
    out, plan, names = run_case(kind, c)
    assert names, "the profiler saw no k_pairs kernel"
    OBSERVED.update(names)
    worst = check_case(kind, c, out, plan)
    _report(kind, c, plan, worst, names)
    RAN.add((name, kind))


def _library_pair_kernels():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sym = subprocess.run([tool, "-symbols", LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted({ln.split()[-1] for ln in sym.splitlines() if "k_pairs" in ln and "STO_ENTRY" in ln})
    dem = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return {_norm(ln) for ln in dem.splitlines() if ln.strip()}


def test_every_pair_instantiation_was_launched():
    """Runs last: the cases above must have launched every k_pairs* instantiation the library holds."""
    expected = {(c.name, k) for c in CASES for k in ("su", "md")}
    assert RAN == expected, "run the whole module: cases missing %s" % sorted(expected - RAN)[:8]
    lib = _library_pair_kernels()
    missing, extra = sorted(lib - OBSERVED), sorted(OBSERVED - lib)
    print("%d of %d k_pairs* instantiations launched" % (len(lib & OBSERVED), len(lib)))
    assert not missing and not extra, "never launched: %s; launched but not in the library: %s" % (missing, extra)
