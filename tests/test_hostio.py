"""CPU suite, part 5: the host-side driver pieces (include/mdqt_io.h) against the LIVE unmodified reference:
directory naming, init() draw order, restart files byte for byte (write, read, round trip), and the main-loop
schedule. Needs oracle/_ref/libref_su.so (skipped when absent); the schedule test runs anywhere."""
import filecmp
import os

import numpy as np
import pytest

from mdqtplasmasims_b200 import hostio
from oracle import pyoracle as po

needs_su = pytest.mark.skipif(not po.ref_available("su"), reason="oracle/_ref/libref_su.so not built")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RESTART_FILES = (["ions_timestep%06d.dat", "conditions_timestep%06d.dat", "wvFns_timestep%06d.dat"] +
                 ["VZERO_timestep%%06d_interval%d.dat" % k for k in range(13)])


def test_io_symbols_exported():
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "mdqt_io.h")).read()
    declared = sorted(set(re.findall(r"\b(mdqt_[a-z0-9_]+)\s*\(", hdr)))
    L = hostio._lib()
    assert declared == sorted(hostio.IO_SYMBOLS)
    for name in declared:
        assert hasattr(L, name)


@pytest.mark.parametrize("kw", [dict(), dict(detuning=-2.5, detuningDP=0.5, Om=0.7, OmDP=1.3, fracOfSig=0.5, density=0.7, Te=25.5, sig0=3.3, Ge=0.083)])
def test_directory_name_matches_reference(kw):
    if not kw:  # the name the reference's main() makes for its default inputs, recorded from it
        assert hostio.dirname() == "dataLaserCool/Ge10Density2000E+11Sig040Te19SigFrac0DetSP-100DetDP100OmSP100OmDP100NumIons3500/job1/"
    if not po.ref_available("su"):
        if kw:
            pytest.skip("oracle/_ref/libref_su.so not built and no recorded reference name for these inputs")
        return
    ref = po.RefSU(**kw)
    # the harness starts from saveDirectory "x/" and job 1 (SU:1147-1159)
    assert hostio.dirname("x/", job=1, **kw) == ref.savedir()


@pytest.mark.parametrize("seed", [12345, 7])
def test_init_draw_order_bitwise(seed):
    """Without the live reference, seed 12345 is checked against the reference's own init() state stored in
    tests/golden/su_forces_N3472.npz (N, L, lDeb, every position and the first 64 wavefunctions)."""
    if po.ref_available("su"):
        ref = po.RefSU()
        n = ref.init(seed)
        s = ref.get_state()
        R, psi, L, lDeb = s["R"], s["psi"], ref.consts["L"], ref.consts["lDeb"]
    elif seed == 12345:
        g = np.load(os.path.join(GOLDEN, "su_forces_N3472.npz"))
        R, psi, L, lDeb = g["R"], g["psi0"], float(g["L"]), float(g["lDeb"])
        n = R.shape[1]
    else:
        pytest.skip("oracle/_ref/libref_su.so not built and no stored reference init() for this seed")
    ours = hostio.init_su(seed)
    assert ours["N"] == n and ours["L"] == L and ours["lDeb"] == lDeb
    assert np.array_equal(ours["R"], R) and np.array_equal(ours["psi"][:len(psi)], psi)
    assert not ours["V"].any() and not ours["tPart"].any()


@needs_su
def test_restart_files_byte_identical_and_round_trip(tmp_path):
    ref = po.RefSU()
    n = ref.init(99)
    s = ref.get_state()
    rng = np.random.default_rng(1)
    # make the state non-trivial: velocities, complex amplitudes incl. negative zeros and tiny numbers
    V = rng.normal(size=(3, n)) * 0.01
    psi = rng.normal(size=(n, 12, 2)) * 10.0 ** rng.integers(-12, 1, size=(n, 12, 2))
    psi[0, 3, 1] = -0.0
    psi[1] = 0.0
    psi[1, 11, 0] = 1.0
    ref.set_state(R=s["R"], V=V, psi=psi, tPart=np.zeros(n), t=1.234)
    da, db, dc = (str(tmp_path / x) + "/" for x in ("a", "b", "c"))
    for d in (da, db, dc):
        os.mkdir(d)
    ref.set_savedir(da)
    ref.set_counters(617, 15)
    ref.write_conditions(617)
    hostio.write_conditions(db, 617, 15, s["R"], V, psi)
    for f in RESTART_FILES:
        assert filecmp.cmp(os.path.join(da, f % 617), os.path.join(db, f % 617), shallow=False), f
    # read what the reference wrote: same values as the reference's own readConditions
    got = hostio.read_conditions(da, 617)
    ref.set_state(R=np.zeros((3, n)), V=np.zeros((3, n)), psi=np.zeros((n, 12, 2)), tPart=np.zeros(n), t=0.0)
    ref.read_conditions(617)
    r = ref.get_state()
    assert got["N"] == n == ref.N and got["counter"] == 15 == ref.counters()[1]
    assert got["t"] == r["t"] == (617 - 9.) * 0.002 + 0.02
    assert np.array_equal(got["R"], r["R"]) and np.array_equal(got["V"], r["V"]) and np.array_equal(got["psi"], r["psi"])
    # text-level round trip: write what we read -> identical bytes ("%lg" of a value parsed from "%lg")
    hostio.write_conditions(dc, 617, got["counter"], got["R"], got["V"], got["psi"], got["vholder"])
    for f in RESTART_FILES:
        assert filecmp.cmp(os.path.join(da, f % 617), os.path.join(dc, f % 617), shallow=False), f


def test_read_conditions_missing_files_is_an_error_not_a_crash(tmp_path):
    from mdqtplasmasims_b200 import MDQTError
    with pytest.raises(MDQTError):
        hostio.read_conditions(str(tmp_path) + "/", 3)


def _reference_loop(c0, tsc, t, ratio, sf, dtq, tmax, max_iter=10 ** 6):
    """Restatement of the reference loop body (SU:1248, 1365-1378) emitting one event per call it would make."""
    ev = []
    while t <= tmax + 0.0009 and len(ev) < max_iter:
        if (c0 + 1) % sf == 0 and tsc == 1:
            ev.append("output")
        if tsc == ratio:
            ev.append("forces")
            c0 += 1
            tsc = 0
        ev.append("sub")
        t += dtq
        tsc += 1
    return ev, c0, tsc, t


@pytest.mark.parametrize("c0,t0,ratio,sf,tmax", [(-1, 0.0, 25, 40, 0.25), (-1, 0.0, 25, 3, 0.05), (120, 0.242, 25, 40, 0.5),
                                                  (-1, 0.0, 1, 2, 0.02), (-1, 0.0, 41, 40, 0.33)])
def test_schedule_matches_reference_loop(c0, t0, ratio, sf, tmax):
    dtq = 0.002 / ratio
    ev_ref, c0_ref, tsc_ref, t_ref = _reference_loop(c0, ratio, t0, ratio, sf, dtq, tmax)
    ev, tsc, t = [], ratio, t0
    while True:
        n, do_out, do_f, c0, tsc, t = hostio.schedule_next(c0, tsc, t, ratio, sf, dtq, tmax)
        if n == 0:
            break
        ev += (["output"] if do_out else []) + (["forces"] if do_f else []) + ["sub"] * n
    assert ev == ev_ref and c0 == c0_ref and tsc == tsc_ref and t == t_ref
    assert ev.count("sub") > 100 or ratio == 1
