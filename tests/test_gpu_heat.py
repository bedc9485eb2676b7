"""GPU suite: the heat (energy) current recorder mdqt_heat_* and `mdqt_run --program md --heat 1`.

Against the test-side reference (tests/heat_reference.py) in both force plans (item walk for N <= 8192, CTA tiles beyond), against
the device's own potential energy and pressure tensor, the sign symmetry under V -> -V, bitwise reproducibility (repeat, batch vs
single, unequal ion counts), no side effects on the state or on later steps, the heat-current autocorrelation against numpy, the
error codes, and the md program's files."""
import os
import subprocess

import numpy as np
import pytest

import heat_reference
from mdqtplasmasims_b200 import Engine, MDQTError, SCHEME_NONE, md_params, su_params

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "mdqtplasmasims_b200", "mdqt_run")
EINVAL, ESTATE = -1, -5
TIGHT = [0, 1, 2, 9, 10, 11, 12]            # kinetic sums: 1e-13 of their scales
PAIR = [3, 4, 5, 6, 7, 8, 13, 14]           # pair sums: 1e-12


def _params(kind, n, **kw):
    if kind == "md":
        return md_params(scheme=SCHEME_NONE, n_ions=n, **kw)
    return su_params(n_ions=n, N0=n, **kw)


def _state(n, L, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0, L, size=(3, n)), rng.normal(size=(3, n)) * 0.3


def _record(e, nslots=1, slot=0):
    e.heat_begin(nslots)
    e.heat_record(slot)
    return e.heat_download(nslots)[..., slot]


def _stress(e):
    e.stress_begin(1)
    e.stress_record(0)
    return e.stress_download(1)[..., 0]


@pytest.mark.parametrize("kind", ["md", "su"])
@pytest.mark.parametrize("n", [300, 3500, 4096, 20000])
def test_heat_matches_the_reference(kind, n):
    p = _params(kind, n)
    R, V = _state(n, p.L, n + (0 if kind == "md" else 1))
    e = Engine(p)
    e.upload(R=R, V=V)
    got = _record(e)
    e.close()
    want, scale = heat_reference.heat(R, V, p.L, p.kappa, p.rcut)
    assert np.all(np.abs(got[TIGHT] - want[TIGHT]) <= 1e-13 * scale[TIGHT]), np.abs(got[TIGHT] - want[TIGHT]) / scale[TIGHT]
    assert np.all(np.abs(got[PAIR] - want[PAIR]) <= 1e-12 * scale[PAIR]), np.abs(got[PAIR] - want[PAIR]) / scale[PAIR]


@pytest.mark.parametrize("n", [3500, 20000])
def test_agrees_with_the_device_energy_and_virial(n):
    """E_pot = n Epotential(), tr W = the trace of the stress record; with V = c, J_pot = E_pot c and J_vir = W c against both."""
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    R, V = _state(n, p.L, 31)
    e = Engine(p)
    e.upload(R=R, V=V)
    rec = _record(e)
    st = _stress(e)
    epot = n * e.Epotential()
    assert rec[13] == pytest.approx(epot, rel=1e-13)
    assert rec[14] == pytest.approx(st[6:9].sum(), rel=1e-13)
    c = np.array([0.4, -0.9, 0.25])
    e.upload(R=R, V=np.repeat(c[:, None], n, axis=1))
    rec = _record(e)
    W6 = _stress(e)[6:]
    e.close()
    W = np.array([[W6[0], W6[3], W6[4]], [W6[3], W6[1], W6[5]], [W6[4], W6[5], W6[2]]])
    assert np.allclose(rec[3:6], epot * c, rtol=1e-12, atol=0)
    assert np.all(np.abs(rec[6:9] - W @ c) <= 1e-12 * (np.abs(W) @ np.abs(c)))


@pytest.mark.parametrize("n", [3500, 20000])
def test_negated_velocities_negate_the_currents_exactly(n):
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    R, V = _state(n, p.L, 41)
    e = Engine(p)
    e.upload(R=R, V=V)
    a = _record(e)
    e.upload(R=R, V=-V)
    b = _record(e)
    e.close()
    assert np.array_equal(b[:12], -a[:12])
    assert np.array_equal(b[12:], a[12:])


def test_records_are_reproducible_and_batch_independent():
    n, B = 3500, 8
    p = md_params(scheme=SCHEME_NONE, n_ions=n, n_traj=B)
    R, V = np.zeros((B, 3, n)), np.zeros((B, 3, n))
    for b in range(B):
        R[b], V[b] = _state(n, p.L, 100 + b)
    e = Engine(p)
    e.upload(R=R, V=V)
    e.heat_begin(2)
    e.heat_record(0)
    e.heat_record(1)
    rec = e.heat_download(2)
    e.close()
    assert rec.shape == (B, 15, 2)
    assert np.array_equal(rec[..., 0], rec[..., 1])
    for b in (0, 3, 7):
        e1 = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
        e1.upload(R=R[b], V=V[b])
        assert np.array_equal(_record(e1), rec[b, :, 0]), b
        e1.close()


def test_unequal_ion_counts_match_single_jobs():
    """A 16-job SU batch whose jobs hold different N (mdqt_set_ion_counts): ions beyond a job's count are left out, and every
    job's record has the bits of a handle of its own size."""
    N0, B = 3500, 16
    rng = np.random.default_rng(9)
    counts = rng.integers(3300, 3700, size=B)
    cap = int(counts.max())
    pb = su_params(n_ions=cap, N0=N0, n_traj=B)
    R, V = np.zeros((B, 3, cap)), np.zeros((B, 3, cap))
    for b, nb in enumerate(counts):
        R[b], V[b] = _state(cap, pb.L, 200 + b)  # ions beyond nb hold real-looking data: they must not count
    eb = Engine(pb)
    eb.set_ion_counts(counts)
    eb.upload(R=R, V=V)
    rec = _record(eb)
    eb.close()
    for b in (0, 5, 11, 15):
        nb = int(counts[b])
        e1 = Engine(su_params(n_ions=nb, N0=N0))
        e1.upload(R=R[b][:, :nb], V=V[b][:, :nb])
        assert np.array_equal(_record(e1), rec[b]), b
        e1.close()


def test_recording_leaves_the_state_untouched():
    n = 3500
    p = su_params(n_ions=n, N0=n, seed=5)
    R, V = _state(n, p.L, 3)
    psi = np.zeros((n, 12, 2))
    psi[:, 0, 0] = 1.0
    e = Engine(p)
    e.upload(R=R, V=V, psi=psi, tPart=np.zeros(n), t=0.0, substep=0)
    e.md_steps(2)
    before, F0 = e.download(), e.download_forces()
    e.heat_begin(4)
    for k in range(4):
        e.heat_record(k)
    after, F1 = e.download(), e.download_forces()
    for k in ("R", "V", "psi", "tPart"):
        assert np.array_equal(before[k], after[k]), k
    assert np.array_equal(F0, F1)
    assert (before["t"], before["substep"]) == (after["t"], after["substep"])
    e.close()


def _twins(p, R, V, **up):
    a, b = Engine(p), Engine(p)
    for e in (a, b):
        e.upload(R=R, V=V, **up)
    return a, b


def test_records_between_steps_change_no_trajectory():
    """mdqt_vv_steps (Andersen collisions on) and mdqt_md_steps (the replayed graph's device clock) with records in between end
    bitwise where the same runs without records end."""
    n = 3500
    p = md_params(scheme=SCHEME_NONE, n_ions=n, seed=17)
    R, V = _state(n, p.L, 21)
    a, b = _twins(p, R, V)
    a.heat_begin(3)
    for k in range(3):
        a.heat_record(k)
        a.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
        b.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
    sa, sb = a.download(), b.download()
    assert np.array_equal(sa["R"], sb["R"]) and np.array_equal(sa["V"], sb["V"])
    a.close(); b.close()

    p = su_params(n_ions=n, N0=n, seed=23)
    psi = np.zeros((n, 12, 2))
    psi[:, 0, 0] = 1.0
    a, b = _twins(p, R * (p.L / md_params(n_ions=n).L), V * 0.1, psi=psi, tPart=np.zeros(n), t=0.0, substep=0)
    a.heat_begin(3)
    for k in range(3):
        a.heat_record(k)
        a.md_steps(2)
        b.md_steps(2)
    sa, sb = a.download(), b.download()
    for k in ("R", "V", "psi", "tPart"):
        assert np.array_equal(sa[k], sb[k]), k
    assert (sa["t"], sa["substep"]) == (sb["t"], sb["substep"])
    a.close(); b.close()


@pytest.mark.parametrize("B", [1, 3])
def test_heat_autocorrelation_matches_numpy(B):
    n, T = 2048, 60
    p = md_params(scheme=SCHEME_NONE, n_ions=n, n_traj=B, seed=4)
    R, V = np.zeros((B, 3, n)), np.zeros((B, 3, n))
    for b in range(B):
        R[b], V[b] = _state(n, p.L, 300 + b)
        V[b, 0] += 0.05 * (b + 1)  # a clear total momentum: the enthalpy current matters
    e = Engine(p)
    e.upload(R=R if B > 1 else R[0], V=V if B > 1 else V[0])
    e.heat_begin(T + 5)  # capacity above the records used: the correlator reads the first T
    for k in range(T):
        e.heat_record(k)
        e.MDSteps(1)
    rec = e.heat_download(T).reshape(B, 15, T)
    acf = e.heat_autocorr(T).reshape(B, T)
    e.close()
    for b in range(B):
        want, scale = heat_reference.autocorr(heat_reference.heat_flux(rec[b], n))
        assert np.all(np.abs(acf[b] - want) <= 1e-12 * scale), b
        assert acf[b][0] == pytest.approx(want[0], rel=1e-12)


def test_without_momentum_the_autocorrelation_is_that_of_the_energy_current():
    n, T = 2048, 40
    p = md_params(scheme=SCHEME_NONE, n_ions=n, seed=6)
    R, V = _state(n, p.L, 61)
    V -= V.mean(axis=1, keepdims=True)
    e = Engine(p)
    e.upload(R=R, V=V)
    e.heat_begin(T)
    for k in range(T):
        e.heat_record(k)
        e.MDSteps(1)
    rec = e.heat_download(T)
    acf = e.heat_autocorr(T)
    e.close()
    JE = rec[0:3] + rec[3:6] + rec[6:9]
    want, scale = heat_reference.autocorr(JE)
    # P = 0 up to rounding: hbar P is below 1e-12 of the scale
    assert np.all(np.abs(acf - want) <= 1e-12 * scale)


def test_errors():
    n = 512
    e = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    L, h = e.lib, e.h
    buf = np.zeros(15 * 8)
    ptr = buf.ctypes.data
    assert L.mdqt_heat_record(h, 0) == ESTATE
    assert L.mdqt_heat_download(h, ptr, 1) == ESTATE
    assert L.mdqt_heat_autocorr(h, 1, ptr) == ESTATE
    assert L.mdqt_heat_begin(h, 0) == EINVAL
    assert L.mdqt_heat_begin(h, (1 << 22) + 1) == EINVAL
    assert L.mdqt_heat_begin(None, 4) == EINVAL
    assert L.mdqt_heat_begin(h, 8) == 0
    assert L.mdqt_heat_record(h, -1) == EINVAL
    assert L.mdqt_heat_record(h, 8) == EINVAL
    assert L.mdqt_heat_record(h, 7) == 0
    assert L.mdqt_heat_download(h, None, 8) == EINVAL
    assert L.mdqt_heat_download(h, ptr, 0) == EINVAL
    assert L.mdqt_heat_download(h, ptr, 9) == EINVAL
    assert L.mdqt_heat_download(h, ptr, 8) == 0
    assert L.mdqt_heat_autocorr(h, 8, None) == EINVAL
    assert L.mdqt_heat_autocorr(h, 0, ptr) == EINVAL
    assert L.mdqt_heat_autocorr(h, 9, ptr) == EINVAL
    assert L.mdqt_heat_autocorr(h, 8, ptr) == 0
    e.close()
    # a row-decomposed handle holds its own rows' sums only
    er = Engine(md_params(scheme=SCHEME_NONE, n_ions=n, row0=0, n_rows=n // 2))
    assert er.lib.mdqt_heat_begin(er.h, 4) == ESTATE
    with pytest.raises(MDQTError):
        er.heat_begin(4)
    er.close()
    # a handle with a communicator (one rank owning all rows)
    ec = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    try:
        ec.comm_init(Engine.comm_unique_id(), 0, 1)
    except MDQTError as ex:
        ec.close()
        pytest.skip("no communicator on this machine: %s" % ex)
    assert ec.lib.mdqt_heat_begin(ec.h, 4) == ESTATE
    ec.close()


def _run_md(save, *extra):
    r = subprocess.run([DRIVER, "--program", "md", "1", "--seed", "4321", "--preSteps", "0", "--recordSteps", "40", "--instSteps", "30",
                        "--reequilSteps", "0", "--establishSteps", "20", "--relaxSteps", "20", "--saveDirectory", save, "--quiet", *extra],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return os.path.join(save, "Gamma300Kappa50NumIons4096", "job1")


def test_md_program_heat_files(tmp_path):
    n, T, dt = 4096, 40, 0.005
    d0 = _run_md(str(tmp_path / "plain") + "/")
    d1 = _run_md(str(tmp_path / "heat") + "/", "--heat", "1")
    f0, f1 = sorted(os.listdir(d0)), sorted(os.listdir(d1))
    assert "heatCurrent.dat" not in f0 and "heatAutoCorr.dat" not in f0
    assert f1 == sorted(f0 + ["heatAutoCorr.dat", "heatCurrent.dat"])
    for f in f0:
        assert open(os.path.join(d0, f), "rb").read() == open(os.path.join(d1, f), "rb").read(), f
    hc = np.loadtxt(os.path.join(d1, "heatCurrent.dat"))
    ac = np.loadtxt(os.path.join(d1, "heatAutoCorr.dat"))
    assert hc.shape == (T, 16) and ac.shape == (T, 3)
    assert np.allclose(hc[:, 0], np.arange(T) * dt, rtol=0, atol=1e-15)
    Jq = heat_reference.heat_flux(hc[:, 1:].T, n)
    assert ac[0, 1] == pytest.approx((Jq ** 2).sum(axis=0).mean() / 3, rel=1e-12)
    temp = np.loadtxt(os.path.join(d1, "temperature.dat"))
    tk = 2 * hc[:, 13] / (3 * n)
    assert [float("%g" % x) for x in tk] == list(temp)
    # lambda(tD): trapezoid integral of C over V Tbar^2
    Lbox = md_params(n_ions=n).L
    lam = np.concatenate([[0.0], np.cumsum(0.5 * (ac[1:, 1] + ac[:-1, 1]) * dt)]) / (Lbox ** 3 * tk.mean() ** 2)
    assert np.allclose(ac[:, 2], lam, rtol=1e-12, atol=1e-15 * np.abs(lam).max())
