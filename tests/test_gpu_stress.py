"""GPU suite: the pressure (stress) tensor recorder mdqt_stress_* and `mdqt_run --program md --stress 1`.

Against the test-side reference (tests/stress_reference.py) in both force plans (item walk for N <= 8192, CTA tiles beyond), the virial scaling identity
against the device's own potential energy, bitwise reproducibility (repeat, batch vs single, unequal ion counts), no side effects
on the state or on later steps, the shear-stress autocorrelation against numpy, the error codes, and the md program's files."""
import os
import subprocess

import numpy as np
import pytest

import stress_reference
from mdqtplasmasims_b200 import Engine, MDQTError, SCHEME_NONE, md_params, su_params

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "mdqtplasmasims_b200", "mdqt_run")
EINVAL, ESTATE = -1, -5


def _params(kind, n, **kw):
    if kind == "md":
        return md_params(scheme=SCHEME_NONE, n_ions=n, **kw)
    return su_params(n_ions=n, N0=n, **kw)


def _state(n, L, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0, L, size=(3, n)), rng.normal(size=(3, n)) * 0.3


def _record(e, nslots=1, slot=0):
    e.stress_begin(nslots)
    e.stress_record(slot)
    return e.stress_download(nslots)[..., slot]


@pytest.mark.parametrize("kind", ["md", "su"])
@pytest.mark.parametrize("n", [300, 3500, 4096, 20000])
def test_stress_matches_the_reference(kind, n):
    p = _params(kind, n)
    R, V = _state(n, p.L, n + (0 if kind == "md" else 1))
    e = Engine(p)
    e.upload(R=R, V=V)
    got = _record(e)
    e.close()
    want, scale = stress_reference.stress(R, V, p.L, p.kappa, p.rcut)
    # K: 1e-13 of sum |v_a v_b| (= |K_aa| on the diagonal: rtol 1e-13 there); W: 1e-12 of sum |d_a d_b f|
    assert np.all(np.abs(got[:6] - want[:6]) <= 1e-13 * scale[:6]), np.abs(got[:6] - want[:6]) / scale[:6]
    assert np.all(np.abs(got[6:] - want[6:]) <= 1e-12 * scale[6:]), np.abs(got[6:] - want[6:]) / scale[6:]


@pytest.mark.parametrize("n", [3500, 20000])
def test_trace_of_w_is_minus_the_scale_derivative_of_the_energy(n):
    """Positions, L and rcut scaled together by s keep the pair set: tr W = -d(N Epot)/ds at s = 1 (central difference of mdqt_epot)."""
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    R, V = _state(n, p.L, 7)
    e = Engine(p)
    e.upload(R=R, V=V)
    trW = _record(e)[6:9].sum()
    e.close()
    h = 1e-4
    E = []
    for s in (1 + h, 1 - h):
        es = Engine(md_params(scheme=SCHEME_NONE, n_ions=n, L=p.L * s, rcut=p.L * s / 2))
        es.upload(R=R * s, V=V)
        E.append(n * es.Epotential())
        es.close()
    dEds = (E[0] - E[1]) / (2 * h)
    assert abs(trW + dEds) <= 1e-7 * abs(trW), (trW, -dEds)


def test_records_are_reproducible_and_batch_independent():
    n, B = 3500, 8
    p = md_params(scheme=SCHEME_NONE, n_ions=n, n_traj=B)
    R, V = np.zeros((B, 3, n)), np.zeros((B, 3, n))
    for b in range(B):
        R[b], V[b] = _state(n, p.L, 100 + b)
    e = Engine(p)
    e.upload(R=R, V=V)
    e.stress_begin(2)
    e.stress_record(0)
    e.stress_record(1)
    rec = e.stress_download(2)
    e.close()
    assert rec.shape == (B, 12, 2)
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
    e.stress_begin(4)
    for k in range(4):
        e.stress_record(k)
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
    """mdqt_vv_steps (Andersen collisions on: the Philox stream follows the step counter) and mdqt_md_steps (the device clock of
    the replayed graph) with records in between end bitwise where the same runs without records end."""
    n = 3500
    p = md_params(scheme=SCHEME_NONE, n_ions=n, seed=17)
    R, V = _state(n, p.L, 21)
    a, b = _twins(p, R, V)
    a.stress_begin(3)
    for k in range(3):
        a.stress_record(k)
        a.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
        b.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
    sa, sb = a.download(), b.download()
    assert np.array_equal(sa["R"], sb["R"]) and np.array_equal(sa["V"], sb["V"])
    a.close(); b.close()

    p = su_params(n_ions=n, N0=n, seed=23)
    psi = np.zeros((n, 12, 2))
    psi[:, 0, 0] = 1.0
    a, b = _twins(p, R * (p.L / md_params(n_ions=n).L), V * 0.1, psi=psi, tPart=np.zeros(n), t=0.0, substep=0)
    a.stress_begin(3)
    for k in range(3):
        a.stress_record(k)
        a.md_steps(2)
        b.md_steps(2)
    sa, sb = a.download(), b.download()
    for k in ("R", "V", "psi", "tPart"):
        assert np.array_equal(sa[k], sb[k]), k
    assert (sa["t"], sa["substep"]) == (sb["t"], sb["substep"])
    a.close(); b.close()


@pytest.mark.parametrize("B", [1, 3])
def test_shear_autocorrelation_matches_numpy(B):
    n, T = 2048, 60
    p = md_params(scheme=SCHEME_NONE, n_ions=n, n_traj=B, seed=4)
    R, V = np.zeros((B, 3, n)), np.zeros((B, 3, n))
    for b in range(B):
        R[b], V[b] = _state(n, p.L, 300 + b)
    e = Engine(p)
    e.upload(R=R if B > 1 else R[0], V=V if B > 1 else V[0])
    e.stress_begin(T + 5)  # capacity above the records used: the correlator reads the first T
    for k in range(T):
        e.stress_record(k)
        e.MDSteps(1)
    rec = e.stress_download(T).reshape(B, 12, T)
    acf = e.stress_autocorr(T).reshape(B, T)
    e.close()
    for b in range(B):
        P = rec[b, 3:6] + rec[b, 9:12]  # P_xy, P_xz, P_yz
        want = np.array([(P[:, :T - t] * P[:, t:]).sum() / (3 * (T - t)) for t in range(T)])
        scale = np.array([np.abs(P[:, :T - t] * P[:, t:]).sum() / (3 * (T - t)) for t in range(T)])
        assert np.all(np.abs(acf[b] - want) <= 1e-12 * scale), b
        assert acf[b][0] == pytest.approx(want[0], rel=1e-12)


def test_errors():
    n = 512
    e = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    L, h = e.lib, e.h
    buf = np.zeros(12 * 8)
    ptr = buf.ctypes.data
    assert L.mdqt_stress_record(h, 0) == ESTATE
    assert L.mdqt_stress_download(h, ptr, 1) == ESTATE
    assert L.mdqt_stress_autocorr(h, 1, ptr) == ESTATE
    assert L.mdqt_stress_begin(h, 0) == EINVAL
    assert L.mdqt_stress_begin(h, (1 << 22) + 1) == EINVAL
    assert L.mdqt_stress_begin(None, 4) == EINVAL
    assert L.mdqt_stress_begin(h, 8) == 0
    assert L.mdqt_stress_record(h, -1) == EINVAL
    assert L.mdqt_stress_record(h, 8) == EINVAL
    assert L.mdqt_stress_record(h, 7) == 0
    assert L.mdqt_stress_download(h, None, 8) == EINVAL
    assert L.mdqt_stress_download(h, ptr, 0) == EINVAL
    assert L.mdqt_stress_download(h, ptr, 9) == EINVAL
    assert L.mdqt_stress_download(h, ptr, 8) == 0
    assert L.mdqt_stress_autocorr(h, 8, None) == EINVAL
    assert L.mdqt_stress_autocorr(h, 0, ptr) == EINVAL
    assert L.mdqt_stress_autocorr(h, 9, ptr) == EINVAL
    assert L.mdqt_stress_autocorr(h, 8, ptr) == 0
    e.close()
    # a row-decomposed handle holds its own rows' sums only
    er = Engine(md_params(scheme=SCHEME_NONE, n_ions=n, row0=0, n_rows=n // 2))
    assert er.lib.mdqt_stress_begin(er.h, 4) == ESTATE
    with pytest.raises(MDQTError):
        er.stress_begin(4)
    er.close()
    # a handle with a communicator (one rank owning all rows)
    ec = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    try:
        ec.comm_init(Engine.comm_unique_id(), 0, 1)
    except MDQTError as ex:
        ec.close()
        pytest.skip("no communicator on this machine: %s" % ex)
    assert ec.lib.mdqt_stress_begin(ec.h, 4) == ESTATE
    ec.close()


def _run_md(save, *extra):
    r = subprocess.run([DRIVER, "--program", "md", "1", "--seed", "4321", "--preSteps", "0", "--recordSteps", "40", "--instSteps", "30",
                        "--reequilSteps", "0", "--establishSteps", "20", "--relaxSteps", "20", "--saveDirectory", save, "--quiet", *extra],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return os.path.join(save, "Gamma300Kappa50NumIons4096", "job1")


def test_md_program_stress_files(tmp_path):
    n, T, dt = 4096, 40, 0.005
    d0 = _run_md(str(tmp_path / "plain") + "/")
    d1 = _run_md(str(tmp_path / "stress") + "/", "--stress", "1")
    f0, f1 = sorted(os.listdir(d0)), sorted(os.listdir(d1))
    assert "stressTensor.dat" not in f0 and "stressAutoCorr.dat" not in f0
    assert f1 == sorted(f0 + ["stressAutoCorr.dat", "stressTensor.dat"])
    for f in f0:
        assert open(os.path.join(d0, f), "rb").read() == open(os.path.join(d1, f), "rb").read(), f
    st = np.loadtxt(os.path.join(d1, "stressTensor.dat"))
    ac = np.loadtxt(os.path.join(d1, "stressAutoCorr.dat"))
    assert st.shape == (T, 13) and ac.shape == (T, 3)
    assert np.allclose(st[:, 0], np.arange(T) * dt, rtol=0, atol=1e-15)
    P = st[:, 4:7] + st[:, 10:13]
    assert ac[0, 1] == pytest.approx((P ** 2).mean(), rel=1e-12)
    temp = np.loadtxt(os.path.join(d1, "temperature.dat"))
    tk = st[:, 1:4].sum(axis=1) / (3 * n)
    assert [float("%g" % x) for x in tk] == list(temp)
    # eta(tD): trapezoid integral of C over V Tbar
    Lbox = md_params(n_ions=n).L
    eta = np.concatenate([[0.0], np.cumsum(0.5 * (ac[1:, 1] + ac[:-1, 1]) * dt)]) / (Lbox ** 3 * tk.mean())
    assert np.allclose(ac[:, 2], eta, rtol=1e-12, atol=1e-15 * np.abs(eta).max())
