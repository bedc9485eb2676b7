"""GPU suite: the density and current Fourier mode recorder mdqt_modes_* and `mdqt_run --program md --modes NMAX`.

Against the test-side reference (tests/modes_reference.py, long double phases) in both parameter families, the exact periodicity of
the fixed-point phase, the sign symmetries under V -> -V and R -> -R, continuity along device velocity-Verlet steps, bitwise
reproducibility (repeat, batch vs single, unequal ion counts), no side effects on the state or on later steps, the correlator against
the reference's loops, equipartition of the currents, the error codes, and the md program's files."""
import math
import os
import subprocess

import numpy as np
import pytest

import modes_reference as mr
from mdqtplasmasims_b200 import Engine, MDQTError, SCHEME_NONE, axis_wavevectors, md_params, su_params

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


def _nvec(seed, nmax=32, extra=6, cmax=200):
    rng = np.random.default_rng(seed)
    r = rng.integers(-cmax, cmax + 1, size=(extra, 3))
    r[np.all(r == 0, axis=1)] = [cmax, -1, 3]
    return np.concatenate([axis_wavevectors(nmax), r]).astype(np.int32)


def _record(e, nvec, nslots=1, slot=0):
    e.modes_begin(nvec, nslots)
    e.modes_record(slot)
    return e.modes_download(nslots)[..., slot]


@pytest.mark.parametrize("kind", ["md", "su"])
@pytest.mark.parametrize("n", [300, 3500, 4096, 20000])
def test_modes_match_the_reference(kind, n):
    p = _params(kind, n)
    R, V = _state(n, p.L, n + (0 if kind == "md" else 1))
    nvec = _nvec(n)
    assert len(nvec) % 4 == 2  # a part-filled last tile of the record kernel
    e = Engine(p)
    e.upload(R=R, V=V)
    got = _record(e, nvec)
    e.close()
    want, scale = mr.modes(R, V, p.L, nvec)
    err = np.abs(got - want) / scale
    assert err.max() <= 1e-14, (err.max(), np.unravel_index(err.argmax(), err.shape))


def test_whole_box_shifts_give_the_same_bits():
    """L = 16 and positions on a 2^-30 grid: shifting ions by +-L or +-2L is exact in double and leaves the fixed-point phase bitwise."""
    n = 2000
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    p.L, p.rcut = 16.0, 8.0
    rng = np.random.default_rng(7)
    R = rng.integers(0, 16 << 30, size=(3, n)) / 2.0 ** 30
    V = rng.normal(size=(3, n))
    nvec = _nvec(8, nmax=8, cmax=(1 << 20) - 1)
    e = Engine(p)
    e.upload(R=R, V=V)
    a = _record(e, nvec)
    for seed in range(3):
        sh = np.random.default_rng(seed).choice([-2, -1, 0, 0, 1, 2], size=(3, n)) * 16.0
        e.upload(R=R + sh, V=V)
        assert np.array_equal(_record(e, nvec), a), seed
    e.close()


def test_sign_symmetries():
    n = 3500
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    R, V = _state(n, p.L, 11)
    nvec = _nvec(11)
    e = Engine(p)
    e.upload(R=R, V=V)
    a = _record(e, nvec)
    e.upload(R=R, V=-V)
    b = _record(e, nvec)
    assert np.array_equal(b[:, :2], a[:, :2])
    assert np.array_equal(b[:, 2:], -a[:, 2:])
    e.upload(R=-R, V=V)
    c = _record(e, nvec)
    e.close()
    _, scale = mr.modes(R, V, p.L, nvec)
    conj = a * np.array([1, -1, 1, -1, 1, -1, 1, -1])
    assert np.all(np.abs(c - conj) <= 1e-15 * scale)


def _lattice_state(side, L, seed, jitter=0.1, sigma=0.6):
    rng = np.random.default_rng(seed)
    g = (np.arange(side) + 0.5) * (L / side)
    R = np.array(np.meshgrid(g, g, g, indexing="ij")).reshape(3, -1)
    R = R + rng.uniform(-jitter, jitter, size=R.shape) * (L / side)
    return R, rng.normal(size=R.shape) * sigma


def test_continuity_along_device_steps():
    """[rho(t + dt) - rho(t - dt)] / (2 dt) = i k.j(t) + O(dt^2) along collisionless velocity-Verlet steps on the device."""
    side = 16
    p = md_params(scheme=SCHEME_NONE, n_ions=side ** 3)
    R, V = _lattice_state(side, p.L, 5)
    nvec = axis_wavevectors(4)
    kv = 2 * np.pi * nvec / p.L
    errs = []
    for dt in (0.02, 0.01):
        e = Engine(p)
        e.upload(R=R, V=V)
        e.modes_begin(nvec, 3)
        for s in range(3):
            e.modes_record(s)
            if s < 2:
                e.MDStep(dt=dt, collisionFreq=0.0)
        rec = e.modes_download(3)
        e.close()
        rho, j = mr.complex_modes(rec)
        d = (rho[:, 2] - rho[:, 0]) / (2 * dt)
        want = 1j * np.einsum("qa,qa->q", kv, j[:, :, 1])
        errs.append(np.abs(d - want).max() / np.abs(want).max())
    assert errs[0] < 1e-3, errs
    assert 3 < errs[0] / errs[1] < 5, errs


def test_records_are_reproducible_and_batch_independent():
    n, B = 3500, 8
    p = md_params(scheme=SCHEME_NONE, n_ions=n, n_traj=B)
    R, V = np.zeros((B, 3, n)), np.zeros((B, 3, n))
    for b in range(B):
        R[b], V[b] = _state(n, p.L, 100 + b)
    nvec = _nvec(3)
    e = Engine(p)
    e.upload(R=R, V=V)
    e.modes_begin(nvec, 2)
    e.modes_record(0)
    e.modes_record(1)
    rec = e.modes_download(2)
    e.close()
    assert rec.shape == (B, len(nvec), 8, 2)
    assert np.array_equal(rec[..., 0], rec[..., 1])
    for b in (0, 3, 7):
        e1 = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
        e1.upload(R=R[b], V=V[b])
        assert np.array_equal(_record(e1, nvec), rec[b, ..., 0]), b
        e1.close()


def test_unequal_ion_counts_match_single_jobs():
    """Ions beyond a job's count hold garbage and are left out: every job's record has the bits of a handle of its own size."""
    N0, B = 3500, 16
    rng = np.random.default_rng(9)
    counts = rng.integers(3300, 3700, size=B)
    cap = int(counts.max())
    pb = su_params(n_ions=cap, N0=N0, n_traj=B)
    R, V = np.zeros((B, 3, cap)), np.zeros((B, 3, cap))
    for b in range(B):
        R[b], V[b] = _state(cap, pb.L, 200 + b)
    nvec = _nvec(4)
    eb = Engine(pb)
    eb.set_ion_counts(counts)
    eb.upload(R=R, V=V)
    rec = _record(eb, nvec)
    for b, nb in enumerate(counts):  # other garbage in the padding
        R[b][:, nb:] = rng.uniform(-1e3, 1e3, size=(3, cap - nb))
        V[b][:, nb:] = rng.normal(size=(3, cap - nb)) * 1e3
    eb.upload(R=R, V=V)
    assert np.array_equal(_record(eb, nvec), rec)
    eb.close()
    for b in (0, 5, 11, 15):
        nb = int(counts[b])
        e1 = Engine(su_params(n_ions=nb, N0=N0))
        e1.upload(R=R[b][:, :nb], V=V[b][:, :nb])
        assert np.array_equal(_record(e1, nvec), rec[b]), b
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
    e.modes_begin(_nvec(5), 4)
    for k in range(4):
        e.modes_record(k)
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
    n = 3500
    nvec = _nvec(6)
    p = md_params(scheme=SCHEME_NONE, n_ions=n, seed=17)
    R, V = _state(n, p.L, 21)
    a, b = _twins(p, R, V)
    a.modes_begin(nvec, 3)
    for k in range(3):
        a.modes_record(k)
        a.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
        b.MDSteps(4, collisionFreq=0.25, sigma_v=0.5)
    sa, sb = a.download(), b.download()
    assert np.array_equal(sa["R"], sb["R"]) and np.array_equal(sa["V"], sb["V"])
    a.close(); b.close()

    p = su_params(n_ions=n, N0=n, seed=23)
    psi = np.zeros((n, 12, 2))
    psi[:, 0, 0] = 1.0
    a, b = _twins(p, R * (p.L / md_params(n_ions=n).L), V * 0.1, psi=psi, tPart=np.zeros(n), t=0.0, substep=0)
    a.modes_begin(nvec, 3)
    for k in range(3):
        a.modes_record(k)
        a.md_steps(2)
        b.md_steps(2)
    sa, sb = a.download(), b.download()
    for k in ("R", "V", "psi", "tPart"):
        assert np.array_equal(sa[k], sb[k]), k
    assert (sa["t"], sa["substep"]) == (sb["t"], sb["substep"])
    a.close(); b.close()


def _scale(rec, n, nvec):
    """The correlations of |components|: a bound on the sums the device forms, for tolerances."""
    a = np.abs(rec)
    F = mr.correlations(a, n, nvec)[0]
    jl = (a[:, 2::2] ** 2 + a[:, 3::2] ** 2).sum(axis=1)  # |j|^2 summed over components bounds both currents' products
    T = rec.shape[-1]
    s = np.array([[np.sqrt(jl[q, :T - t] * jl[q, t:]).sum() / (n * (T - t)) for t in range(T)] for q in range(len(nvec))])
    return F, s


def test_autocorrelation_matches_the_reference():
    """T = 2500 records of two SU trajectories with unequal ion counts."""
    N0, B, T = 3500, 2, 2500
    counts = np.array([3500, 3120])
    p = su_params(n_ions=int(counts.max()), N0=N0, n_traj=B, seed=8)
    R, V = np.zeros((B, 3, p.n_ions)), np.zeros((B, 3, p.n_ions))
    for b in range(B):
        R[b], V[b] = _state(p.n_ions, p.L, 400 + b)
    V *= 0.2
    psi = np.zeros((B, p.n_ions, 12, 2))
    psi[..., 0, 0] = 1.0
    nvec = np.concatenate([axis_wavevectors(2), [[1, 1, 0], [2, -1, 3]]]).astype(np.int32)
    e = Engine(p)
    e.set_ion_counts(counts)
    e.upload(R=R, V=V, psi=psi, tPart=np.zeros((B, p.n_ions)), t=0.0, substep=0)
    e.modes_begin(nvec, T + 7)  # capacity above the records used: the correlator reads the first T
    for k in range(T):
        e.modes_record(k)
        e.md_steps(1)
    rec = e.modes_download(T)
    F, CL, CT = e.modes_autocorr(T)
    Fs, CLs, CTs = e.modes_autocorr(T // 2)
    e.close()
    assert F.shape == CL.shape == CT.shape == (B, len(nvec), T)
    for b in range(B):
        n = int(counts[b])
        want = mr.correlations(rec[b], n, nvec)
        sF, sJ = _scale(rec[b], n, nvec)
        for got, w, s in zip((F[b], CL[b], CT[b]), want, (sF, sJ, sJ)):
            assert np.all(np.abs(got - w) <= 1e-12 * s), b
        rho, j = mr.complex_modes(rec[b])
        assert np.allclose(CL[b, :, 0] + 2 * CT[b, :, 0], (np.abs(j) ** 2).sum(axis=(1, 2)) / (n * T), rtol=1e-12, atol=0)
        assert np.allclose(F[b, :, 0], (np.abs(rho) ** 2).sum(axis=1) / (n * T), rtol=1e-12, atol=0)
        wF = mr.correlations(rec[b][..., :T // 2], n, nvec)[0]
        assert np.allclose(Fs[b], wF, rtol=0, atol=1e-12 * np.abs(wF).max())


def test_autocorrelation_skips_null_outputs():
    n, T = 1000, 20
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    R, V = _state(n, p.L, 12)
    e = Engine(p)
    e.upload(R=R, V=V)
    nvec = _nvec(12, nmax=2, extra=1)
    e.modes_begin(nvec, T)
    for k in range(T):
        e.modes_record(k)
        e.MDStep()
    F, CL, CT = e.modes_autocorr(T)
    out = np.full((len(nvec), T), np.nan)
    assert e.lib.mdqt_modes_autocorr(e.h, T, None, out.ctypes.data, None) == 0
    assert np.array_equal(out, CL)
    e.close()


def test_equipartition_of_the_currents():
    """Maxwellian V independent of R: C_L(k, 0) and C_T(k, 0), averaged over k and records, equal <v_a^2>."""
    n, T = 4096, 200
    p = md_params(scheme=SCHEME_NONE, n_ions=n)
    nvec = axis_wavevectors(32)
    rng = np.random.default_rng(13)
    e = Engine(p)
    e.modes_begin(nvec, T)
    v2 = 0.0
    for k in range(T):
        V = rng.normal(size=(3, n)) * 0.7
        e.upload(R=rng.uniform(0, p.L, size=(3, n)), V=V)
        e.modes_record(k)
        v2 += (V ** 2).mean() / T
    F, CL, CT = e.modes_autocorr(T)
    e.close()
    assert CL[:, 0].mean() == pytest.approx(v2, rel=0.05)
    assert CT[:, 0].mean() == pytest.approx(v2, rel=0.05)
    assert F[:, 0].mean() == pytest.approx(1.0, rel=0.05)  # uncorrelated positions: S(k) = 1


def test_errors():
    n = 512
    e = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    L, h = e.lib, e.h
    buf = np.zeros(8 * 64)
    ptr = buf.ctypes.data
    nv = np.ascontiguousarray(axis_wavevectors(2), dtype=np.int32)
    nvp = nv.ctypes.data

    def begin(vecs, K=None, nslots=4):
        a = np.ascontiguousarray(vecs, dtype=np.int32)
        return L.mdqt_modes_begin(h, a.ctypes.data, len(a) if K is None else K, nslots)

    assert L.mdqt_modes_record(h, 0) == ESTATE
    assert L.mdqt_modes_download(h, ptr, 1) == ESTATE
    assert L.mdqt_modes_autocorr(h, 1, ptr, None, None) == ESTATE
    assert L.mdqt_modes_begin(None, nvp, 6, 4) == EINVAL
    assert L.mdqt_modes_begin(h, None, 6, 4) == EINVAL
    assert L.mdqt_modes_begin(h, nvp, 0, 4) == EINVAL
    assert begin(np.ones((1025, 3))) == EINVAL
    assert L.mdqt_modes_begin(h, nvp, 6, 0) == EINVAL
    assert begin([[1, 0, 0], [0, 0, 0]]) == EINVAL
    assert begin([[1 << 20, 0, 0]]) == EINVAL
    assert begin([[0, -(1 << 20), 1]]) == EINVAL
    assert begin([[(1 << 20) - 1, -(1 << 20) + 1, 1]]) == 0
    assert begin(np.ones((1024, 3))) == 0
    assert L.mdqt_modes_begin(h, nvp, 6, 8) == 0
    assert L.mdqt_modes_record(h, -1) == EINVAL
    assert L.mdqt_modes_record(h, 8) == EINVAL
    assert L.mdqt_modes_record(h, 7) == 0
    assert L.mdqt_modes_download(h, None, 8) == EINVAL
    assert L.mdqt_modes_download(h, ptr, 0) == EINVAL
    assert L.mdqt_modes_download(h, ptr, 9) == EINVAL
    assert L.mdqt_modes_download(h, ptr, 8) == 0
    assert L.mdqt_modes_autocorr(h, 0, ptr, None, None) == EINVAL
    assert L.mdqt_modes_autocorr(h, 9, ptr, None, None) == EINVAL
    assert L.mdqt_modes_autocorr(h, 8, ptr, None, None) == 0
    # above the correlator's limit of 6144 records
    assert L.mdqt_modes_begin(h, nvp, 1, 6145) == 0
    assert L.mdqt_modes_autocorr(h, 6145, ptr, None, None) == EINVAL
    with pytest.raises(MDQTError):
        e.modes_begin(np.zeros((2, 3)), 4)
    e.close()
    # a row-decomposed handle holds its own rows only
    er = Engine(md_params(scheme=SCHEME_NONE, n_ions=n, row0=0, n_rows=n // 2))
    assert er.lib.mdqt_modes_begin(er.h, nvp, 6, 4) == ESTATE
    with pytest.raises(MDQTError):
        er.modes_begin(nv, 4)
    er.close()
    # a handle with a communicator (one rank owning all rows)
    ec = Engine(md_params(scheme=SCHEME_NONE, n_ions=n))
    try:
        ec.comm_init(Engine.comm_unique_id(), 0, 1)
    except MDQTError as ex:
        ec.close()
        pytest.skip("no communicator on this machine: %s" % ex)
    assert ec.lib.mdqt_modes_begin(ec.h, nvp, 6, 4) == ESTATE
    ec.close()


def _run_md(save, *extra):
    r = subprocess.run([DRIVER, "--program", "md", "1", "--seed", "4321", "--preSteps", "0", "--recordSteps", "200", "--instSteps", "30",
                        "--reequilSteps", "0", "--establishSteps", "20", "--relaxSteps", "20", "--saveDirectory", save, "--quiet", *extra],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return os.path.join(save, "Gamma300Kappa50NumIons4096", "job1")


def _mt19937_normals(seed, count, sigma):
    """std::normal_distribution<double>(0, sigma) over std::mt19937(seed) as libstdc++ draws it (Marsaglia's polar method on
    generate_canonical<double, 53>, two 32-bit words per uniform): the md program's Maxwellian init()."""
    rs = np.random.RandomState(seed)  # the same init_genrand seeding and 32-bit output sequence as std::mt19937

    def canonical():
        lo, hi = (int(x) for x in rs.randint(0, 2 ** 32, size=2, dtype=np.uint64))
        r = (lo + hi * 2.0 ** 32) / 2.0 ** 64
        return r if r < 1.0 else math.nextafter(1.0, 0.0)

    out = []
    while len(out) < count:
        while True:
            x, y = 2.0 * canonical() - 1.0, 2.0 * canonical() - 1.0
            r2 = x * x + y * y
            if r2 <= 1.0 and r2 != 0.0:
                break
        mult = math.sqrt(-2 * math.log(r2) / r2)
        out += [y * mult * sigma, x * mult * sigma]
    return out[:count]


def test_md_program_modes_files(tmp_path):
    N, T, dt, nmax, Gamma, seed = 4096, 200, 0.005, 8, 3.0, 4321
    d0 = _run_md(str(tmp_path / "plain") + "/")
    dz = _run_md(str(tmp_path / "zero") + "/", "--modes", "0")
    d1 = _run_md(str(tmp_path / "modes") + "/", "--modes", str(nmax))
    new = ["currentCorrL.dat", "currentCorrT.dat", "intermediateScattering.dat", "staticStructureFactor.dat"]
    f0, fz, f1 = sorted(os.listdir(d0)), sorted(os.listdir(dz)), sorted(os.listdir(d1))
    assert fz == f0 and not set(new) & set(f0)
    assert f1 == sorted(f0 + new)
    for f in f0:
        b0 = open(os.path.join(d0, f), "rb").read()
        assert open(os.path.join(dz, f), "rb").read() == b0, f
        assert open(os.path.join(d1, f), "rb").read() == b0, f
    tabs = {f: np.loadtxt(os.path.join(d1, f)) for f in new}
    for f in new[:3]:
        assert tabs[f].shape == (T, nmax + 1), f
        assert np.allclose(tabs[f][:, 0], np.arange(T) * dt, rtol=0, atol=1e-15)
    sk = tabs["staticStructureFactor.dat"]
    L = md_params(n_ions=N).L
    assert sk.shape == (nmax, 3)
    assert np.array_equal(sk[:, 0], np.arange(1, nmax + 1))
    assert np.allclose(sk[:, 1], 2 * np.pi * np.arange(1, nmax + 1) / L, rtol=1e-15, atol=0)
    assert np.array_equal(sk[:, 2], tabs["intermediateScattering.dat"][0, 1:])

    # the same recording stage on an engine: the program's lattice + Maxwellian init() with the same seed, then T collisionless
    # steps with a record before each
    side = 16
    R = np.zeros((3, N))
    V = np.array(_mt19937_normals(seed, 3 * N, math.sqrt(1 / Gamma))).reshape(N, 3).T
    for i0, (i, j, k) in enumerate((i, j, k) for i in range(side) for j in range(side) for k in range(side)):
        R[:, i0] = [c * L / N ** (1 / 3.) + 0.5 for c in (i, j, k)]
    p = md_params(scheme=SCHEME_NONE, n_ions=N)
    p.traj0, p.seed = 1, seed
    e = Engine(p)
    e.upload(R=R, V=V)
    e.modes_begin(axis_wavevectors(nmax), T)
    for k in range(T):
        e.modes_record(k)
        e.MDStep(dt=dt, collisionFreq=0.0, sigma_v=math.sqrt(1 / Gamma))
    rec = e.modes_download(T)
    e.close()
    s0 = ((rec[:, 0] ** 2 + rec[:, 1] ** 2).mean(axis=1) / N).reshape(nmax, 3).mean(axis=1)
    assert np.allclose(tabs["intermediateScattering.dat"][0, 1:], s0, rtol=1e-9, atol=0)
