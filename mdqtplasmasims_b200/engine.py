"""Host-side mirror of the reference's hot-path interface, over the C ABI of ``libmdqt_b200.so``.

The reference (tlangin/MDQTPlasmaSims) exposes its hot path as ``void f(void)`` functions working on file-scope
globals (``forces()`` SU:192, ``step()`` SU:418, ``qstep()`` SU:438, ``Epotential()`` SU:244, ``output()`` SU:917;
``calculateAccelerations()`` MD:387, ``MDStep()`` MD:504; 7-level ``qstep()`` MC408L:555).  :class:`Engine` keeps
those names and argument meanings, with the globals living in GPU memory behind a handle.  Everything here is
plumbing (ctypes + numpy); all arithmetic happens in the CUDA kernels.  There is no CPU fallback: if the shared
library is missing or no GPU is present, construction raises.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MDQT_LIB_PATH") or os.path.join(HERE, "libmdqt_b200.so")  # env: kernel A/B builds

SCHEME_NONE, SCHEME_SR7, SCHEME_SR12, SCHEME_CA5, SCHEME_V3 = 0, 7, 12, 5, 3
c_double_p = ctypes.POINTER(ctypes.c_double)


class MDQTError(RuntimeError):
    pass


class Params(ctypes.Structure):
    """``mdqt_params`` of include/mdqt.h (same field order)."""
    _fields_ = [(k, ctypes.c_int32) for k in (
        "struct_bytes", "scheme", "n_ions", "n_traj", "traj0", "row0", "n_rows", "device", "substeps_per_md",
        "renormalize", "quad", "plan_n")] + [(k, ctypes.c_double) for k in (
            "L", "kappa", "rcut", "dtq", "detuning", "detuningDP", "Om", "OmDP", "dR", "kRat", "vKick", "vKickDP", "g2E",
            "pv2qv", "fracOfSig", "Te", "sig0", "density")] + [("seed", ctypes.c_uint64)]


class Diag(ctypes.Structure):
    _fields_ = [(k, ctypes.c_double) for k in ("t", "ekin_x", "ekin_y", "ekin_z", "epot", "vx_avg")]


# every symbol include/mdqt.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "mdqt_params_su", "mdqt_params_md", "mdqt_device_count", "mdqt_last_error", "mdqt_version", "mdqt_create",
    "mdqt_destroy", "mdqt_sync", "mdqt_upload_state", "mdqt_download_state", "mdqt_upload_forces",
    "mdqt_download_forces", "mdqt_set_time", "mdqt_get_time", "mdqt_forces", "mdqt_substeps", "mdqt_md_steps",
    "mdqt_md_steps_host", "mdqt_epot", "mdqt_diagnostics", "mdqt_vel_dist", "mdqt_populations", "mdqt_vv_step",
    "mdqt_qsteps", "mdqt_set_forced_uniforms", "mdqt_set_forced_collisions", "mdqt_philox_uniforms", "mdqt_device_ptr",
    "mdqt_device_ld", "mdqt_stream", "mdqt_mark_wrapped", "mdqt_force_plan", "mdqt_enable_timing",
    "mdqt_kernel_time_ms", "mdqt_fp64_peak", "mdqt_params_ts", "mdqt_leapfrog_step", "mdqt_advance_time",
    "mdqt_tag_particles", "mdqt_vaf", "mdqt_vsq_autocorr", "mdqt_set_forced_tag_uniforms", "mdqt_pair_correlation", "mdqt_vstore_begin",
    "mdqt_vstore_record", "mdqt_vstore_upload", "mdqt_autocorrelations", "mdqt_diag_partial", "mdqt_vel_dist_partial",
    "mdqt_vv_steps", "mdqt_set_ion_counts", "mdqt_set_traj_seeds", "mdqt_time_forces", "mdqt_comm_unique_id", "mdqt_comm_init", "mdqt_comm_destroy",
    "mdqt_comm_exchange_positions", "mdqt_comm_allreduce", "mdqt_populations_rows", "mdqt_download_rows", "mdqt_set_tags", "mdqt_moments_begin", "mdqt_moments_record",
    "mdqt_moments_download", "mdqt_scale_velocities", "mdqt_vel_dist_tagged", "mdqt_stress_begin", "mdqt_stress_record",
    "mdqt_stress_download", "mdqt_stress_autocorr", "mdqt_heat_begin", "mdqt_heat_record", "mdqt_heat_download", "mdqt_heat_autocorr",
    "mdqt_modes_begin", "mdqt_modes_record", "mdqt_modes_download", "mdqt_modes_autocorr",
]

_lib = None


def load_library():
    """dlopen libmdqt_b200.so (built in-tree by mdqtplasmasims_b200/build.py). Fails loudly when missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MDQTError("libmdqt_b200.so not built: run `python -m mdqtplasmasims_b200.build` (no CPU fallback exists)")
    L = ctypes.CDLL(LIB_PATH)
    L.mdqt_last_error.restype = ctypes.c_char_p
    L.mdqt_version.restype = ctypes.c_char_p
    L.mdqt_device_ptr.restype = ctypes.c_void_p
    L.mdqt_stream.restype = ctypes.c_void_p
    vp = ctypes.c_void_p
    L.mdqt_params_su.argtypes = [ctypes.POINTER(Params)] + [ctypes.c_double] * 9 + [ctypes.c_int, ctypes.c_int]
    L.mdqt_params_md.argtypes = [ctypes.POINTER(Params), ctypes.c_int, ctypes.c_int] + [ctypes.c_double] * 5 + [ctypes.c_int]
    L.mdqt_create.argtypes = [ctypes.POINTER(Params), ctypes.POINTER(vp)]
    L.mdqt_destroy.argtypes = [vp]
    L.mdqt_sync.argtypes = [vp]
    L.mdqt_upload_state.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int]
    L.mdqt_download_state.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int]
    L.mdqt_upload_forces.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_download_forces.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_set_time.argtypes = [vp, ctypes.c_double, ctypes.c_uint64]
    L.mdqt_get_time.argtypes = [vp, c_double_p, ctypes.POINTER(ctypes.c_uint64)]
    L.mdqt_forces.argtypes = [vp]
    L.mdqt_substeps.argtypes = [vp, ctypes.c_int]
    L.mdqt_md_steps.argtypes = [vp, ctypes.c_int]
    L.mdqt_md_steps_host.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int]
    L.mdqt_epot.argtypes = [vp, c_double_p]
    L.mdqt_diagnostics.argtypes = [vp, ctypes.POINTER(Diag)]
    L.mdqt_vel_dist.argtypes = [vp, c_double_p]
    L.mdqt_populations.argtypes = [vp, c_double_p]
    L.mdqt_vv_step.argtypes = [vp, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_double]
    L.mdqt_qsteps.argtypes = [vp, ctypes.c_int]
    L.mdqt_set_forced_uniforms.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_set_forced_collisions.argtypes = [vp, vp, vp]
    L.mdqt_philox_uniforms.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64, c_double_p]
    L.mdqt_device_ptr.argtypes = [vp, ctypes.c_int]
    L.mdqt_device_ld.argtypes = [vp]
    L.mdqt_stream.argtypes = [vp]
    L.mdqt_mark_wrapped.argtypes = [vp, ctypes.c_int]
    L.mdqt_force_plan.argtypes = [vp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    L.mdqt_enable_timing.argtypes = [vp, ctypes.c_int]
    L.mdqt_kernel_time_ms.argtypes = [vp, ctypes.c_int, c_double_p, ctypes.POINTER(ctypes.c_int)]
    L.mdqt_fp64_peak.argtypes = [vp, c_double_p]
    L.mdqt_params_ts.argtypes = [ctypes.POINTER(Params), ctypes.c_int, ctypes.c_double, ctypes.c_double]
    L.mdqt_leapfrog_step.argtypes = [vp, ctypes.c_double]
    L.mdqt_advance_time.argtypes = [vp, ctypes.c_int]
    L.mdqt_tag_particles.argtypes = [vp, vp, vp]
    L.mdqt_vaf.argtypes = [vp, ctypes.c_int, c_double_p]
    L.mdqt_vsq_autocorr.argtypes = [vp, ctypes.c_int, c_double_p]
    L.mdqt_set_forced_tag_uniforms.argtypes = [vp, vp]
    L.mdqt_pair_correlation.argtypes = [vp, ctypes.c_double, ctypes.c_double, ctypes.c_int, vp, vp]
    L.mdqt_vstore_begin.argtypes = [vp, ctypes.c_int]
    L.mdqt_vstore_record.argtypes = [vp, ctypes.c_int]
    L.mdqt_vstore_upload.argtypes = [vp, vp]
    L.mdqt_autocorrelations.argtypes = [vp, ctypes.c_double, vp, vp, vp, vp]
    L.mdqt_vv_steps.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                ctypes.c_double]
    L.mdqt_set_ion_counts.argtypes = [vp, vp]
    L.mdqt_comm_unique_id.argtypes = [vp]
    L.mdqt_comm_init.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int]
    L.mdqt_comm_destroy.argtypes = [vp]
    L.mdqt_comm_exchange_positions.argtypes = [vp]
    L.mdqt_comm_allreduce.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_populations_rows.argtypes = [vp, vp]
    L.mdqt_download_rows.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int]
    L.mdqt_set_tags.argtypes = [vp, vp]
    L.mdqt_moments_begin.argtypes = [vp, ctypes.c_int]
    L.mdqt_moments_record.argtypes = [vp, ctypes.c_int]
    L.mdqt_moments_download.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_stress_begin.argtypes = [vp, ctypes.c_int]
    L.mdqt_stress_record.argtypes = [vp, ctypes.c_int]
    L.mdqt_stress_download.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_stress_autocorr.argtypes = [vp, ctypes.c_int, vp]
    L.mdqt_heat_begin.argtypes = [vp, ctypes.c_int]
    L.mdqt_heat_record.argtypes = [vp, ctypes.c_int]
    L.mdqt_heat_download.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_heat_autocorr.argtypes = [vp, ctypes.c_int, vp]
    L.mdqt_modes_begin.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int]
    L.mdqt_modes_record.argtypes = [vp, ctypes.c_int]
    L.mdqt_modes_download.argtypes = [vp, vp, ctypes.c_int]
    L.mdqt_modes_autocorr.argtypes = [vp, ctypes.c_int, vp, vp, vp]
    L.mdqt_scale_velocities.argtypes = [vp, ctypes.c_double, ctypes.c_double, ctypes.c_double]
    L.mdqt_vel_dist_tagged.argtypes = [vp, vp]
    L.mdqt_time_forces.argtypes = [vp, ctypes.c_int, c_double_p]
    L.mdqt_set_traj_seeds.argtypes = [vp, vp]
    L.mdqt_diag_partial.argtypes = [vp, vp, vp]
    L.mdqt_vel_dist_partial.argtypes = [vp, vp, vp]
    _lib = L
    return L


def su_params(Ge=0.1, density=2.0, sig0=4.0, Te=19.0, fracOfSig=0.0, detuning=-1.0, detuningDP=1.0, Om=1.0, OmDP=1.0,
              N0=3500, n_ions=None, **overrides):
    """``mdqt_params`` for the SU family from the reference's user inputs (SU:56-74)."""
    p = Params()
    rc = load_library().mdqt_params_su(ctypes.byref(p), Ge, density, sig0, Te, fracOfSig, detuning, detuningDP, Om, OmDP,
                                       N0, N0 if n_ions is None else n_ions)
    if rc:
        raise MDQTError(load_library().mdqt_last_error().decode())
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


def md_params(scheme=SCHEME_NONE, n_ions=4096, kappa=0.5, density=0.4, timeStep=0.005, detuning=-2.5, Om=0.7, quad=0,
              **overrides):
    """``mdqt_params`` for the MD family (MD:66-88; MC408L:79-122)."""
    p = Params()
    rc = load_library().mdqt_params_md(ctypes.byref(p), scheme, n_ions, kappa, density, timeStep, detuning, Om, quad)
    if rc:
        raise MDQTError(load_library().mdqt_last_error().decode())
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


def ts_params(n_ions=1000, detuning=-0.5, Om=0.5, **overrides):
    """``mdqt_params`` of the 3-level test program without plasma (TS:55-58, 91, 390)."""
    p = Params()
    rc = load_library().mdqt_params_ts(ctypes.byref(p), n_ions, detuning, Om)
    if rc:
        raise MDQTError(load_library().mdqt_last_error().decode())
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


def philox_uniforms(seed, traj, n_ions, substep):
    """The u[n_ions][5] the device draws for trajectory ``traj`` at global substep ``substep`` (host replica)."""
    L = load_library()
    u = np.empty((n_ions, 5))
    for i in range(n_ions):
        L.mdqt_philox_uniforms(seed, traj, i, substep, u[i].ctypes.data_as(c_double_p))
    return u


def axis_wavevectors(nmax):
    """The 3 nmax integer vectors (n,0,0), (0,n,0), (0,0,n) for n = 1..nmax, in that order: int32 [3 nmax][3], so that a result over
    them reshaped to [nmax][3] averages over the three axes along its second index."""
    return np.concatenate([n * np.eye(3, dtype=np.int32) for n in range(1, nmax + 1)]).reshape(3 * nmax, 3)


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _chk64(a, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise MDQTError("array has shape %s, expected %s" % (a.shape, shape))
    return a


class Engine:
    """One handle = the reference's global simulation state, resident on one GPU.

    Method names follow the reference: ``forces()``, ``step_qstep(n)`` (n x { step(); qstep(); }), ``md_steps(n)``
    (the main-loop body), ``Epotential()``, ``MDStep()``, ``qstep7(n)``.
    """

    def __init__(self, params):
        self.lib = load_library()
        self.params = params
        h = ctypes.c_void_p()
        rc = self.lib.mdqt_create(ctypes.byref(params), ctypes.byref(h))
        if rc:
            raise MDQTError("mdqt_create failed (%d): %s" % (rc, self.lib.mdqt_last_error().decode()))
        self.h = h
        self.N, self.B, self.S = params.n_ions, params.n_traj, params.scheme
        self._modes_K = 0  # wave vectors of the mode log (modes_begin)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mdqt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise MDQTError("libmdqt_b200 error %d: %s" % (rc, self.lib.mdqt_last_error().decode()))

    def _lead(self):
        return (self.B,) if self.B > 1 else ()

    # ---- state -------------------------------------------------------------------------------------------
    def upload(self, R=None, V=None, psi=None, tPart=None, t=None, substep=None):
        N = self.N
        R = _chk64(R, self._lead() + (3, N))
        V = _chk64(V, self._lead() + (3, N))
        psi = _chk64(psi, self._lead() + (N, self.S, 2)) if psi is not None else None
        tPart = _chk64(tPart, self._lead() + (N,))
        self._ck(self.lib.mdqt_upload_state(self.h, _ptr(R), _ptr(V), _ptr(psi), _ptr(tPart), N))
        if t is not None or substep is not None:
            t0, s0 = self.time()
            self._ck(self.lib.mdqt_set_time(self.h, t0 if t is None else t, s0 if substep is None else substep))

    def download(self, want=("R", "V", "psi", "tPart")):
        N = self.N
        out = {}
        R = np.empty(self._lead() + (3, N)) if "R" in want else None
        V = np.empty(self._lead() + (3, N)) if "V" in want else None
        psi = np.empty(self._lead() + (N, self.S, 2)) if ("psi" in want and self.S) else None
        tp = np.empty(self._lead() + (N,)) if "tPart" in want else None
        self._ck(self.lib.mdqt_download_state(self.h, _ptr(R), _ptr(V), _ptr(psi), _ptr(tp), N))
        for k, v in (("R", R), ("V", V), ("psi", psi), ("tPart", tp)):
            if v is not None:
                out[k] = v
        out["t"], out["substep"] = self.time()
        return out

    def upload_forces(self, F):
        F = _chk64(F, self._lead() + (3, self.N))
        self._ck(self.lib.mdqt_upload_forces(self.h, _ptr(F), self.N))

    def download_forces(self):
        F = np.empty(self._lead() + (3, self.N))
        self._ck(self.lib.mdqt_download_forces(self.h, _ptr(F), self.N))
        return F

    def time(self):
        t = ctypes.c_double()
        s = ctypes.c_uint64()
        self._ck(self.lib.mdqt_get_time(self.h, ctypes.byref(t), ctypes.byref(s)))
        return t.value, s.value

    def sync(self):
        self._ck(self.lib.mdqt_sync(self.h))

    def set_ion_counts(self, counts):
        """Ensemble whose jobs drew different N (SU:299-337): trajectory b holds counts[b] <= n_ions ions."""
        if counts is None:
            self._ck(self.lib.mdqt_set_ion_counts(self.h, None))
            return
        c = np.ascontiguousarray(counts, dtype=np.int32)
        assert c.shape == (self.B,)
        self._ck(self.lib.mdqt_set_ion_counts(self.h, ctypes.c_void_p(c.ctypes.data)))

    def set_traj_seeds(self, seeds):
        """One Philox key per trajectory (the reference seeds every SLURM-array job separately, SU:1219)."""
        if seeds is None:
            self._ck(self.lib.mdqt_set_traj_seeds(self.h, None))
            return
        c = np.ascontiguousarray(seeds, dtype=np.uint64)
        assert c.shape == (self.B,)
        self._ck(self.lib.mdqt_set_traj_seeds(self.h, ctypes.c_void_p(c.ctypes.data)))

    # ---- the reference's hot-path functions -----------------------------------------------------------------
    def forces(self):
        """forces() SU:192-236 / calculateAccelerations() MD:387-448."""
        self._ck(self.lib.mdqt_forces(self.h))

    calculateAccelerations = forces

    def step_qstep(self, nsub=1):
        """nsub x { step(); qstep(); } (SU:1376-1377)."""
        self._ck(self.lib.mdqt_substeps(self.h, nsub))

    def md_steps(self, nsteps=1):
        """nsteps x { forces(); ratio x { step(); qstep(); } } (SU:1369-1378)."""
        self._ck(self.lib.mdqt_md_steps(self.h, nsteps))

    def md_steps_host(self, nsteps, R, V, psi, tPart):
        """End-to-end call on HOST arrays (updated in place): upload, nsteps MD steps, download."""
        for a in (R, V, psi, tPart):
            assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        self._ck(self.lib.mdqt_md_steps_host(self.h, nsteps, _ptr(R), _ptr(V), _ptr(psi), _ptr(tPart), self.N))

    def Epotential(self):
        """Epotential() SU:244-281 (per particle)."""
        e = np.empty(self.B)
        self._ck(self.lib.mdqt_epot(self.h, e.ctypes.data_as(c_double_p)))
        return e if self.B > 1 else float(e[0])

    def diagnostics(self):
        d = (Diag * self.B)()
        self._ck(self.lib.mdqt_diagnostics(self.h, d))
        out = [{k: getattr(x, k) for k, _ in Diag._fields_} for x in d]
        return out if self.B > 1 else out[0]

    def diag_partial(self, vx_mean=None):
        """Partial sums of output()'s observables over this handle's rows: [sum vx, sum (vx-mean)^2/2, sum vy^2/2,
        sum vz^2/2, Epot share] per trajectory (row-decomposed runs; all-reduce over the ranks completes them)."""
        s = np.empty((self.B, 5))
        m = None if vx_mean is None else np.ascontiguousarray(np.broadcast_to(np.asarray(vx_mean, dtype=np.float64), (self.B,)))
        self._ck(self.lib.mdqt_diag_partial(self.h, _ptr(m), _ptr(s)))
        return s if self.B > 1 else s[0]

    def vel_dist_partial(self, vx_mean):
        p = np.empty(self._lead() + (3, 2001))
        m = np.ascontiguousarray(np.broadcast_to(np.asarray(vx_mean, dtype=np.float64), (self.B,)))
        self._ck(self.lib.mdqt_vel_dist_partial(self.h, _ptr(m), _ptr(p)))
        return p

    def vel_dist(self):
        p = np.empty(self._lead() + (3, 2001))
        self._ck(self.lib.mdqt_vel_dist(self.h, p.ctypes.data_as(c_double_p)))
        return p

    def populations(self):
        p = np.empty(self._lead() + (self.N, 3))
        self._ck(self.lib.mdqt_populations(self.h, p.ctypes.data_as(c_double_p)))
        return p

    def MDStep(self, dt=0.005, collisionFreq=0.0, sigma_v=1.0, laser=0, laser_coeff=0.0):
        """MDStep() MD:504-511."""
        self._ck(self.lib.mdqt_vv_step(self.h, dt, collisionFreq, sigma_v, laser, laser_coeff))

    def MDSteps(self, nsteps, dt=0.005, collisionFreq=0.0, sigma_v=1.0, laser=0, laser_coeff=0.0, qsteps=0):
        """nsteps x { qsteps x qstep(); MDStep(); } (MD:1081-1083; MC408L:1227-1232), replayed as one CUDA graph."""
        self._ck(self.lib.mdqt_vv_steps(self.h, nsteps, qsteps, dt, collisionFreq, sigma_v, laser, laser_coeff))

    def qstep7(self, nsub=1):
        """nsub x qstep() of the 7-level pump (MC408L:555-756), velocities frozen, no kick."""
        self._ck(self.lib.mdqt_qsteps(self.h, nsub))

    qstep5 = qstep7  # 5-level 422 nm pump (MC422L:552-727): same call, scheme decides
    qstep3 = qstep7  # 3-level test system (TS:140-293): V_x kicked, tPart tracked

    def step(self, dt=0.002):
        """FZ-family step() (FZ408L:377-390): leap-frog with forces() inside; 2nd-order start while t <= 0."""
        self._ck(self.lib.mdqt_leapfrog_step(self.h, dt))

    def advance_time(self, nsub=1):
        """t += quantumTimestep, nsub times (FZ408L:1066, outside the pump window)."""
        self._ck(self.lib.mdqt_advance_time(self.h, nsub))

    def tagParticles(self):
        """tagParticles() MC408L:1022-1067 / MC422L:992-1036 == measureSpinUps() FZ408L:600-647.
        Returns (tagged int32 [n_traj?][n_ions], count)."""
        tagged = np.zeros(self._lead() + (self.N,), dtype=np.int32)
        cnt = np.zeros(self.B, dtype=np.int32)
        self._ck(self.lib.mdqt_tag_particles(self.h, ctypes.c_void_p(tagged.ctypes.data), ctypes.c_void_p(cnt.ctypes.data)))
        return tagged, (cnt if self.B > 1 else int(cnt[0]))

    measureSpinUps = tagParticles

    def Zfunc(self, c1V):
        """Zfunc() FZ408L:938-961: VAF against the velocities stored when c1V == 0."""
        v = np.empty(self.B)
        self._ck(self.lib.mdqt_vaf(self.h, 1 if c1V == 0 else 0, v.ctypes.data_as(c_double_p)))
        return v if self.B > 1 else float(v[0])

    def ZfuncLongKin(self, c1V):
        """Zfunc() of the Quad program (FZ408Q:942-967): the v_x^2 autocorrelation against the velocities stored when c1V == 0."""
        v = np.empty(self.B)
        self._ck(self.lib.mdqt_vsq_autocorr(self.h, 1 if c1V == 0 else 0, v.ctypes.data_as(c_double_p)))
        return v if self.B > 1 else float(v[0])

    def recordPairPairCorr(self, pairPairStep=0.05, pairPairMax=None):
        """recordPairPairCorr() MD:584-652 without the file: returns (r bins, g(r), raw ordered-pair counts)."""
        rmax = self.params.L / 2 if pairPairMax is None else pairPairMax
        nb = int(rmax / pairPairStep)
        g = np.empty(self._lead() + (nb,))
        cnt = np.zeros(self._lead() + (nb,), dtype=np.uint64)
        self._ck(self.lib.mdqt_pair_correlation(self.h, pairPairStep, rmax, nb, _ptr(g), ctypes.c_void_p(cnt.ctypes.data)))
        return np.arange(nb) * pairPairStep, g, cnt

    def vstore_begin(self, T):
        self._ck(self.lib.mdqt_vstore_begin(self.h, T))
        self._T = T

    def recordVelsForAutocorrelations(self, tS):
        """MD:513-520: vStore[:, :, tS] = V."""
        self._ck(self.lib.mdqt_vstore_record(self.h, tS))

    def vstore_upload(self, v):
        v = _chk64(v, self._lead() + (3, self.N, self._T))
        self._ck(self.lib.mdqt_vstore_upload(self.h, _ptr(v)))

    def autocorrelations(self, Gamma):
        """recordVAF, recordLongViscAutoCorr, recordVCubeAutoCorr, recordVFourthAutoCorr (MD:654-823): [4][T]."""
        out = [np.empty(self._lead() + (self._T,)) for _ in range(4)]
        self._ck(self.lib.mdqt_autocorrelations(self.h, Gamma, *[_ptr(o) for o in out]))
        return out

    # ---- test hooks / plumbing ---------------------------------------------------------------------------------
    def set_forced_uniforms(self, u):
        if u is None:
            self._ck(self.lib.mdqt_set_forced_uniforms(self.h, None, 0))
            return
        u = _chk64(u)
        assert u.ndim == 3 and u.shape[1:] == (self.N, 5)
        self._ck(self.lib.mdqt_set_forced_uniforms(self.h, _ptr(u), u.shape[0]))

    def set_forced_tag_uniforms(self, u):
        if u is None:
            self._ck(self.lib.mdqt_set_forced_tag_uniforms(self.h, None))
            return
        u = _chk64(u, (self.N, 2))
        self._ck(self.lib.mdqt_set_forced_tag_uniforms(self.h, _ptr(u)))

    def set_forced_collisions(self, u, v):
        if u is None:
            self._ck(self.lib.mdqt_set_forced_collisions(self.h, None, None))
            return
        u, v = _chk64(u, (self.N,)), _chk64(v, (self.N, 3))
        self._ck(self.lib.mdqt_set_forced_collisions(self.h, _ptr(u), _ptr(v)))

    def force_plan(self):
        a, b = ctypes.c_int(), ctypes.c_int()
        self._ck(self.lib.mdqt_force_plan(self.h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def device_ptr(self, which):
        return self.lib.mdqt_device_ptr(self.h, which)

    @property
    def ld(self):
        return self.lib.mdqt_device_ld(self.h)

    def mark_wrapped(self, wrapped=True):
        self._ck(self.lib.mdqt_mark_wrapped(self.h, 1 if wrapped else 0))

    def enable_timing(self, on=True):
        self._ck(self.lib.mdqt_enable_timing(self.h, int(on)))  # 1: event pairs on stream launches; 2: stamps inside the graph

    def kernel_time_ms(self, which):
        ms, n = ctypes.c_double(), ctypes.c_int()
        self._ck(self.lib.mdqt_kernel_time_ms(self.h, which, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    # ---- MD-family recorders over the velocities (MD:525-582, 923-1029) ------------------------------------------------
    def set_tags(self, tags):
        t = None if tags is None else np.ascontiguousarray(tags, dtype=np.uint8)
        self._ck(self.lib.mdqt_set_tags(self.h, None if t is None else ctypes.c_void_p(t.ctypes.data)))

    def moments_begin(self, nslots):
        self._ck(self.lib.mdqt_moments_begin(self.h, nslots))

    def moments_record(self, slot):
        self._ck(self.lib.mdqt_moments_record(self.h, slot))

    def moments_download(self, nslots):
        out = np.empty((nslots,) + self._lead() + (23,))
        self._ck(self.lib.mdqt_moments_download(self.h, _ptr(out), nslots))
        return out

    # ---- pressure (stress) tensor recorder ------------------------------------------------------------------------------
    def stress_begin(self, nslots):
        """Allocate and zero a device log of ``nslots`` pressure-tensor records."""
        self._ck(self.lib.mdqt_stress_begin(self.h, nslots))

    def stress_record(self, slot):
        """Record K_ab = sum_i v_a v_b and W_ab = sum_{i<j} d_a d_b f(r) into ``slot`` (no synchronisation; the state is untouched)."""
        self._ck(self.lib.mdqt_stress_record(self.h, slot))

    def stress_download(self, nslots):
        """The first ``nslots`` records: [n_traj?][12][nslots] = K_xx, K_yy, K_zz, K_xy, K_xz, K_yz, W_xx, ..., W_yz."""
        out = np.empty(self._lead() + (12, nslots))
        self._ck(self.lib.mdqt_stress_download(self.h, _ptr(out), nslots))
        return out

    def stress_autocorr(self, nslots):
        """Shear-stress autocorrelation C(t) = 1/(3 (T - t)) sum_{ab = xy, xz, yz} sum_j P_ab(j) P_ab(j + t) of the first ``nslots``
        records (P = K + W): [n_traj?][nslots]."""
        out = np.empty(self._lead() + (nslots,))
        self._ck(self.lib.mdqt_stress_autocorr(self.h, nslots, _ptr(out)))
        return out

    # ---- heat (energy) current recorder -----------------------------------------------------------------------------------
    def heat_begin(self, nslots):
        """Allocate and zero a device log of ``nslots`` heat-current records."""
        self._ck(self.lib.mdqt_heat_begin(self.h, nslots))

    def heat_record(self, slot):
        """Record the heat current and its companions into ``slot`` (no synchronisation; the state is untouched)."""
        self._ck(self.lib.mdqt_heat_record(self.h, slot))

    def heat_download(self, nslots):
        """The first ``nslots`` records: [n_traj?][15][nslots] = J_kin (3), J_pot (3), J_vir (3), P (3), E_kin, E_pot, tr W
        (definitions: include/mdqt.h)."""
        out = np.empty(self._lead() + (15, nslots))
        self._ck(self.lib.mdqt_heat_download(self.h, _ptr(out), nslots))
        return out

    def heat_autocorr(self, nslots):
        """Heat-current autocorrelation C(t) = 1/(3 (T - t)) sum_a sum_j J_q,a(j) J_q,a(j + t) of the first ``nslots`` records, with
        J_q = J_kin + J_pot + J_vir - hbar P and hbar the records' mean enthalpy per ion: [n_traj?][nslots]."""
        out = np.empty(self._lead() + (nslots,))
        self._ck(self.lib.mdqt_heat_autocorr(self.h, nslots, _ptr(out)))
        return out

    # ---- density and current Fourier modes ----------------------------------------------------------------------------------
    def modes_begin(self, nvec, nslots):
        """Allocate and zero a device log of ``nslots`` records of rho_k and j_k for the integer vectors ``nvec`` [K][3]
        (k = 2 pi n / L; 1 <= K <= 1024, n != 0, |n_a| < 2^20)."""
        nv = np.ascontiguousarray(nvec, dtype=np.int32)
        if nv.ndim != 2 or nv.shape[1] != 3:
            raise MDQTError("nvec has shape %s, expected [K][3]" % (nv.shape,))
        self._ck(self.lib.mdqt_modes_begin(self.h, _ptr(nv), nv.shape[0], nslots))
        self._modes_K = nv.shape[0]

    def modes_record(self, slot):
        """Record rho_k and j_k of every vector into ``slot`` (no synchronisation; the state is untouched)."""
        self._ck(self.lib.mdqt_modes_record(self.h, slot))

    def modes_download(self, nslots):
        """The first ``nslots`` records: [n_traj?][K][8][nslots] = Re rho, Im rho, Re j_x, Im j_x, Re j_y, Im j_y, Re j_z, Im j_z
        (definitions: include/mdqt.h)."""
        out = np.empty(self._lead() + (self._modes_K, 8, nslots))
        self._ck(self.lib.mdqt_modes_download(self.h, _ptr(out), nslots))
        return out

    def modes_autocorr(self, nslots):
        """(F, C_L, C_T) of the first ``nslots`` records, each [n_traj?][K][nslots]: the intermediate scattering function and the
        longitudinal and transverse current correlations (definitions: include/mdqt.h); S(k) = F[..., 0]."""
        out = [np.empty(self._lead() + (self._modes_K, nslots)) for _ in range(3)]
        self._ck(self.lib.mdqt_modes_autocorr(self.h, nslots, *(_ptr(o) for o in out)))
        return tuple(out)

    def vel_dist_tagged(self):
        p = np.empty(self._lead() + (4001,))
        self._ck(self.lib.mdqt_vel_dist_tagged(self.h, _ptr(p)))
        return p

    def scale_velocities(self, sx, sy, sz):
        self._ck(self.lib.mdqt_scale_velocities(self.h, sx, sy, sz))

    # ---- row-decomposed runs: NCCL communicator inside the library -------------------------------------------------
    @staticmethod
    def comm_unique_id():
        """128-byte NCCL unique id (rank 0 makes it and hands it to the other ranks)."""
        buf = ctypes.create_string_buffer(128)
        L = load_library()
        if L.mdqt_comm_unique_id(buf):
            raise MDQTError(L.mdqt_last_error().decode())
        return buf.raw

    def comm_init(self, unique_id, rank, world):
        """Collective: every rank calls it with the same id; the handle must own rows [rank N/world, (rank+1) N/world)."""
        self._ck(self.lib.mdqt_comm_init(self.h, ctypes.c_char_p(unique_id), rank, world))

    def comm_exchange_positions(self):
        self._ck(self.lib.mdqt_comm_exchange_positions(self.h))

    def populations_rows(self):
        p = np.empty(self._lead() + (self.params.n_rows or self.N, 3))
        self._ck(self.lib.mdqt_populations_rows(self.h, _ptr(p)))
        return p

    def time_forces(self, reps=20):
        """ms per force-kernel launch: CUDA events around one replayed graph of ``reps`` back-to-back launches."""
        v = ctypes.c_double()
        self._ck(self.lib.mdqt_time_forces(self.h, reps, ctypes.byref(v)))
        return v.value

    def fp64_peak_tflops(self):
        v = ctypes.c_double()
        self._ck(self.lib.mdqt_fp64_peak(self.h, ctypes.byref(v)))
        return v.value
