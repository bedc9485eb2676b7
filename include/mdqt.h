/* include/mdqt.h -- C ABI of libmdqt_b200.so: the B200-native replacement for the per-timestep MDQT hot path
 * of tlangin/MDQTPlasmaSims (Yukawa force evaluation, position/velocity update, per-ion quantum-trajectory step).
 *
 * The reference has NO plugin / FFI API: its seam is a set of `void f(void)` free functions that main() calls on
 * file-scope global arrays (SU = laserCoolingPlusExpansionMDQTSpeedUp.cpp, MD =
 * MonteCarloFollowedByMDAndTempAnisotropy.cpp, MC408L = MonteCarloFollowedByQTTagging408Linear.cpp):
 *
 *     double R[3][N0+1000], V[3][..], F[3][..]; unsigned N;      SU:126-129      -> mdqt_upload_state / mdqt_download_state
 *     cx_mat wvFns[N0+1000]; double tPart[..]; double t;         SU:151-152,114  -> same (psi as double [n][S][2])
 *     void forces(void)                                          SU:192-236      -> mdqt_forces
 *     void step(void); void qstep(void)   (one quantum substep)  SU:418-430, 438-717 -> mdqt_substeps(h, nsub)
 *     main loop: forces() every `ratio` substeps                 SU:1369-1378    -> mdqt_md_steps(h, nsteps)
 *     void Epotential(void)                                      SU:244-281      -> mdqt_epot
 *     output(): <v_x>, E_kin, KDE P(v), S/P/D populations        SU:917-1032     -> mdqt_diagnostics / mdqt_vel_dist / mdqt_populations
 *     void calculateAccelerations(int); void MDStep(int)         MD:387-448, 504-511 -> mdqt_forces / mdqt_vv_step
 *     void qstep(void)  7-level pump, no kick                    MC408L:555-756  -> mdqt_qsteps
 *
 * Plain pointers and sizes only; every call returns 0 on success or a negative MDQT_E* code, and
 * mdqt_last_error() gives the message. The library never calls exit() and has NO CPU fallback: without a CUDA
 * device every compute entry point fails with MDQT_ENODEVICE.
 *
 * Host array layouts are the reference's: R, V, F = double [3][ld] (component-major, ld >= n_ions);
 * psi = double [n_ions][S][2] (re, im) with S = scheme (12, 7, 5 or 3); tPart = double [n_ions].
 * With n_traj > 1 (an ensemble shard batched in one handle) every array gains a leading [n_traj] dimension.
 * A handle is bound to one GPU; calls on one handle are stream-ordered and must not be made concurrently.
 */
#ifndef MDQT_H
#define MDQT_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MDQT_OK 0
#define MDQT_EINVAL (-1)
#define MDQT_ENODEVICE (-2)
#define MDQT_ECUDA (-3)
#define MDQT_ENOMEM (-4)
#define MDQT_ESTATE (-5)

#define MDQT_SCHEME_NONE 0 /* MD only: no wavefunctions (MD family) */
#define MDQT_SCHEME_SR7 7  /* 7-level 408 nm pump, MC408L / MC408Q / FZ408L */
#define MDQT_SCHEME_SR12 12 /* 12-level Sr+ S1/2,P3/2,D5/2 laser cooling, SU / MG */
#define MDQT_SCHEME_CA5 5  /* 5-level 422 nm pump (S1/2, P1/2, D reservoir), MC422L / FZ422L */
#define MDQT_SCHEME_V3 3   /* 3-level J=0 <-> J=1 test system without plasma, laserCoolNoPlasmaThreeState.cpp (TS) */

typedef struct mdqt_handle mdqt_handle;

typedef struct mdqt_params {
  int32_t struct_bytes; /* = sizeof(mdqt_params): ABI check */
  int32_t scheme;       /* MDQT_SCHEME_* */
  int32_t n_ions;       /* N: ions per trajectory (SU:129) */
  int32_t n_traj;       /* trajectories batched in this handle (ensemble shard; SLURM --array replacement). >= 1 */
  int32_t traj0;        /* global index of the first trajectory (the reference's `job`): selects the RNG stream */
  int32_t row0, n_rows; /* large-N row decomposition: this handle owns ions [row0,row0+n_rows); n_rows = 0 -> all */
  int32_t device;       /* CUDA device ordinal */
  int32_t substeps_per_md; /* plasmaToQuantumTimestepRatio (SU:83) */
  int32_t renormalize;  /* reNormalizewvFns (SU:74) */
  int32_t quad;         /* 7-level only: circular-pump coupling mask of MC408Q:596 */
  int32_t plan_n;       /* 0 (recommended): the summation order of the force kernel for a trajectory follows from that
                           trajectory's OWN ion count -- n_ions, or its entry in mdqt_set_ion_counts -- so a job gives the
                           same bits alone (a handle of its size) and inside any batch, and gets the plan that fits its N.
                           > 0: one order for every trajectory, planned for this NOMINAL ion number (the reference's N0);
                           handles created with the same plan_n agree bit for bit whatever else they hold. */
  double L;             /* box length (SU:297, MD:73) */
  double kappa;         /* 1/lDeb = sqrt(3 Ge) (SU:295) or kappa (MD:67) */
  double rcut;          /* L/2 (SU:195, MD:74) */
  double dtq;           /* quantumTimestep (SU:84) */
  double detuning, detuningDP, Om, OmDP; /* SU:70-73 */
  double dR, kRat;      /* decayRatioD5Halves, kRat (SU:146-147) */
  double vKick, vKickDP;/* SU:148-149 */
  double g2E, pv2qv;    /* gamToEinsteinFreq, plasVelToQuantVel (SU:79, 85) */
  double fracOfSig, Te, sig0, density; /* expansion detuning (SU:447) */
  uint64_t seed;        /* Philox key; the reference seeds drand48 from time(NULL)+job (SU:1219) */
} mdqt_params;

typedef struct mdqt_diag {   /* what output() prints to energies.dat (SU:934-955) */
  double t, ekin_x, ekin_y, ekin_z, epot, vx_avg;
} mdqt_diag;

/* Fill `p` with the SU-family derived constants exactly as the reference evaluates them (SU:79-85, 146-149,
 * 295-297) for the user inputs Ge, density, sig0, Te, fracOfSig, detuning, detuningDP, Om, OmDP and N0. */
int mdqt_params_su(mdqt_params* p, double Ge, double density, double sig0, double Te, double fracOfSig,
                   double detuning, double detuningDP, double Om, double OmDP, int N0, int n_ions);
/* MD-family constants (MD:66-74, 88; MC408L:79-122): kappa, Gamma-independent box for n_ions, pump parameters. */
int mdqt_params_md(mdqt_params* p, int scheme, int n_ions, double kappa, double density, double timeStep,
                   double detuning, double Om, int quad);

/* 3-level test program constants (TS:55-58, 91, 390): dt = 0.01/gamma, velocities already in quantum units. */
int mdqt_params_ts(mdqt_params* p, int n_ions, double detuning, double Om);

int mdqt_device_count(void);
const char* mdqt_last_error(void);
const char* mdqt_version(void);

int mdqt_create(const mdqt_params* p, mdqt_handle** out);
int mdqt_destroy(mdqt_handle* h);
int mdqt_sync(mdqt_handle* h);

/* Upload / download the reference's global state. Any pointer may be NULL (that array is skipped).
 * `ld` is the leading dimension of the host R/V/F arrays (the reference's N0+1000, SU:126). */
int mdqt_upload_state(mdqt_handle* h, const double* R, const double* V, const double* psi, const double* tPart, int ld);
int mdqt_download_state(mdqt_handle* h, double* R, double* V, double* psi, double* tPart, int ld);
int mdqt_upload_forces(mdqt_handle* h, const double* F, int ld);
int mdqt_download_forces(mdqt_handle* h, double* F, int ld);
int mdqt_set_time(mdqt_handle* h, double t, uint64_t substep_index); /* global t (SU:114) and RNG substep counter */
int mdqt_get_time(mdqt_handle* h, double* t, uint64_t* substep_index);

/* Ensembles whose jobs drew different ion numbers (every reference job draws N ~ Binomial around N0, SU:299-337): trajectory
 * b of the batch holds n_ions[b] <= mdqt_params.n_ions ions (the handle's capacity; host arrays keep the capacity as their
 * stride, entries beyond n_ions[b] are ignored). Honoured by mdqt_forces, mdqt_substeps, mdqt_md_steps(_host), mdqt_epot,
 * mdqt_diagnostics, mdqt_vel_dist and mdqt_populations; the MD-/FZ-family entry points return MDQT_ESTATE while counts are
 * set. NULL restores "all trajectories hold n_ions". */
int mdqt_set_ion_counts(mdqt_handle* h, const int32_t* n_ions /*[n_traj]*/);
/* One Philox key per trajectory instead of mdqt_params.seed (the reference seeds every job of a SLURM array from
 * time + job, SU:1219): trajectory b then draws exactly what a single-trajectory handle with seed = seeds[b] and
 * traj0 = traj0 + b draws. NULL restores the common seed. */
int mdqt_set_traj_seeds(mdqt_handle* h, const uint64_t* seeds /*[n_traj]*/);

/* forces() (SU:192-236) / calculateAccelerations() (MD:387-448): all-pairs minimum-image Yukawa, r < L/2. */
int mdqt_forces(mdqt_handle* h);
/* nsub x { step(); qstep(); } (SU:1376-1377) with F held fixed, fused per ion. */
int mdqt_substeps(mdqt_handle* h, int nsub);
/* nsteps x { forces(); substeps_per_md x { step(); qstep(); } } -- the body of the main loop (SU:1369-1378). */
int mdqt_md_steps(mdqt_handle* h, int nsteps);
/* Same as mdqt_md_steps but through HOST buffers: upload state, run, download state (the end-to-end call). */
int mdqt_md_steps_host(mdqt_handle* h, int nsteps, double* R, double* V, double* psi, double* tPart, int ld);
/* Epotential() (SU:244-281): sum_{i<j} exp(-kappa r)/r / N. */
int mdqt_epot(mdqt_handle* h, double* epot);
/* output() observables (SU:934-1023). pvel = double [3][2001] (X,Y,Z) on the reference's bins i*0.0025;
 * pops = double [n_ions][3] (S,P,D). For n_traj > 1 results are per trajectory, leading [n_traj]. */
int mdqt_diagnostics(mdqt_handle* h, mdqt_diag* out);
int mdqt_vel_dist(mdqt_handle* h, double* pvel);
int mdqt_populations(mdqt_handle* h, double* pops);

/* Row-decomposed runs (n_rows < n_ions): the observables of output() as partial sums over the handle's own rows, to be
 * completed by an all-reduce (SUM) over the ranks. sums = double [n_traj][5]: sum v_x, sum (v_x - mean)^2/2, sum v_y^2/2,
 * sum v_z^2/2 (none divided by N) and the handle's share of Epotential() (already divided by N). vx_mean = double
 * [n_traj] or NULL (0): call once with NULL, all-reduce sums[0]/N into the mean, call again. pvel as mdqt_vel_dist. */
int mdqt_diag_partial(mdqt_handle* h, const double* vx_mean, double* sums);
int mdqt_vel_dist_partial(mdqt_handle* h, const double* vx_mean, double* pvel);

/* MD family: MDStep() (MD:504-511) = stepPositions, calculateAccelerations, stepVelocities with Andersen
 * collisions (probability dt*collisionFreq, velocities ~ N(0, sigma_v^2)) and the optional laser friction term
 * (laser: 0 none, 1 three-axis MD:494-496, 2 x only MD:491; coefficient = 1.234e-6*beta/sqrt(n)). */
int mdqt_vv_step(mdqt_handle* h, double dt, double collisionFreq, double sigma_v, int laser, double laser_coeff);
/* nsteps x { qsteps x qstep(); MDStep(); } in one call: the MD-family loops (MD:1081-1083, 1107-1165 with qsteps = 0) and the
 * pump stage (MC408L:1227-1232 with qsteps = plasmaToQuantumTimestepRatio). Two or more steps are replayed as one CUDA
 * graph (bitwise the same results as the single calls). */
int mdqt_vv_steps(mdqt_handle* h, int nsteps, int qsteps, double dt, double collisionFreq, double sigma_v, int laser,
                  double laser_coeff);
/* nsub x qstep() without step(): the 7-level (MC408L:555-756, FZ408L:396-598) and 5-level (MC422L:552-727) pump
 * sweeps at frozen velocities without kick, and the 3-level test system (TS:140-293; V_x += kick, tPart tracked). */
int mdqt_qsteps(mdqt_handle* h, int nsub);
/* FZ family: step() (FZ408L:377-390) = step_R(dt/2), step_V(dt) with forces() inside, step_R(dt/2); while t <= 0 the
 * drifts are the 2nd-order start that recomputes forces() (FZ408L:332-340). Does not advance t. */
int mdqt_leapfrog_step(mdqt_handle* h, double dt);
/* FZ family main loop outside the pump window: t += nsub * quantumTimestep by repeated addition (FZ408L:1066). */
int mdqt_advance_time(mdqt_handle* h, int nsub);
/* Projective spin measurement after the pump: tagParticles() (MC408L:1022-1067, MC422L:992-1036) ==
 * measureSpinUps() (FZ408L:600-647, FZ422L:570-611). tagged = int32 [n_traj][n_ions] (may be NULL),
 * n_tagged = int32 [n_traj]. Two uniforms per ion from the Philox stream at the current substep index. */
int mdqt_tag_particles(mdqt_handle* h, int32_t* tagged, int32_t* n_tagged);
/* Zfunc() (FZ408L:938-961): velocity autocorrelation <v_x(t0) v_x(t)>; start != 0 stores v_x(t0) first. vaf[n_traj]. */
int mdqt_vaf(mdqt_handle* h, int start, double* vaf);
/* Zfunc() of the Quad program (randomFrozenStartTag408Quad.cpp:942-967): the v_x^2 autocorrelation "LongKin"
 * sum_j (1/N) (v_x(t0)^2 - a)(v_x(t)^2 - a) with a = <v_x(t)^2>; start != 0 stores v_x(t0) first. out[n_traj]. */
int mdqt_vsq_autocorr(mdqt_handle* h, int start, double* out);

/* Test hook: replace the Philox stream by caller-supplied uniforms u[nsub][n_ions][5] (rand, rand2, randDOrS,
 * randDir, rand3) for the next substeps/qsteps calls (n_traj must be 1). NULL restores Philox. */
int mdqt_set_forced_uniforms(mdqt_handle* h, const double* u, int nsub);
/* recordPairPairCorr() (MD:584-652): g(r) over the N(N-1) ordered minimum-image pairs in bins of `step` up to
 * rmax (the reference: 0.05 and L/2); nbins must equal (int)(rmax/step). g = double [n_traj][nbins] normalised as
 * the reference does (MD:627-635), counts = uint64 [n_traj][nbins] raw pair counts; either may be NULL. */
int mdqt_pair_correlation(mdqt_handle* h, double step, double rmax, int nbins, double* g, uint64_t* counts);
/* Velocity store vStore[3][N][T] (MD:121) on the device: begin(T) allocates and zeroes it, record(tS) is
 * recordVelsForAutocorrelations(tS) (MD:513-520), upload() replaces it from a host array [n_traj][3][n_ions][T]. */
int mdqt_vstore_begin(mdqt_handle* h, int T);
int mdqt_vstore_record(mdqt_handle* h, int tS);
int mdqt_vstore_upload(mdqt_handle* h, const double* v);
/* recordVAF / recordLongViscAutoCorr / recordVCubeAutoCorr / recordVFourthAutoCorr (MD:654-823) over the stored
 * velocities: each output is double [n_traj][T] (NULL = skip); Gamma enters the subtracted constants (MD:710, 785). */
int mdqt_autocorrelations(mdqt_handle* h, double Gamma, double* vaf, double* longvisc, double* vcube, double* vfourth);
/* MD-family recorders that are reductions over the velocities: recordTemperature() (MD:525-546), recordTempForEachAxis()
 * (MD:560-582), recordTaggedParticleMoments() (MD:923-1029, MC408L:1069). tags = uint8 [n_traj][n_ions], bit k = member of tag
 * set k (the reference's taggedOne..taggedFour, MD:809-921; NULL clears). mdqt_moments_begin(nslots) allocates a device log,
 * mdqt_moments_record(slot) writes one record there WITHOUT synchronising (call it every MD step), mdqt_moments_download copies
 * the first nslots records: double [nslots][n_traj][23] = { sum v_x^2, sum v_y^2, sum v_z^2 over all ions; then for each tag set:
 * count, sum v_x, sum v_x^2, sum v_x^3, sum v_x^4 }. The caller divides and subtracts the equilibrium constants as the reference does. */
int mdqt_set_tags(mdqt_handle* h, const uint8_t* tags);
int mdqt_moments_begin(mdqt_handle* h, int nslots);
int mdqt_moments_record(mdqt_handle* h, int slot);
int mdqt_moments_download(mdqt_handle* h, double* out, int nslots);
/* Pressure tensor (virial stress) recorder: K_ab = sum_i v_a v_b, W_ab = sum_{i<j, 0<r<rcut} d_a d_b f(r) with d = r_i - r_j the
 * minimum image and f(r) = (1/r + kappa) exp(-kappa r) / r^2 (so that F_i = sum_j d f), in the units of R, V and mdqt_forces (unit mass),
 * NOT divided by the volume: the virial pressure is (tr K + tr W) / (3 L^3). Ions beyond a trajectory's count (mdqt_set_ion_counts)
 * are left out. Single-GPU handles only (a row-decomposed handle or one with a communicator: MDQT_ESTATE).
 * mdqt_stress_begin(nslots) allocates and zeroes a device log like mdqt_moments_begin; mdqt_stress_record(slot) writes one record
 * there WITHOUT synchronising and leaves R, V, F, the wavefunctions, tPart, t and the step counters untouched; mdqt_stress_download
 * copies the first nslots records as double [n_traj][12][nslots] -- series-major, each of the 12 components a contiguous series:
 * K_xx, K_yy, K_zz, K_xy, K_xz, K_yz, W_xx, W_yy, W_zz, W_xy, W_xz, W_yz. mdqt_stress_autocorr gives the Green-Kubo shear-stress
 * autocorrelation of the first nslots records (nslots <= 6144), acf = double [n_traj][nslots]:
 *   C(t) = 1/(3 (nslots - t)) sum_{ab = xy, xz, yz} sum_{j < nslots - t} P_ab(j) P_ab(j + t),  P = K + W;
 * the shear viscosity is eta = 1/(L^3 T) integral C(t) dt. */
int mdqt_stress_begin(mdqt_handle* h, int nslots);
int mdqt_stress_record(mdqt_handle* h, int slot);
int mdqt_stress_download(mdqt_handle* h, double* out, int nslots);
int mdqt_stress_autocorr(mdqt_handle* h, int nslots, double* acf);
/* Heat (energy) current recorder, in the units of R, V and mdqt_forces (unit mass), with d = r_i - r_j the minimum image, r = |d|,
 * only pairs with 0 < r < rcut, phi(r) = exp(-kappa r) / r and f(r) = (1/r + kappa) exp(-kappa r) / r^2 (so that F_i = sum_j d f).
 * Ions beyond a trajectory's count (mdqt_set_ion_counts) are left out. Per ion phi_i = sum_{j != i} phi(r_ij) and
 * e_i = |v_i|^2 / 2 + phi_i / 2; the energy current (Irving-Kirkwood) is J_E = sum_i e_i v_i + 1/2 sum_i sum_{j != i} d (f d.v_i).
 * One record of a trajectory holds 15 numbers:
 *   0-2   J_kin,a = 1/2 sum_i |v_i|^2 v_ia          9-11  P_a = sum_i v_ia (total momentum)
 *   3-5   J_pot,a = 1/2 sum_i phi_i v_ia            12    E_kin = 1/2 sum_i |v_i|^2
 *   6-8   J_vir,a = 1/2 sum_i sum_{j != i} d_a f (d.v_i)   13    E_pot = 1/2 sum_i phi_i (= N mdqt_epot)
 *                                                   14    tr W = 1/2 sum_i sum_{j != i} f r^2 (= W_xx + W_yy + W_zz of mdqt_stress)
 * Single-GPU handles only (a row-decomposed handle or one with a communicator: MDQT_ESTATE). mdqt_heat_begin(nslots) allocates and
 * zeroes a device log; mdqt_heat_record(slot) writes one record there WITHOUT synchronising and leaves R, V, F, the wavefunctions,
 * tPart, t and the step counters untouched; mdqt_heat_download copies the first nslots records as double [n_traj][15][nslots]
 * (series-major). mdqt_heat_autocorr gives the Green-Kubo heat-current autocorrelation of the first nslots = T records
 * (T <= 6144), acf = double [n_traj][T]:
 *   J_q(j) = J_kin + J_pot + J_vir - hbar P (j),  hbar = 1/(T N_b) sum_{j < T} [E_kin + E_pot + (2 E_kin + tr W)/3](j),
 *   C(t) = 1/(3 (T - t)) sum_{a = x, y, z} sum_{j < T - t} J_q,a(j) J_q,a(j + t);
 * hbar P is the enthalpy current, which a non-zero (conserved) total momentum would otherwise leave as a plateau in C. The thermal
 * conductivity is lambda = 1/(L^3 T^2) integral C(t) dt, T here the temperature. */
int mdqt_heat_begin(mdqt_handle* h, int nslots);
int mdqt_heat_record(mdqt_handle* h, int slot);
int mdqt_heat_download(mdqt_handle* h, double* out, int nslots);
int mdqt_heat_autocorr(mdqt_handle* h, int nslots, double* acf);
/* Velocity distribution of the tagged ions (bit 0 of the tags), x component: pv = double [n_traj][4001] on the bins
 * (j - 2000) * 0.0025, as recordTaggedParticleMoments() / output() of the tagging programs write it (MC408L:1069-1137, FZ408L:835-893). */
int mdqt_vel_dist_tagged(mdqt_handle* h, double* pv);
/* anisotropizeVelocities() (MD:548-558): V_x *= sx, V_y *= sy, V_z *= sz. */
int mdqt_scale_velocities(mdqt_handle* h, double sx, double sy, double sz);
/* Test hook: uniforms u[n_ions][2] for the next mdqt_tag_particles calls (n_traj must be 1). NULL restores Philox. */
int mdqt_set_forced_tag_uniforms(mdqt_handle* h, const double* u);
/* Test hook for the MD-family Andersen thermostat: per-ion collision uniforms u[n_ions] and the velocities
 * v[n_ions][3] assigned on collision, instead of the Philox/Box-Muller draws. NULL restores Philox. */
int mdqt_set_forced_collisions(mdqt_handle* h, const double* u, const double* v);
/* The five Philox uniforms ion `ion` of trajectory `traj` consumes at substep `substep` (host-side replica). */
int mdqt_philox_uniforms(uint64_t seed, uint32_t traj, uint32_t ion, uint64_t substep, double u[5]);

/* Multi-GPU plumbing (row decomposition): raw device pointers so that the caller's NCCL all-gather can write
 * remote rows of R in place. which: 0 = R, 1 = V, 2 = F. Layout on device: double [n_traj][3][mdqt_device_ld].
 * The F pointer is valid until the next mdqt_vv_step(s) call only: MDStep() exchanges the A and oldA buffers (MD:505-506).
 * (Row-decomposed runs no longer need this plumbing: see mdqt_comm_init.) */
void* mdqt_device_ptr(mdqt_handle* h, int which);
int mdqt_device_ld(mdqt_handle* h);
void* mdqt_stream(mdqt_handle* h);

/* Row-decomposed large-N runs inside the library (one process or thread per GPU, NCCL over NVLink). Rank `rank` of `world`
 * creates its handle with row0 = rank * N/world, n_rows = N/world (N divisible by world) and uploads ALL N positions (the
 * other arrays matter for its own rows only). Rank 0 makes the 128-byte id (ncclGetUniqueId) and hands it to the others by
 * any means; all ranks then call mdqt_comm_init concurrently (it is a collective). From then on:
 *   mdqt_md_steps(h, n)      n x { forces over the own rows x all j; substeps of the own rows; all-gather of positions } --
 *                            ONE in-place ncclAllGather of a [3][rows] block of fixed-point positions per rank and MD step, on a
 *                            communication stream, overlapped with the j chunks of the next force call that lie inside the own rows;
 *   mdqt_diagnostics, mdqt_vel_dist   whole-system values on every rank (partial sums + ncclAllReduce);
 *   mdqt_populations_rows, mdqt_download_state   the rank's own rows (remote rows of R are NOT kept current: only their
 *                            fixed-point copy, which is what the pair kernels read);
 *   mdqt_comm_exchange_positions   the bare all-gather, after the caller's own mdqt_substeps.
 * Forces, hence trajectories, are bitwise independent of the number of ranks. */
int mdqt_comm_unique_id(void* id_out /* 128 bytes */);
int mdqt_comm_init(mdqt_handle* h, const void* unique_id /* 128 bytes */, int rank, int world);
int mdqt_comm_destroy(mdqt_handle* h);
int mdqt_comm_exchange_positions(mdqt_handle* h);
int mdqt_comm_allreduce(mdqt_handle* h, double* values, int n); /* sum over the ranks, in place, n <= 6019 */
/* The handle's own rows only, written at their place in host arrays of the usual full layouts (R, V = [3][ld], psi =
 * [n_ions][S][2], tPart = [n_ions]): the ranks of a row-decomposed run assemble one host state without overlap. n_traj = 1. */
int mdqt_download_rows(mdqt_handle* h, double* R, double* V, double* psi, double* tPart, int ld);
/* S/P/D populations of the handle's own rows: pops = double [n_traj][n_rows][3] (row-decomposed handles). */
int mdqt_populations_rows(mdqt_handle* h, double* pops);

/* After an external write into the device R buffer (e.g. the caller's own NCCL all-gather): tells the handle that R
 * changed, so the periodic fixed-point copy read by the pair kernels is refreshed before the next force evaluation. The
 * `wrapped` argument is ignored (the fixed-point minimum image is exact for wrapped and unwrapped coordinates alike). */
int mdqt_mark_wrapped(mdqt_handle* h, int wrapped);
/* The j-range decomposition of the force kernel (a function of n_ions and n_traj only). */
int mdqt_force_plan(mdqt_handle* h, int* nsplit, int* jlen);

/* Per-kernel device timing of the most recent mdqt_md_steps call (ms, averaged per launch).
 *   on = 1: a CUDA-event pair around every launch on the handle's stream (MD steps are then issued as stream launches);
 *   on = 2: %globaltimer stamps written by the kernels themselves INSIDE the replayed CUDA graph (earliest CTA start to
 *           latest CTA end of every launch) -- the durations as they are in production, plus the gaps between the kernels.
 * which: 0 = force kernel, 1 = substep kernel, 2 = gap force -> substep, 3 = gap substep -> next force (2, 3: on = 2 only). */
int mdqt_enable_timing(mdqt_handle* h, int on);
int mdqt_kernel_time_ms(mdqt_handle* h, int which, double* ms_per_launch, int* launches);
/* Average duration of one force-kernel launch (ms), timed with a CUDA-event pair on the handle's stream around ONE replayed
 * graph of `reps` back-to-back launches (after a warm-up replay): no per-launch event or launch-latency overhead. F is
 * overwritten with the same values every launch, so the state is unchanged. */
int mdqt_time_forces(mdqt_handle* h, int reps, double* ms_per_launch);
/* FP64 FMA-chain microbenchmark on the handle's device: returns achieved TFLOP/s (2 flop per DFMA). */
int mdqt_fp64_peak(mdqt_handle* h, double* tflops);

#ifdef __cplusplus
}
#endif
#endif
