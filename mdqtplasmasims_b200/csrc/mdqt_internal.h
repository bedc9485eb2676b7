// mdqt_internal.h -- shared declarations between the kernel translation units and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mdqt {

constexpr int kForceThreads = 128;   // threads per CTA of the pair kernels
constexpr int kExpTable = 1024;      // entries of the 2^(j/T) table used by the fp64 exp (degree-3 polynomial)
constexpr int kVelBins = 2001;       // KDE bins of output() (SU:120-123)
constexpr int kTagBins = 4001;        // velocity bins of the tagged-ion distribution (MC408L:1069, FZ408L:835)
constexpr int kMomentsPerRecord = 23; // 3 axis sums of v^2 + 4 tag sets x {count, sum v_x^1..4}
// pair-once force tiles at small and medium N (k_pairs_items, mdqt_force.cu): ions per block, and resident warps per SM (one CTA)
constexpr int kTileIons = 64;
constexpr int kTileWarps = 12;

struct ForceArgs {
  const double* R;   // [B][3][ld] all positions
  const long long* Rfix;  // [B][3][ld] the same positions in periodic fixed point (mdqt_fixed.cuh)
  // F: [B][3][ld] result. The heat-current pair pass (kModeHeat) writes no forces and reads the velocities V [B][3][ld] in the same
  // slot instead: a field of its own would move the kernels' second parameter and change the code of every other pair kernel
  union { double* F; const double* V; };
  double* Fpart;     // [nsplit][B][3][ld] partial sums when nsplit > 1
  unsigned* counters;// [B][itiles] arrival counters (self-resetting)
  int N, ld, B;
  int row0, nrows;   // rows owned by this handle
  int nsplit, jlen;  // j-range decomposition (depends on N and B only -> rank-count independent sums)
  // CTA-tile kernel launched over a SUBSET of the j chunks (row-decomposed runs overlap the position all-gather with the
  // chunks that need local positions only): chunk = blockIdx.y + js0, and chunks >= js_skip0 are shifted by js_skipn.
  // The partial-sum / arrival-counter protocol still counts all nsplit chunks, across the launches.
  int js0, js_skip0, js_skipn, js_count;  // js_count = chunks in this launch (0: all nsplit)
  int ipt;           // ion rows per thread (1 or 2)
  int jsub;          // intra-CTA split of each j tile over thread groups (1, 2, 4; 4 or 8 with 32-row groups)
  int rg;            // ion rows per thread group: 128 (default) or 32 (small systems)
  // device clock {t, substep index}: inside a replayed CUDA graph kernel arguments are frozen, so the simulation time lives
  // in device memory; the force kernel of MD step k >= 1 advances it by the substeps of step k-1 (clock_advance of them,
  // t by the reference's repeated addition, SU:716) before the substep kernel of step k reads it. Null outside graphs.
  double* clock; int clock_advance; double clock_dtq;
  int half_l;        // rcut == L/2 exactly (every reference program): the cut-off is a power of two in fixed-point units
  double L, halfL, invL, invL_lo, kappa, rc2;  // 1/L = invL + invL_lo (double-double)
  double inv_u, rc2_u;  // fixed-point unit u = L/2^64: 1/u, and the squared cut-off in units u^2
  // k_pairs_items (small and medium systems, any batch size): the persistent grid of the pair-once force tiles and of the diagnostics'
  // gather over (trajectory, 32-row group, j chunk) items. items = 1 selects it; gcap = row groups per trajectory (at capacity)
  int items, gcap;
  const int* jl;                          // gather: [B] chunk length of every trajectory, or null (all jlen, which plan_force sets)
  int pdl;                                // launch with programmatic stream serialisation (pdl_mode)
  unsigned long long mg_chunk, mg_gcap, mg_gcap2;  // ceil(2^40 / nsplit), ceil(2^40 / groups of 32 rows), ... of 64 rows: item index -> (b, g, chunk) without division
  const int* nb;     // [B] ions per trajectory (ensembles whose jobs drew different N, SU:299-337) or null: all N
  // the force tiles (b, I, J) the handle runs, packed b << 16 | I << 8 | J (mdqt_capi.cu, build_tiles)
  const unsigned* ilist; int icount;
  unsigned long long* stamp;  // {min start, max end} of this launch in %globaltimer ns (in-graph kernel timing) or null
};

struct QTArgs {
  double* R; double* V; const double* F;  // [B][3][ld]
  long long* Rfix;                        // [B][3][ld] fixed-point copy of R, refreshed on exit
  double invL, invL_lo;
  double* psi;                            // [B][2*S][ld] component-major: (2*k+{0,1})*ld + i
  double* tPart;                          // [B][ld]
  const double* forced_u;                 // [nsub][N][5] or null
  int N, ld, B, row0, nrows, traj0;
  int nsub;
  int scheme, S;                          // level scheme (12, 7, 5, 3) and its number of states (psi stride)
  int do_step;                            // 1: step() before every qstep(), global t advanced (SU); 0: qstep only
  int do_kick;                            // 1: V_x += optical-force / recoil kick (SU:705, TS:283); 0: frozen V (MC408L:754)
  int do_tpart;                           // 1: tPart tracked (+= dtq, reset on a jump; SU:482, TS:155)
  int renorm, quad;
  int lanes;                              // lanes per ion of the 12-level kernel: 0 = by (N, B), 2 or 4 = pinned
  int pdl;                                // launch with programmatic stream serialisation (pdl_mode)
  double t0; uint64_t substep0; uint64_t seed;
  const int* nb;                          // [B] ions per trajectory or null (all N)
  const double* fpart; double* Fw;        // item-kernel partials [chunk][B][3][ld] to add up (then written to Fw), or null: F is complete
  int fp_jlen;                            // chunk length of those partials ...
  const int* jl;                          // ... or [B], one per trajectory, or null (the force tiles: one length for all)
  const uint64_t* seeds;                  // [B] Philox key per trajectory or null (all `seed`)
  unsigned long long* stamp;              // {min start, max end} of this launch in %globaltimer ns, or null
  const double* clock;                    // {t, substep index (as uint64 bits)} in device memory: overrides t0/substep0 when non-null
  double L, dtq;
  double detuning, detuningDP, Om, OmDP, dR, kRat, vKick, vKickDP, g2E, pv2qv;
  double fracOfSig, Te, sig0, density;
};

struct VVArgs {
  double* R; double* V; const double* A; const double* oldA;  // [B][3][ld]
  long long* Rfix; double invL, invL_lo;
  int N, ld, B, row0, nrows, traj0;
  double L, dt, collisionFreq, sigma_v, laser_coeff;
  int laser;
  uint64_t step; uint64_t seed;
  const double* forced_u;   // [N] collision uniforms or null
  const double* forced_n;   // [N][3] velocities assigned on collision or null
  // device clock {t, substep index, MDStep index} for replayed CUDA graphs (null outside): the position kernel -- which runs
  // after the pump sweeps and the velocity kernel of the previous step and before any reader of the new values -- adds
  // adv_sub to the substep index and adv_vv to the MDStep index; the velocity kernel reads the MDStep index from it
  double* clock; int adv_sub, adv_vv;
};

// Programmatic dependent launch (sm_90+): the hot kernels of an MD step call griddepcontrol.launch_dependents at
// their start and griddepcontrol.wait before touching data of their predecessor, so the next kernel's launch latency
// and prologue overlap the current kernel's tail. `pdl` = launch with the programmatic-serialization attribute.
int pdl_mode();  // MDQT_PDL: 1 = always, 0 = never, unset = -1: where the plan says the kernels' warps finish together (mdqt_capi.cu)
template <typename... KArgs, typename A0, typename A1>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t s, bool pdl, A0 a0, A1 a1) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute at[1];
  int n = 0;
  if (pdl) { at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[n].val.programmaticStreamSerializationAllowed = 1; n++; }
  cfg.attrs = at; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, a0, a1);
}
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// in-graph kernel timing: every CTA (or warp) folds its start / end time into the launch's {min start, max end} slot
__device__ __forceinline__ void stamp_time(unsigned long long* stamp, int end) {
  if (!stamp) return;
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  if (end) atomicMax(stamp + 1, t); else atomicMin(stamp, t);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

void launch_forces(const ForceArgs& a, cudaStream_t s, bool finalize = true);
// the item kernel with more than one chunk leaves one partial sum per chunk in Fpart[chunk][B][3][ld] instead of F
inline bool forces_are_partial(const ForceArgs& a) { return a.items && a.nsplit > 1; }
#ifdef __CUDACC__
// sum of `nch` partials src[0], src[stride], ... in ascending order, fetched as batches of 12 independent L2 loads
template <int BATCH = 12>
__device__ __forceinline__ double sum_partials(const double* __restrict__ src, size_t stride, int nch) {
  double sum = 0.0;
  for (int s0 = 0; s0 < nch; s0 += BATCH) {
    double v[BATCH];
#pragma unroll
    for (int q = 0; q < BATCH; q++) v[q] = (s0 + q < nch) ? __ldcg(src + (size_t)(s0 + q) * stride) : 0.0;
#pragma unroll
    for (int q = 0; q < BATCH; q++) sum += v[q];  // + 0.0 for absent chunks: exact
  }
  return sum;
}
#endif
// Rfix[k] = to_fixed(R[k]) for all B*3*ld entries (after an upload or an external write into R)
void launch_to_fixed(const double* R, long long* Rfix, size_t n, double invL, double invL_lo, cudaStream_t s);
void launch_epot(const ForceArgs& a, double* block_partials, double* result, cudaStream_t s);  // result[B]
int epot_partials_needed(const ForceArgs& a);
// pressure tensor record (mdqt_force.cu): the pair pass in stress mode + K from V; out[b][12][nslots] at column `slot`
constexpr int kStressPerRecord = 12;  // K_xx K_yy K_zz K_xy K_xz K_yz, W_xx W_yy W_zz W_xy W_xz W_yz
void launch_stress(const ForceArgs& a, double* partials, const double* V, double* out, int nslots, int slot, cudaStream_t s);
int stress_partials_needed(const ForceArgs& a);
// shear-stress autocorrelation (mdqt_diag.cu): acf[b][t] = 1/(3 (T - t)) sum_{ab in xy, xz, yz} sum_{j < T - t} P_ab(j) P_ab(j + t)
// over the first T records of the stress log [B][12][nslots]; series = [B][3][T] and partials = [B][1][4][T] scratch, out = [B][4][T]
int stress_autocorr_max_T();
void launch_stress_autocorr(const double* log, int nslots, int B, int T, double* series, double* partials, double* out, cudaStream_t s);
// heat current record (mdqt_force.cu): the pair pass in heat mode (it reads V) + the kinetic sums; out[b][15][nslots] at column `slot`
constexpr int kHeatPerRecord = 15;  // J_kin (3), J_pot (3), J_vir (3), P (3), E_kin, E_pot, tr W
void launch_heat(const ForceArgs& a, double* partials, const double* V, double* out, int nslots, int slot, cudaStream_t s);
int heat_partials_needed(const ForceArgs& a);
// heat-current autocorrelation (mdqt_diag.cu): acf[b][t] = 1/(3 (T - t)) sum_a sum_{j < T - t} J_q,a(j) J_q,a(j + t) over the first T
// records of the heat log [B][15][nslots], J_q = J_kin + J_pot + J_vir - hbar P with hbar the mean enthalpy per ion of the T records;
// nb = per-trajectory ion counts or null (all N); series = [B][3][T] and partials = [B][1][4][T] scratch, out = [B][4][T]
void launch_heat_autocorr(const double* log, int nslots, int B, int T, int N, const int* nb, double* series, double* partials, double* out,
                          cudaStream_t s);
// density and current Fourier modes (mdqt_diag.cu): rho_k, j_k of the K vectors nvec [ceil(K / kModesTile) * kModesTile][3] (the tail
// zero vectors) from the fixed-point positions; out[b][q][8][nslots] at column `slot`; nb = per-trajectory ion counts or null (all N)
constexpr int kModesPerRecord = 8;  // Re rho, Im rho, Re j_x, Im j_x, Re j_y, Im j_y, Re j_z, Im j_z
constexpr int kModesTile = 4;       // vectors per CTA of the record kernel
constexpr int kModesMaxK = 1024;
void launch_modes_record(const long long* Rfix, const double* V, int N, int ld, int B, const int* nb, const int* nvec, int K, double* out,
                         int nslots, int slot, cudaStream_t s);
// mode correlations over the first T records of the mode log [B][K][8][nslots]: out[0] = F, out[1] = C_L, out[2] = C_T, each [B][K][T]
// or null (skipped); series = [B K][10][T] and partials = [B K][4][T] scratch
void launch_modes_autocorr(const double* log, int nslots, int B, int K, int T, int N, const int* nb, const int* nvec, double* series,
                           double* partials, double* const out[3], cudaStream_t s);
struct QTConsts;
void launch_substeps(const QTArgs& a, const QTConsts& C, int scheme, cudaStream_t s);
void launch_vv_positions(const VVArgs& a, cudaStream_t s);
void launch_vv_velocities(const VVArgs& a, cudaStream_t s);
// diag_out[B][8]: vx_avg, ekin_x, ekin_y, ekin_z; pvel[B][3][2001]; pops[B][N][3]; nb = per-trajectory ion counts or null
void launch_diag(const double* V, int N, int ld, int B, const int* nb, double* diag_out, cudaStream_t s);
void launch_vel_dist(const double* V, const double* diag_out, int N, int ld, int B, const int* nb, double* pvel, cudaStream_t s);
void launch_diag_partial(const double* V, int row0, int nrows, int ld, int B, const double* mean, double* out, cudaStream_t s);
void launch_vel_dist_rows(const double* V, const double* diag, int row0, int nrows, int ld, int B, double* pvel, cudaStream_t s);
// recorders over the velocities (mdqt_diag.cu): one 23-entry record per trajectory; V_c *= scale_c
void launch_moments(const double* V, const unsigned char* tags, int N, int ld, int B, double* out, cudaStream_t s);
void launch_vel_dist_tagged(const double* V, const unsigned char* tags, int N, int ld, int B, double* pv, cudaStream_t s);
void launch_scale_velocities(double* V, int N, int ld, int B, double sx, double sy, double sz, cudaStream_t s);
void launch_populations(const double* psi, int S, int N, int ld, int B, double* pops, cudaStream_t s);
// projective spin measurement after the pump (tagParticles MC408L:1022-1067 / MC422L:992-1036; measureSpinUps
// FZ408L:600-647): tagged[B][N] (0/1), count[B]; u = forced uniforms [N][2] or null (Philox call 6)
void launch_tag(const double* psi, int S, int N, int ld, int B, int traj0, uint64_t seed, uint64_t substep,
                const double* forced_u, int* tagged, int* count, cudaStream_t s);
// FZ-family leap-frog pieces (FZ408L:317-369): R += DT*V [+ DT^2*F when first], single wrap; V += DT*F
struct LFArgs {
  double* R; double* V; const double* F; long long* Rfix;
  double invL, invL_lo, L, DT;
  int N, ld, B, row0, nrows, first, kick, drift;  // kick: V += DTV*F first; drift: R += DT*V (2nd-order start if first)
  double DTV;
};
void launch_lf(const LFArgs& a, cudaStream_t s);
// Zfunc (FZ408L:938-961): vaf[B] = 1/N sum_j Vhold_x[j] V_x[j]
void launch_vaf(const double* V, const double* Vhold, int N, int ld, int B, double* out, cudaStream_t s, int squares = 0);
void launch_transpose_psi_in(const double* psi_aos, double* psi_soa, int S, int N, int ld, int B, cudaStream_t s);
void launch_transpose_psi_out(const double* psi_soa, double* psi_aos, int S, int N, int ld, int B, cudaStream_t s);
// recordPairPairCorr (MD:584-625): counts[B][nbins] of ordered pairs per distance bin (nbins <= gr_max_bins())
int gr_max_bins();
void launch_gr(const double* R, int N, int ld, int B, double L, double step, int nbins, unsigned long long* counts, cudaStream_t s);
// vStore (MD:121, 513-520) and the four power autocorrelations (MD:654-823); T*8 bytes of dynamic shared memory (T <= 5000)
void launch_vstore_record(const double* V, double* vstore, int N, int ld, int B, int T, int tS, cudaStream_t s);
int autocorr_chunks(int nseries);
void launch_autocorr(const double* vstore, int N, int B, int T, double sub2, double sub4, double* partials, double* out, cudaStream_t s);
double run_fp64_peak(cudaStream_t s);
void upload_exp_table();

}  // namespace mdqt
