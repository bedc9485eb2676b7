// mdqt_diag.cu -- K4: the observables of output() (reference laserCoolingPlusExpansionMDQTSpeedUp.cpp:917-1032)
// computed on the device, and the AoS <-> SoA wavefunction marshalling used at the C-ABI boundary.
//   <v_x>, E_kin,x (about <v_x>), E_kin,y, E_kin,z            SU:934-947
//   symmetrised Gaussian KDE of the velocity distribution      SU:958-979  (2001 bins of 0.0025, width 0.002)
//   S/P/D populations per ion                                  SU:1016-1023
// All reductions run in a fixed order (thread-strided partial sums + tree), so results are reproducible.
#include "mdqt_internal.h"
#include <math.h>

namespace mdqt {

__device__ __forceinline__ double block_sum_1024(double v, double* sred) {
  const int tid = threadIdx.x;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((tid & 31) == 0) sred[tid >> 5] = v;
  __syncthreads();
  double tot = 0.0;
  if (tid < 32) {
    tot = (tid < (int)(blockDim.x >> 5)) ? sred[tid] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_down_sync(0xffffffffu, tot, o);
  }
  __syncthreads();
  if (tid == 0) sred[0] = tot;
  __syncthreads();
  return sred[0];
}

// one CTA per trajectory; out[b][0..3] = vx_avg, ekin_x, ekin_y, ekin_z
__global__ void __launch_bounds__(1024) k_diag(const double* __restrict__ V, int Ncap, int ld, const int* __restrict__ nb,
                                               double* __restrict__ out) {
  __shared__ double sred[32];
  const int b = blockIdx.x;
  const int N = nb ? nb[b] : Ncap;
  const double* vx = V + (size_t)b * 3 * ld;
  const double* vy = vx + ld;
  const double* vz = vy + ld;
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += vx[i];
  const double avg = block_sum_1024(s, sred) / (double)N;
  double ex = 0.0, ey = 0.0, ez = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    double d = vx[i] - avg;
    ex += 0.5 * (d * d); ey += 0.5 * (vy[i] * vy[i]); ez += 0.5 * (vz[i] * vz[i]);
  }
  ex = block_sum_1024(ex, sred);
  ey = block_sum_1024(ey, sred);
  ez = block_sum_1024(ez, sred);
  if (threadIdx.x == 0) {
    out[b * 8 + 0] = avg; out[b * 8 + 1] = ex / (double)N; out[b * 8 + 2] = ey / (double)N; out[b * 8 + 3] = ez / (double)N;
  }
}

void launch_diag(const double* V, int N, int ld, int B, const int* nb, double* diag_out, cudaStream_t s) {
  k_diag<<<B, 1024, 0, s>>>(V, N, ld, nb, diag_out);
}

// Row-decomposed runs (SURVEY 8(e)): every rank owns the velocities of its rows only, so output() needs partial sums that
// an all-reduce completes. out[b][0..3] = sum vx, sum (vx - mean)^2/2, sum vy^2/2, sum vz^2/2 over rows [row0,row0+nrows),
// NOT normalised; mean[b] comes from the caller (the all-reduced sum vx / N of a first call with mean = 0).
__global__ void __launch_bounds__(1024) k_diag_partial(const double* __restrict__ V, int row0, int nrows, int ld,
                                                       const double* __restrict__ mean, double* __restrict__ out) {
  __shared__ double sred[32];
  const int b = blockIdx.x;
  const double* vx = V + (size_t)b * 3 * ld;
  const double* vy = vx + ld;
  const double* vz = vy + ld;
  const double avg = mean ? mean[b] : 0.0;
  double s = 0.0, ex = 0.0, ey = 0.0, ez = 0.0;
  for (int i = row0 + threadIdx.x; i < row0 + nrows; i += blockDim.x) {
    const double d = vx[i] - avg;
    s += vx[i]; ex += 0.5 * (d * d); ey += 0.5 * (vy[i] * vy[i]); ez += 0.5 * (vz[i] * vz[i]);
  }
  s = block_sum_1024(s, sred); ex = block_sum_1024(ex, sred); ey = block_sum_1024(ey, sred); ez = block_sum_1024(ez, sred);
  if (threadIdx.x == 0) { out[b * 8 + 0] = s; out[b * 8 + 1] = ex; out[b * 8 + 2] = ey; out[b * 8 + 3] = ez; }
}
void launch_diag_partial(const double* V, int row0, int nrows, int ld, int B, const double* mean, double* out, cudaStream_t s) {
  k_diag_partial<<<B, 1024, 0, s>>>(V, row0, nrows, ld, mean, out);
}

// grid: (ceil(2001/8), 3, B); 256 threads = 8 bins x 32 lanes; lanes stride over ions [row0, row0 + nrows)
__global__ void __launch_bounds__(256) k_vel_dist(const double* __restrict__ V, const double* __restrict__ diag, int Ncap, int ld,
                                                  double* __restrict__ pvel, int row0, const int* __restrict__ nb) {
  const int b = blockIdx.z, c = blockIdx.y;
  const int N = nb ? nb[b] : Ncap;
  const int bin = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const double* v = V + ((size_t)b * 3 + c) * ld + row0;
  const double avg = (c == 0) ? diag[b * 8] : 0.0;
  const double V2 = 1. / (2. * 0.002 * 0.002);
  const double vb = (double)bin * 0.0025;
  double s = 0.0;
  if (bin < kVelBins)
    for (int i = lane; i < N; i += 32) {
      double d = v[i] - avg;
      double a = vb - d, e = vb + d;
      s += exp(-V2 * a * a) + exp(-V2 * e * e);
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0 && bin < kVelBins) pvel[((size_t)b * 3 + c) * kVelBins + bin] = s / (6.0 * sqrt(2 * M_PI * 0.002 * 0.002));
}

void launch_vel_dist(const double* V, const double* diag_out, int N, int ld, int B, const int* nb, double* pvel, cudaStream_t s) {
  dim3 grid((kVelBins + 7) / 8, 3, B);
  k_vel_dist<<<grid, 256, 0, s>>>(V, diag_out, N, ld, pvel, 0, nb);
}
// the same KDE restricted to rows [row0,row0+nrows) about an externally supplied <v_x> (diag[b*8]): additive over ranks
void launch_vel_dist_rows(const double* V, const double* diag, int row0, int nrows, int ld, int B, double* pvel, cudaStream_t s) {
  dim3 grid((kVelBins + 7) / 8, 3, B);
  k_vel_dist<<<grid, 256, 0, s>>>(V, diag, nrows, ld, pvel, row0, nullptr);
}

// Zfunc() (FZ408L:938-961): out[b] = sum_j (1/N) Vhold_x[j] V_x[j], fixed-order block reduction; one CTA per trajectory
__global__ void __launch_bounds__(1024) k_vaf(const double* __restrict__ V, const double* __restrict__ Vhold, int N, int ld,
                                              double* __restrict__ out) {
  __shared__ double sred[32];
  const int b = blockIdx.x;
  const double* vx = V + (size_t)b * 3 * ld;
  const double* v0 = Vhold + (size_t)b * ld;
  const double invN = 1 / ((double)N);
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += invN * (v0[i] * vx[i]);
  s = block_sum_1024(s, sred);
  if (threadIdx.x == 0) out[b] = s;
}
// Zfunc() of the Quad program (FZ408Q:942-967): the v_x^2 ("longitudinal stress") autocorrelation
// out[b] = sum_j (1/N) (Vhold_x[j]^2 - a) (V_x[j]^2 - a), a = <V_x^2> NOW (FZ408Q:947-952); two fixed-order block reductions
__global__ void __launch_bounds__(1024) k_vsq_autocorr(const double* __restrict__ V, const double* __restrict__ Vhold, int N, int ld,
                                                       double* __restrict__ out) {
  __shared__ double sred[32];
  __shared__ double savg;
  const int b = blockIdx.x;
  const double* vx = V + (size_t)b * 3 * ld;
  const double* v0 = Vhold + (size_t)b * ld;
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += vx[i] * vx[i];
  s = block_sum_1024(s, sred);
  if (threadIdx.x == 0) savg = s / N;
  __syncthreads();
  const double a = savg, invN = 1 / ((double)N);
  s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += invN * (v0[i] * v0[i] - a) * (vx[i] * vx[i] - a);
  s = block_sum_1024(s, sred);
  if (threadIdx.x == 0) out[b] = s;
}
void launch_vaf(const double* V, const double* Vhold, int N, int ld, int B, double* out, cudaStream_t s, int squares) {
  if (squares) k_vsq_autocorr<<<B, 1024, 0, s>>>(V, Vhold, N, ld, out);
  else k_vaf<<<B, 1024, 0, s>>>(V, Vhold, N, ld, out);
}

// ------------------------------------------------------------------------------------------------------------
// recordPairPairCorr() (MD:584-625): histogram of the N(N-1) ordered minimum-image distances in bins of `step`.
// A diagnostic called every 100 MD steps, so it is written for IDENTICAL bins rather than speed: plain fp64 with the
// reference's own operations and roundings (round(), one rounding per product/sum, sqrt, division). Counts are
// integers -> order-independent. grid (i tiles of 256, j splits, B).
// ------------------------------------------------------------------------------------------------------------
constexpr int kGrMaxBins = 2048;
__global__ void __launch_bounds__(256) k_gr(const double* __restrict__ R, int N, int ld, double L, double step, int nbins,
                                            int jlen, unsigned long long* __restrict__ counts) {
  __shared__ double sx[256], sy[256], sz[256];
  __shared__ unsigned hist[kGrMaxBins];
  const int b = blockIdx.z;
  const double* X = R + (size_t)b * 3 * ld;
  const double* Y = X + ld;
  const double* Z = Y + ld;
  for (int k = threadIdx.x; k < nbins; k += 256) hist[k] = 0;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const bool live = i < N;
  const double xi = live ? X[i] : 0.0, yi = live ? Y[i] : 0.0, zi = live ? Z[i] : 0.0;
  const int jbeg = blockIdx.y * jlen, jend = min(N, jbeg + jlen);
  for (int jc = jbeg; jc < jend; jc += 256) {
    __syncthreads();
    const int j = jc + threadIdx.x;
    if (j < jend) { sx[threadIdx.x] = X[j]; sy[threadIdx.x] = Y[j]; sz[threadIdx.x] = Z[j]; }
    __syncthreads();
    const int cnt = min(256, jend - jc);
    if (live)
      for (int k = 0; k < cnt; k++) {
        if (jc + k == i) continue;                                    // MD:597
        double dx = xi - sx[k], dy = yi - sy[k], dz = zi - sz[k];
        dx = __dadd_rn(dx, -__dmul_rn(L, round(__ddiv_rn(dx, L))));   // MD:608-610
        dy = __dadd_rn(dy, -__dmul_rn(L, round(__ddiv_rn(dy, L))));
        dz = __dadd_rn(dz, -__dmul_rn(L, round(__ddiv_rn(dz, L))));
        const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
        const int bin = (int)__ddiv_rn(__dsqrt_rn(d2), step);         // MD:613-615
        if (bin < nbins) atomicAdd(&hist[bin], 1u);
      }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < nbins; k += 256)
    if (hist[k]) atomicAdd(&counts[(size_t)b * nbins + k], (unsigned long long)hist[k]);
}
int gr_max_bins() { return kGrMaxBins; }
void launch_gr(const double* R, int N, int ld, int B, double L, double step, int nbins, unsigned long long* counts, cudaStream_t s) {
  cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * (size_t)B * nbins, s);
  const int tiles = (N + 255) / 256;
  int nsplit = (148 * 4 + tiles * B - 1) / (tiles * B);  // enough CTAs to fill the chip at small N
  nsplit = max(1, min(nsplit, (N + 255) / 256));
  const int jlen = ((N + nsplit - 1) / nsplit + 255) & ~255;
  dim3 grid(tiles, (N + jlen - 1) / jlen, B);
  k_gr<<<grid, 256, 0, s>>>(R, N, ld, L, step, nbins, jlen, counts);
}

// ------------------------------------------------------------------------------------------------------------
// Velocity store and the four power autocorrelations recordVAF / recordLongViscAutoCorr / recordVCubeAutoCorr /
// recordVFourthAutoCorr (MD:654-823): C_p[t] = 1/(N (T-t)) sum_i sum_c sum_{j<T-t} (v(j) v(j+t))^p, p = 1..4 (the
// reference writes the p-th powers out as products of pow(.,2) factors), minus 3/Gamma^2 (p = 2) and 27/Gamma^4 (p = 4).
// vstore = [B][3][N][T] like the reference's vStore[3][N][T]. One CTA = (chunk of series, tile of 256 lags): the series
// is staged in shared memory, thread <-> lag, s[j] is a broadcast read and s[j+t] a conflict-free one. Chunk partials
// are summed in ascending chunk order by a second kernel -> reproducible.
// ------------------------------------------------------------------------------------------------------------
__global__ void k_vstore_record(const double* __restrict__ V, double* __restrict__ vstore, int N, int ld, int T, int tS) {
  const int b = blockIdx.y;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= 3LL * N) return;
  const int c = (int)(g / N), i = (int)(g % N);
  vstore[(((size_t)b * 3 + c) * N + i) * T + tS] = V[((size_t)b * 3 + c) * ld + i];  // MD:513-520
}
void launch_vstore_record(const double* V, double* vstore, int N, int ld, int B, int T, int tS, cudaStream_t s) {
  dim3 grid((unsigned)((3LL * N + 255) / 256), B);
  k_vstore_record<<<grid, 256, 0, s>>>(V, vstore, N, ld, T, tS);
}

constexpr int kAcSeries = 32;  // series per CTA chunk
__global__ void __launch_bounds__(256) k_autocorr(const double* __restrict__ vstore, int nseries, int T,
                                                  double* __restrict__ partials) {
  extern __shared__ double sser[];  // [T]
  const int b = blockIdx.z;
  const int t = blockIdx.y * 256 + threadIdx.x;  // this thread's lag
  const int s0 = blockIdx.x * kAcSeries, s1 = min(nseries, s0 + kAcSeries);
  const double* base = vstore + (size_t)b * nseries * T;
  double a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0;
  for (int s = s0; s < s1; s++) {
    __syncthreads();
    for (int k = threadIdx.x; k < T; k += 256) sser[k] = base[(size_t)s * T + k];
    __syncthreads();
    if (t < T) {
      const int n = T - t;
#pragma unroll 4
      for (int j = 0; j < n; j++) {
        const double p = sser[j] * sser[j + t];
        const double p2 = p * p;
        a1 += p; a2 += p2; a3 = fma(p2, p, a3); a4 = fma(p2, p2, a4);
      }
    }
  }
  if (t < T) {
    double* o = partials + (((size_t)b * gridDim.x + blockIdx.x) * 4) * T + t;
    o[0] = a1; o[T] = a2; o[2 * (size_t)T] = a3; o[3 * (size_t)T] = a4;
  }
}
// out[b][p][t] = sum over chunks (ascending) / (N (T - t)) - sub[p]
__global__ void k_autocorr_final(const double* __restrict__ partials, int nchunks, int T, int N, double sub2, double sub4,
                                 double* __restrict__ out) {
  const int b = blockIdx.z, p = blockIdx.y;
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (t >= T) return;
  double s = 0.0;
  for (int c = 0; c < nchunks; c++) s += partials[(((size_t)b * nchunks + c) * 4 + p) * T + t];
  const double sub = (p == 1) ? sub2 : (p == 3) ? sub4 : 0.0;
  out[((size_t)b * 4 + p) * T + t] = s / ((double)N * (double)(T - t)) - sub;
}
int autocorr_chunks(int nseries) { return (nseries + kAcSeries - 1) / kAcSeries; }

// Green-Kubo shear-stress autocorrelation over the pressure-tensor log [B][12][nslots] (mdqt_stress_record): the three total
// off-diagonal series P_ab = K_ab + W_ab (ab = xy, xz, yz: entries 3..5 and 9..11) are formed into series[B][3][T], then the
// velocity-power correlator above runs on them as 3 series of one "ion" each: its first output, divided by 3 (T - t), is
// C(t) = 1/(3 (T - t)) sum_ab sum_{j < T - t} P_ab(j) P_ab(j + t). One chunk of series per trajectory: a fixed order.
__global__ void k_stress_series(const double* __restrict__ log, int nslots, int T, double* __restrict__ series) {
  const int b = blockIdx.y;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= 3 * T) return;
  const int q = g / T, j = g % T;
  const double* l = log + (size_t)b * kStressPerRecord * nslots;
  series[((size_t)b * 3 + q) * T + j] = l[(size_t)(3 + q) * nslots + j] + l[(size_t)(9 + q) * nslots + j];
}
int stress_autocorr_max_T() { return 48 * 1024 / (int)sizeof(double); }  // k_autocorr stages one series in shared memory
void launch_stress_autocorr(const double* log, int nslots, int B, int T, double* series, double* partials, double* out, cudaStream_t s) {
  k_stress_series<<<dim3((3 * T + 255) / 256, B), 256, 0, s>>>(log, nslots, T, series);
  static_assert(3 <= kAcSeries, "the three series of a trajectory form one chunk");
  k_autocorr<<<dim3(1, (T + 255) / 256, B), 256, (size_t)T * sizeof(double), s>>>(series, 3, T, partials);
  k_autocorr_final<<<dim3((T + 255) / 256, 1, B), 256, 0, s>>>(partials, 1, T, 3, 0.0, 0.0, out);  // the first power only: out[b][0][t]
}

// Green-Kubo heat-current autocorrelation over the heat log [B][15][nslots] (mdqt_heat_record). One CTA per trajectory forms
//   hbar = 1/(T N_b) sum_{j < T} [E_kin + E_pot + (2 E_kin + tr W)/3](j)   (thread-strided over the slots, then a fixed tree)
// -- the mean enthalpy per ion, so that hbar P is the enthalpy current that the conserved momentum P carries -- and the three series
// J_q,a(j) = J_kin,a + J_pot,a + J_vir,a - hbar P_a (j) into series[B][3][T]; the velocity-power correlator then runs on them as for
// the shear stress.
__global__ void __launch_bounds__(256) k_heat_series(const double* __restrict__ log, int nslots, int T, int N, const int* __restrict__ nb,
                                                     double* __restrict__ series) {
  __shared__ double sred[256];
  const int b = blockIdx.x, tid = threadIdx.x;
  const double* l = log + (size_t)b * kHeatPerRecord * nslots;
  const double* ekin = l + (size_t)12 * nslots;
  const double* epot = l + (size_t)13 * nslots;
  const double* trw = l + (size_t)14 * nslots;
  double h = 0.0;
  for (int j = tid; j < T; j += 256) h += ekin[j] + epot[j] + (2.0 * ekin[j] + trw[j]) / 3.0;
  sred[tid] = h;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) sred[tid] += sred[tid + o];
    __syncthreads();
  }
  const double hbar = sred[0] / ((double)T * (double)(nb ? nb[b] : N));
  for (int g = tid; g < 3 * T; g += 256) {
    const int q = g / T, j = g % T;
    series[((size_t)b * 3 + q) * T + j] = l[(size_t)q * nslots + j] + l[(size_t)(3 + q) * nslots + j] + l[(size_t)(6 + q) * nslots + j] -
                                          hbar * l[(size_t)(9 + q) * nslots + j];
  }
}
void launch_heat_autocorr(const double* log, int nslots, int B, int T, int N, const int* nb, double* series, double* partials, double* out,
                          cudaStream_t s) {
  k_heat_series<<<B, 256, 0, s>>>(log, nslots, T, N, nb, series);
  k_autocorr<<<dim3(1, (T + 255) / 256, B), 256, (size_t)T * sizeof(double), s>>>(series, 3, T, partials);
  k_autocorr_final<<<dim3((T + 255) / 256, 1, B), 256, 0, s>>>(partials, 1, T, 3, 0.0, 0.0, out);  // the first power only: out[b][0][t]
}
void launch_autocorr(const double* vstore, int N, int B, int T, double sub2, double sub4, double* partials, double* out,
                     cudaStream_t s) {
  const int nseries = 3 * N, nchunks = autocorr_chunks(nseries);
  dim3 grid(nchunks, (T + 255) / 256, B);
  k_autocorr<<<grid, 256, (size_t)T * sizeof(double), s>>>(vstore, nseries, T, partials);
  dim3 g2((T + 255) / 256, 4, B);
  k_autocorr_final<<<g2, 256, 0, s>>>(partials, nchunks, T, N, sub2, sub4, out);
}

// ------------------------------------------------------------------------------------------------------------
// MD-family recorders that are plain reductions over the velocities: recordTemperature() (MD:525-546),
// recordTempForEachAxis() (MD:560-582) and recordTaggedParticleMoments() (MD:923-1029; MC408L:1069). One record =
// 23 sums per trajectory: sum v_x^2, v_y^2, v_z^2 over all ions, then for each of the four tag sets (bit k of tags[i]):
// count, sum v_x, v_x^2, v_x^3, v_x^4 (powers formed left to right as the reference writes them). The host divides and
// subtracts the equilibrium constants. One CTA per trajectory, thread-strided sums + a fixed tree: reproducible.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_moments(const double* __restrict__ V, const unsigned char* __restrict__ tags, int N, int ld,
                                                  double* __restrict__ out) {
  __shared__ double sred[32];
  const int b = blockIdx.x;
  const double* vx = V + (size_t)b * 3 * ld;
  const double* vy = vx + ld;
  const double* vz = vy + ld;
  const unsigned char* tg = tags ? tags + (size_t)b * N : nullptr;
  double acc[kMomentsPerRecord];
#pragma unroll
  for (int k = 0; k < kMomentsPerRecord; k++) acc[k] = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double x = vx[i], y = vy[i], z = vz[i];
    acc[0] += x * x; acc[1] += y * y; acc[2] += z * z;
    const unsigned m = tg ? tg[i] : 0u;
    const double x2 = x * x, x3 = x2 * x, x4 = x3 * x;
#pragma unroll
    for (int k = 0; k < 4; k++)
      if (m & (1u << k)) { acc[3 + 5 * k] += 1.0; acc[4 + 5 * k] += x; acc[5 + 5 * k] += x2; acc[6 + 5 * k] += x3; acc[7 + 5 * k] += x4; }
  }
#pragma unroll
  for (int k = 0; k < kMomentsPerRecord; k++) {
    const double tot = block_sum_1024(acc[k], sred);
    if (threadIdx.x == 0) out[(size_t)b * kMomentsPerRecord + k] = tot;
  }
}
void launch_moments(const double* V, const unsigned char* tags, int N, int ld, int B, double* out, cudaStream_t s) {
  k_moments<<<B, 1024, 0, s>>>(V, tags, N, ld, out);
}

// Velocity distribution of the TAGGED ions (bit 0 of tags), x component, as recordTaggedParticleMoments() of the tagging programs
// forms it (MC408L:1069-1137; output() FZ408L:835-893): 4001 bins vel_j = (j - 2000) * 0.0025, Gaussian weights of width 0.002,
// divided by 6 sqrt(2 pi 0.002^2). grid (ceil(4001/8), B), 256 threads = 8 bins x 32 lanes striding over the ions.
__global__ void __launch_bounds__(256) k_vel_dist_tagged(const double* __restrict__ V, const unsigned char* __restrict__ tags, int N, int ld,
                                                         double* __restrict__ pv) {
  const int b = blockIdx.y;
  const int bin = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const double* vx = V + (size_t)b * 3 * ld;
  const unsigned char* tg = tags + (size_t)b * N;
  const double V2 = 1. / (2. * 0.002 * 0.002), vb = (double)(bin - 2000) * 0.0025;
  double s = 0.0;
  if (bin < kTagBins)
    for (int i = lane; i < N; i += 32)
      if (tg[i] & 1) { const double d = vb - vx[i]; s += exp(-V2 * d * d); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0 && bin < kTagBins) pv[(size_t)b * kTagBins + bin] = s / (6.0 * sqrt(2 * M_PI * 0.002 * 0.002));
}
void launch_vel_dist_tagged(const double* V, const unsigned char* tags, int N, int ld, int B, double* pv, cudaStream_t s) {
  dim3 grid((kTagBins + 7) / 8, B);
  k_vel_dist_tagged<<<grid, 256, 0, s>>>(V, tags, N, ld, pv);
}

// anisotropizeVelocities() (MD:548-558): V_c *= scale_c
__global__ void k_scale_velocities(double* __restrict__ V, int N, int ld, int B, double sx, double sy, double sz) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= 3LL * N * B) return;
  const int i = (int)(g % N), bc = (int)(g / N), c = bc % 3;
  double* v = V + (size_t)bc * ld + i;
  *v = __dmul_rn(c == 0 ? sx : (c == 1 ? sy : sz), *v);
}
void launch_scale_velocities(double* V, int N, int ld, int B, double sx, double sy, double sz, cudaStream_t s) {
  const long long n = 3LL * N * B;
  k_scale_velocities<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(V, N, ld, B, sx, sy, sz);
}

// pops[b][i][3] = popS, popP, popD with the reference's state grouping (12/7-level: S 0,1; P 2..5; D 6..S-1)
__global__ void k_populations(const double* __restrict__ psi, int S, int N, int ld, double* __restrict__ pops) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double* p = psi + (size_t)b * 2 * S * ld;
  double pop[3] = {0.0, 0.0, 0.0};
  // ground / excited / reservoir grouping: 12- and 7-level 2+4(+D), 5-level 2+2+1 (MC422L:104-108), 3-level 1+2 (TS:95-97)
  const int nS = (S == 3) ? 1 : 2, nP = (S >= 7) ? 4 : 2;
  for (int k = 0; k < S; k++) {
    double re = p[(size_t)(2 * k) * ld + i], im = p[(size_t)(2 * k + 1) * ld + i];
    pop[k < nS ? 0 : (k < nS + nP ? 1 : 2)] += re * re + im * im;
  }
  double* o = pops + ((size_t)b * N + i) * 3;
  o[0] = pop[0]; o[1] = pop[1]; o[2] = pop[2];
}

void launch_populations(const double* psi, int S, int N, int ld, int B, double* pops, cudaStream_t s) {
  dim3 grid((N + 255) / 256, B);
  k_populations<<<grid, 256, 0, s>>>(psi, S, N, ld, pops);
}

// psi_aos[b][i][k][2]  <->  psi_soa[b][2k+c][ld]
__global__ void k_psi_in(const double* __restrict__ aos, double* __restrict__ soa, int S, int N, int ld) {
  const int b = blockIdx.y;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)N * 2 * S) return;
  const int i = (int)(g / (2 * S)), kc = (int)(g % (2 * S));
  soa[((size_t)b * 2 * S + kc) * ld + i] = aos[(size_t)b * N * 2 * S + g];
}
__global__ void k_psi_out(const double* __restrict__ soa, double* __restrict__ aos, int S, int N, int ld) {
  const int b = blockIdx.y;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)N * 2 * S) return;
  const int i = (int)(g / (2 * S)), kc = (int)(g % (2 * S));
  aos[(size_t)b * N * 2 * S + g] = soa[((size_t)b * 2 * S + kc) * ld + i];
}
void launch_transpose_psi_in(const double* psi_aos, double* psi_soa, int S, int N, int ld, int B, cudaStream_t s) {
  long long n = (long long)N * 2 * S;
  dim3 grid((unsigned)((n + 255) / 256), B);
  k_psi_in<<<grid, 256, 0, s>>>(psi_aos, psi_soa, S, N, ld);
}
void launch_transpose_psi_out(const double* psi_soa, double* psi_aos, int S, int N, int ld, int B, cudaStream_t s) {
  long long n = (long long)N * 2 * S;
  dim3 grid((unsigned)((n + 255) / 256), B);
  k_psi_out<<<grid, 256, 0, s>>>(psi_soa, psi_aos, S, N, ld);
}

}  // namespace mdqt
