// mdqt_capi.cu -- the C ABI declared in include/mdqt.h: handle management, state marshalling between the
// reference's host layouts (double R[3][ld], cx_mat wvFns[], SU:126-152) and the device SoA layout, and the
// stream-ordered sequencing of the hot-path kernels (the body of the reference's main loop, SU:1369-1378).
// There is no CPU fallback anywhere in this file: without a CUDA device every entry point fails.
#include "mdqt_handle.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <new>
#include <string>
#include <vector>

using namespace mdqt;
#define force_args mdqt_force_args
#define qt_args mdqt_qt_args
#define refresh_fixed mdqt_refresh_fixed
#define enqueue_substeps mdqt_enqueue_substeps

static thread_local std::string g_err;
int mdqt_fail(int code, const std::string& msg) { g_err = msg; return code; }
static int fail(int code, const std::string& msg) { return mdqt_fail(code, msg); }

__global__ void k_init_stamps(unsigned long long* s, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) { s[2 * k] = ~0ULL; s[2 * k + 1] = 0ULL; }
}

__global__ void k_set_clock(double* clock, double t, unsigned long long substep, unsigned long long vv_step) {
  clock[0] = t;
  reinterpret_cast<unsigned long long*>(clock)[1] = substep;
  reinterpret_cast<unsigned long long*>(clock)[2] = vv_step;
}

static size_t state_elems(const mdqt_handle* h) { return (size_t)h->B * 3 * h->ld; }

extern "C" {

const char* mdqt_last_error(void) { return g_err.c_str(); }
const char* mdqt_version(void) { return "mdqt_b200 0.1 (sm_100a)"; }

int mdqt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int mdqt_params_su(mdqt_params* p, double Ge, double density, double sig0, double Te, double fracOfSig, double detuning,
                   double detuningDP, double Om, double OmDP, int N0, int n_ions) {
  if (!p) return fail(MDQT_EINVAL, "null params");
  memset(p, 0, sizeof(*p));
  p->struct_bytes = (int32_t)sizeof(*p);
  p->scheme = MDQT_SCHEME_SR12;
  p->n_ions = n_ions; p->n_traj = 1; p->traj0 = 1; p->row0 = 0; p->n_rows = 0; p->device = 0;
  p->substeps_per_md = (int)ceil(34.81 / sqrt(density));          // SU:83
  p->L = pow(N0 * 4. * M_PI / 3., 0.333333333);                   // SU:297 (literal exponent)
  p->kappa = 1.0 / (1. / sqrt(3. * Ge));                          // 1/lDeb, SU:295
  p->rcut = p->L / 2.;                                            // SU:195
  p->dtq = 0.002 / p->substeps_per_md;                            // SU:80, 84
  p->detuning = detuning; p->detuningDP = detuningDP; p->Om = Om; p->OmDP = OmDP;
  p->dR = 0.0617; p->kRat = 0.395;                                // SU:146-147
  p->g2E = 174.07 / sqrt(density);                                // SU:79
  p->pv2qv = 1.1821 * pow(density, 1. / 6);                       // SU:85
  p->vKick = 0.001208 / p->pv2qv;                                 // SU:148
  p->vKickDP = p->vKick * p->kRat;                                // SU:149
  p->fracOfSig = fracOfSig; p->Te = Te; p->sig0 = sig0; p->density = density;
  p->seed = 12345;
  return MDQT_OK;
}

int mdqt_params_md(mdqt_params* p, int scheme, int n_ions, double kappa, double density, double timeStep, double detuning,
                   double Om, int quad) {
  if (!p) return fail(MDQT_EINVAL, "null params");
  memset(p, 0, sizeof(*p));
  p->struct_bytes = (int32_t)sizeof(*p);
  p->scheme = scheme;
  p->n_ions = n_ions; p->n_traj = 1; p->traj0 = 1; p->device = 0;
  p->L = pow(n_ions * 4. * M_PI / 3., 1. / 3);                    // MD:73
  p->kappa = kappa; p->rcut = p->L / 2.;                          // MD:67, 74
  p->substeps_per_md = (int)round(87 / sqrt(density));            // MC408L:116
  p->dtq = timeStep / p->substeps_per_md;                         // MC408L:117
  p->detuning = detuning; p->Om = Om; p->quad = quad;
  p->dR = 0.0617;                                                 // MC408L:121
  p->g2E = 174.07 / sqrt(density);                                // MC408L:115
  p->pv2qv = 1.1821 * pow(density, 1. / 6);                       // MC408L:118
  p->vKick = 0.001208 / p->pv2qv;                                 // MC408L:122
  p->density = density; p->sig0 = 1.0;
  p->seed = 12345;
  if (scheme == MDQT_SCHEME_CA5) {                                // 422 nm constants (MC422L:113-121)
    p->g2E = 174.07 * .894 / sqrt(density);
    p->substeps_per_md = (int)round(87 * .894 / sqrt(density));
    p->dtq = timeStep / p->substeps_per_md;
    p->pv2qv = 1.1821 * pow(density, 1. / 6) * .967;
    p->dR = 0.0753;
    p->vKick = 0.001257 / p->pv2qv;
  }
  return MDQT_OK;
}

int mdqt_params_ts(mdqt_params* p, int n_ions, double detuning, double Om) {
  if (!p) return fail(MDQT_EINVAL, "null params");
  memset(p, 0, sizeof(*p));
  p->struct_bytes = (int32_t)sizeof(*p);
  p->scheme = MDQT_SCHEME_V3;
  p->n_ions = n_ions; p->n_traj = 1; p->traj0 = 1; p->device = 0;
  p->L = 1.0; p->kappa = 0.0; p->rcut = 0.5;                      // no plasma in this program: unused
  p->substeps_per_md = 1;
  p->dtq = 0.01;                                                  // dt (TS:390), already in units of 1/gamma
  p->g2E = 1.0; p->pv2qv = 1.0;                                   // velQuant = V[0][i] (TS:154)
  p->detuning = detuning; p->Om = Om;
  p->vKick = 0.0012076;                                           // TS:91
  p->density = 1.0; p->sig0 = 1.0;
  p->seed = 12345;
  return MDQT_OK;
}

// j-range decomposition: a function of (N, B) only, so that every rank of a row-decomposed run sums the same
// j-chunks in the same order (bitwise identical forces for any GPU count).
// Item-walking kernel (k_pairs_items): chunk length for `np` ions, chosen for ONE trajectory on the chip's 148 x 2 x 8
// resident warps -- the latency-critical case; a batch walks B times as many equal items whatever the choice. A function of
// np alone (a trajectory's own ion count -- n_ions, or its entry in mdqt_set_ion_counts -- or the nominal mdqt_params.plan_n): not of
// the batch size, the row range or the environment.
static int plan_items_jlen(int np) {
  const long long W = 148LL * 2 * 8;
  const long long G = (np + 31) / 32;
  double best = 1e300;
  int best_jl = 8;
  for (int jl = 8; jl <= 256; jl += 8) {  // kItemMaxJ
    const long long nch = (np + jl - 1) / jl;
    const long long rounds = (G * nch + W - 1) / W;
    // per item: jl pair iterations + ~14 iterations' worth of tile wait, partial store, fence and arrival; the last warp of
    // a group fetches the partials in batches of 12 (one L2 round trip ~ 6 iterations each)
    const double cost = (double)rounds * (jl + 14) + (nch > 1 ? 6.0 * ((nch + 11) / 12) : 0.0);
    if (cost < best) { best = cost; best_jl = jl; }
  }
  return best_jl;
}
constexpr int kItemsMaxN = 8192;  // beyond this the partial-sum buffer (chunks x 3 x N) grows and CTA tiles win anyway

static void plan_force(mdqt_handle* h) {
  // developer knobs (kernel A/B runs) are honoured on whole-system handles only: the ranks of a row-decomposed run must take the
  // same plan whatever their environments, or the rank-count-independent bits are gone
  auto knob = [h](const char* name) -> const char* { return h->nrows == h->N ? getenv(name) : nullptr; };
  h->items = 0;
  h->pdl = pdl_mode() == 1 ? 1 : 0;
  {
    const int np = h->p.plan_n > 0 ? h->p.plan_n : h->N;
    const char* e = knob("MDQT_K1_ITEMS");  // developer knob (A/B runs): 0 = CTA-tile kernel everywhere
    const bool off = e && e[0] == '0' && h->p.plan_n == 0;
    // the chunk length must cover every trajectory's ions in <= 64 chunks even when n_ions exceeds the nominal plan_n
    const long long total_items = (long long)h->B * ((h->nrows + 31) / 32) * ((h->N + 7) / 8);  // bound for any chunk length
    if (np <= kItemsMaxN && h->N <= 2 * np && total_items < (1LL << 24) && !off) {
      h->items = 1;
      h->jlen = plan_items_jlen(np);
      h->nsplit = (h->N + h->jlen - 1) / h->jlen;
      h->ipt = 1; h->jsub = 1; h->rg = 32;
      h->itiles = (h->nrows + 31) / 32;
      // one trajectory whose items fit ONE round of the resident warps: all force warps finish together, which is when programmatic
      // dependent launch pays (pdl_mode)
      if (pdl_mode() < 0) h->pdl = (h->B == 1 && h->nrows == h->N && (long long)h->itiles * h->nsplit <= 148LL * 2 * 8) ? 1 : 0;
      return;
    }
  }
  // Cost model (fitted to B200 timings, profiles/): the kernel is issue-bound, so an SM's time is the work of the
  // CTAs assigned to it -- ceil(ctas/148) x (jlen + fixed CTA overhead) x rows per thread -- as long as >= 4 CTAs
  // are co-resident; two rows per thread amortise the shared-memory reads (~3 % fewer issue slots per pair).
  const int N = h->N, B = h->B;
  double best = 1e300; int best_ns = 1, best_jlen = N, best_ipt = 1;
  for (int ipt = 1; ipt <= 2; ipt++) {
    const long long tiles = ((long long)N + kForceThreads * ipt - 1) / (kForceThreads * ipt) * B;
    for (int ns = 1; ns <= 64; ns++) {
      int jlen = ((N + ns - 1) / ns + 7) & ~7;
      int real_ns = (N + jlen - 1) / jlen;
      long long ctas = tiles * real_ns;
      double per_sm = (double)ctas / 148.0;
      // +1: expected load imbalance of one CTA per SM; below ~3.5 CTAs (14 warps) per SM the issue slots starve
      double sat = per_sm >= 3.5 ? 1.0 : per_sm / 3.5;
      double cost = (per_sm + 1.0) * (jlen + 60 + 2 * real_ns) * ipt * (ipt == 2 ? 0.97 : 1.0) / sat;
      if (cost < best * 0.999) { best = cost; best_ns = real_ns; best_jlen = jlen; best_ipt = ipt; }
    }
  }
  const int ipt = best_ipt;
  h->nsplit = best_ns; h->jlen = best_jlen; h->ipt = ipt;
  // few CTAs per SM (small N): split every j tile over two 128-thread groups inside the CTA -> twice the resident warps
  {
    const long long tiles1 = ((long long)N + kForceThreads - 1) / kForceThreads * B;
    h->jsub = (ipt == 1 && tiles1 * h->nsplit < 148LL * 7) ? 2 : 1;
  }
  h->rg = kForceThreads;
  // Small and medium systems (one row per thread in the plan above): compare that plan with 32-row groups whose j range
  // is split over 4 or 8 warps INSIDE the CTA, so a row's force is spread over 4-8x fewer CTAs (often over one: no partial
  // sums, no arrival counter, no final reduction at all). Model from the per-CTA phase trace and the plan timings on
  // B200 (profiles/r01c_k1_trace.txt): time = (largest number of CTAs on one SM) x (warp-pairs per CTA) x ~81 issue
  // cycles / 4 sub-partitions + a plan-independent ~5.5 us; what separates plans is almost only the first term, i.e.
  // how evenly the CTA count divides over 148 SMs (measured launch times move in ~2 us steps).
  if (h->ipt == 1 && !knob("MDQT_FORCE_IPT") && !knob("MDQT_FORCE_NSPLIT")) {
    auto model = [&](long long ctas, int warps, double pairs_per_warp, int ns) {
      const double per_sm = (double)((ctas + 147) / 148);
      const double resident = std::min(per_sm * warps, 32.0);
      const double starve = resident >= 16.0 ? 1.0 : 16.0 / resident;  // fewer than 4 warps per sub-partition
      // + launch gap and CTA prologue/epilogue (~5.5 us whatever the plan), a mild cost per CTA wave, and one L2 round
      // trip per 8 partial sums in the final reduction
      return per_sm * warps * pairs_per_warp * 81.0 / (4 * 1965.0) * starve + 5.5 + 0.15 * per_sm + (ns > 1 ? 0.9 * ((ns + 7) / 8) : 0.0);
    };
    const long long tiles128 = ((long long)N + 127) / 128 * B, tiles32 = ((long long)N + 31) / 32 * B;
    double best_t = model(tiles128 * h->nsplit, 4 * h->jsub, (double)h->jlen / h->jsub, h->nsplit);
    for (int js = 8; js >= 4; js /= 2)
      for (int ns = 1; ns <= 16; ns++) {
        // chunk length = a multiple of (in-CTA groups x loop unroll = js x 8): every warp's share is whole unrolled
        // iterations (the scalar remainder loop has no ILP and all warps reach it together)
        const int q = js * 8;
        const int jlen = ((N + ns - 1) / ns + q - 1) / q * q;
        const int real_ns = (N + jlen - 1) / jlen;
        if (real_ns != ns) continue;
        const double t = model(tiles32 * ns, js, (double)jlen / js, ns);
        if (t < best_t * 0.98) { best_t = t; h->rg = 32; h->jsub = js; h->nsplit = ns; h->jlen = jlen; h->ipt = 1; }
      }
  }
  if (const char* e = knob("MDQT_FORCE_RG")) {  // developer knob: MDQT_FORCE_RG=32 with MDQT_FORCE_JSUB=4|8 and MDQT_FORCE_NSPLIT
    if (atoi(e) == 32) { h->rg = 32; h->ipt = 1; h->jsub = 8; }
    else h->rg = kForceThreads;
  }
  if (const char* e = knob("MDQT_FORCE_JSUB")) {
    int js = atoi(e);
    if (h->rg == 32) h->jsub = js == 4 ? 4 : 8;
    else h->jsub = (js == 2 || (js == 4 && knob("MDQT_FORCE_IPT") && atoi(knob("MDQT_FORCE_IPT")) == 2)) ? js : 1;
  }
  // developer tuning knobs (kernel A/B runs): override the plan
  if (const char* e = knob("MDQT_FORCE_IPT")) h->ipt = (atoi(e) == 2 && h->rg != 32) ? 2 : 1;
  if (const char* e = knob("MDQT_FORCE_NSPLIT")) {
    int ns = std::max(1, std::min(1024, atoi(e)));
    h->jlen = ((N + ns - 1) / ns + 7) & ~7;
    h->nsplit = (N + h->jlen - 1) / h->jlen;
  }
  // (Row-decomposed handles keep the rows-per-thread choice of the whole-system plan: choosing it per rank from a CTA-wave count
  // was measured slower -- N = 2e5 on 8 ranks: 10.18 ms with one row per thread (4.97 waves) against 9.88 ms with two (2.48 waves);
  // CTAs are scheduled dynamically, so partial waves cost little, while two rows per thread issue 3 % fewer instructions.)
  h->itiles = (h->nrows + 31) / 32;  // upper bound on i-tiles of this handle (32-row groups)
}

int mdqt_create(const mdqt_params* p, mdqt_handle** out) {
  if (!p || !out) return fail(MDQT_EINVAL, "null argument");
  *out = nullptr;
  if (p->struct_bytes != (int32_t)sizeof(mdqt_params)) return fail(MDQT_EINVAL, "mdqt_params size mismatch (ABI)");
  if (p->scheme != MDQT_SCHEME_NONE && p->scheme != MDQT_SCHEME_SR7 && p->scheme != MDQT_SCHEME_SR12 &&
      p->scheme != MDQT_SCHEME_CA5 && p->scheme != MDQT_SCHEME_V3)
    return fail(MDQT_EINVAL, "unknown level scheme");
  if (p->n_ions < 1 || p->n_traj < 1) return fail(MDQT_EINVAL, "n_ions and n_traj must be >= 1");
  if (!(p->L > 0) || !(p->rcut > 0) || !(p->kappa >= 0)) return fail(MDQT_EINVAL, "L, rcut must be > 0 and kappa >= 0");
  if (p->kappa * p->rcut > 700.0) return fail(MDQT_EINVAL, "kappa*rcut too large for the fp64 exp range");
  if (p->rcut > p->L / 2. * (1 + 1e-12)) return fail(MDQT_EINVAL, "rcut must not exceed L/2 (minimum image)");
  int row0 = p->row0, nrows = p->n_rows == 0 ? p->n_ions : p->n_rows;
  if (row0 < 0 || nrows < 1 || row0 + nrows > p->n_ions) return fail(MDQT_EINVAL, "row range outside [0,n_ions)");
  if (p->scheme != MDQT_SCHEME_NONE && !(p->dtq > 0)) return fail(MDQT_EINVAL, "dtq must be > 0");
  int ndev = mdqt_device_count();
  if (ndev <= 0) return fail(MDQT_ENODEVICE, "no CUDA device: libmdqt_b200 has no CPU fallback");
  if (p->device < 0 || p->device >= ndev) return fail(MDQT_EINVAL, "device ordinal out of range");
  CU(cudaSetDevice(p->device));

  mdqt_handle* h = new (std::nothrow) mdqt_handle();
  if (!h) return fail(MDQT_ENOMEM, "host allocation failed");
  h->p = *p;
  h->N = p->n_ions; h->B = p->n_traj; h->S = p->scheme; h->row0 = row0; h->nrows = nrows;
  h->ld = (p->n_ions + 31) & ~31;
  h->t = 0.0; h->substep = 0; h->vv_step = 0; h->Rfix = nullptr; h->rfix_dirty = 1;
  h->forced_u = nullptr; h->forced_nsub = 0; h->forced_cursor = 0; h->forced_cu = h->forced_cn = nullptr;
  h->vhold = nullptr; h->forced_tag = nullptr; h->tagged = nullptr;
  h->gr_counts = nullptr; h->vstore = h->ac_partials = h->ac_out = nullptr; h->vstore_T = 0;
  h->clock = nullptr; h->nb = nullptr; h->seeds = nullptr; h->comm = nullptr; h->ilist = nullptr; h->icount = 0;
  h->tags = nullptr; h->moments = nullptr; h->moments_slots = 0;
  h->stress = h->stress_partials = h->stress_series = h->stress_ac_partials = h->stress_ac_out = nullptr;
  h->stress_slots = h->stress_ac_cap = 0; h->stress_partials_cap = 0;
  h->heat = h->heat_partials = h->heat_series = h->heat_ac_partials = h->heat_ac_out = nullptr;
  h->heat_slots = h->heat_ac_cap = 0; h->heat_partials_cap = 0;
  h->timing = 0; h->ev_used = 0; h->stamps = nullptr; h->stamps_cap = 0;
  for (int k = 0; k < 4; k++) { h->time_ms[k] = 0; h->time_n[k] = 0; }
  plan_force(h);
  if (h->S) fill_qt_consts(h->qc, h->S, p->Om, p->OmDP, p->dR, p->vKick, p->vKickDP, p->dtq, p->g2E, p->quad);
  upload_exp_table();

  cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  size_t ne = state_elems(h);
  auto alloc = [&](double** ptr, size_t n) {
    if (e == cudaSuccess) { e = cudaMalloc((void**)ptr, std::max<size_t>(n, 1) * sizeof(double)); if (e == cudaSuccess) e = cudaMemset(*ptr, 0, std::max<size_t>(n, 1) * sizeof(double)); }
  };
  alloc(&h->R, ne); alloc(&h->V, ne); alloc(&h->F, ne); alloc(&h->oldF, ne);
  alloc(&h->psi, (size_t)h->B * 2 * h->S * h->ld);
  alloc(&h->psi_stage, (size_t)h->B * 2 * h->S * h->N);
  alloc(&h->tPart, (size_t)h->B * h->ld);
  alloc(&h->Fpart, h->nsplit > 1 ? (size_t)h->nsplit * ne : 1);
  alloc(&h->epot_partials, (size_t)h->itiles * h->nsplit * h->B);
  alloc(&h->scalars, (size_t)h->B * 16);
  alloc(&h->pvel, (size_t)h->B * 3 * kVelBins);
  alloc(&h->pops, (size_t)h->B * h->N * 3);
  alloc(&h->clock, 4);
  if (e == cudaSuccess) {
    e = cudaMalloc((void**)&h->Rfix, sizeof(long long) * std::max<size_t>(ne, 1));
    if (e == cudaSuccess) e = cudaMemset(h->Rfix, 0, sizeof(long long) * std::max<size_t>(ne, 1));
  }
  if (e == cudaSuccess) {
    e = cudaMalloc((void**)&h->counters, sizeof(unsigned) * (size_t)h->B * h->itiles);
    if (e == cudaSuccess) e = cudaMemset(h->counters, 0, sizeof(unsigned) * (size_t)h->B * h->itiles);
  }
  if (e != cudaSuccess) {
    std::string m = std::string("device allocation failed: ") + cudaGetErrorString(e);
    mdqt_destroy(h);
    return fail(e == cudaErrorMemoryAllocation ? MDQT_ENOMEM : MDQT_ECUDA, m);
  }
  *out = h;
  return MDQT_OK;
}

int mdqt_destroy(mdqt_handle* h) {
  if (!h) return MDQT_OK;
  cudaSetDevice(h->p.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  mdqt_comm_release(h);
  double* bufs[] = {h->R, h->V, h->F, h->oldF, h->psi, h->psi_stage, h->tPart, h->Fpart, h->epot_partials, h->scalars,
                    h->pvel, h->pops, h->forced_u, h->forced_cu, h->forced_cn, h->vhold, h->forced_tag};
  for (double* b : bufs) if (b) cudaFree(b);
  if (h->tagged) cudaFree(h->tagged);
  if (h->clock) cudaFree(h->clock);
  if (h->nb) cudaFree(h->nb);
  if (h->jl) cudaFree(h->jl);
  if (h->ilist) cudaFree(h->ilist);
  if (h->tags) cudaFree(h->tags);
  if (h->moments) cudaFree(h->moments);
  for (double* b : {h->stress, h->stress_partials, h->stress_series, h->stress_ac_partials, h->stress_ac_out}) if (b) cudaFree(b);
  for (double* b : {h->heat, h->heat_partials, h->heat_series, h->heat_ac_partials, h->heat_ac_out}) if (b) cudaFree(b);
  if (h->stamps) cudaFree(h->stamps);
  if (h->seeds) cudaFree(h->seeds);
  for (GraphEntry& g : h->graphs) cudaGraphExecDestroy(g.exec);
  if (h->gr_counts) cudaFree(h->gr_counts);
  if (h->vstore) cudaFree(h->vstore);
  if (h->ac_partials) cudaFree(h->ac_partials);
  if (h->ac_out) cudaFree(h->ac_out);
  if (h->counters) cudaFree(h->counters);
  if (h->Rfix) cudaFree(h->Rfix);
  for (cudaEvent_t ev : h->ev) cudaEventDestroy(ev);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return MDQT_OK;
}

int mdqt_sync(mdqt_handle* h) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (h->comm) mdqt_comm_sync_pending(h);
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

// [B][3][ld_host] host <-> [B][3][ld] device, N valid columns
static cudaError_t copy_state(mdqt_handle* h, double* dev, const double* host_in, double* host_out, int ld_host) {
  const int rows = h->B * 3;
  if (host_in)
    return cudaMemcpy2DAsync(dev, (size_t)h->ld * 8, host_in, (size_t)ld_host * 8, (size_t)h->N * 8, rows, cudaMemcpyHostToDevice, h->stream);
  return cudaMemcpy2DAsync(host_out, (size_t)ld_host * 8, dev, (size_t)h->ld * 8, (size_t)h->N * 8, rows, cudaMemcpyDeviceToHost, h->stream);
}

int mdqt_upload_state(mdqt_handle* h, const double* R, const double* V, const double* psi, const double* tPart, int ld) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (ld < h->N) return fail(MDQT_EINVAL, "ld smaller than n_ions");
  CU(cudaSetDevice(h->p.device));
  if (R) {
    h->rfix_dirty = 1;
    CU(copy_state(h, h->R, R, nullptr, ld));
  }
  if (V) CU(copy_state(h, h->V, V, nullptr, ld));
  if (psi) {
    if (!h->S) return fail(MDQT_ESTATE, "handle has no wavefunctions (scheme NONE)");
    CU(cudaMemcpyAsync(h->psi_stage, psi, (size_t)h->B * h->N * 2 * h->S * 8, cudaMemcpyHostToDevice, h->stream));
    launch_transpose_psi_in(h->psi_stage, h->psi, h->S, h->N, h->ld, h->B, h->stream);
  }
  if (tPart)
    CU(cudaMemcpy2DAsync(h->tPart, (size_t)h->ld * 8, tPart, (size_t)h->N * 8, (size_t)h->N * 8, h->B, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));  // host buffers are caller-owned: do not hold on to them
  return MDQT_OK;
}

int mdqt_download_state(mdqt_handle* h, double* R, double* V, double* psi, double* tPart, int ld) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (ld < h->N) return fail(MDQT_EINVAL, "ld smaller than n_ions");
  CU(cudaSetDevice(h->p.device));
  if (R) CU(copy_state(h, h->R, nullptr, R, ld));
  if (V) CU(copy_state(h, h->V, nullptr, V, ld));
  if (psi) {
    if (!h->S) return fail(MDQT_ESTATE, "handle has no wavefunctions (scheme NONE)");
    launch_transpose_psi_out(h->psi, h->psi_stage, h->S, h->N, h->ld, h->B, h->stream);
    CU(cudaMemcpyAsync(psi, h->psi_stage, (size_t)h->B * h->N * 2 * h->S * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  if (tPart)
    CU(cudaMemcpy2DAsync(tPart, (size_t)h->N * 8, h->tPart, (size_t)h->ld * 8, (size_t)h->N * 8, h->B, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_upload_forces(mdqt_handle* h, const double* F, int ld) {
  if (!h || !F) return fail(MDQT_EINVAL, "null argument");
  if (ld < h->N) return fail(MDQT_EINVAL, "ld smaller than n_ions");
  CU(cudaSetDevice(h->p.device));
  CU(copy_state(h, h->F, F, nullptr, ld));
  CU(cudaStreamSynchronize(h->stream));
  return MDQT_OK;
}
int mdqt_download_forces(mdqt_handle* h, double* F, int ld) {
  if (!h || !F) return fail(MDQT_EINVAL, "null argument");
  if (ld < h->N) return fail(MDQT_EINVAL, "ld smaller than n_ions");
  CU(cudaSetDevice(h->p.device));
  CU(copy_state(h, h->F, nullptr, F, ld));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_set_time(mdqt_handle* h, double t, uint64_t substep_index) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  h->t = t; h->substep = substep_index;
  return MDQT_OK;
}
int mdqt_get_time(mdqt_handle* h, double* t, uint64_t* substep_index) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (t) *t = h->t;
  if (substep_index) *substep_index = h->substep;
  return MDQT_OK;
}

int mdqt_set_ion_counts(mdqt_handle* h, const int32_t* n_ions) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (!n_ions) {
    if (h->nb) { cudaFree(h->nb); h->nb = nullptr; }
    h->nb_host.clear();
  } else {
    if (h->S != MDQT_SCHEME_SR12 && h->S != MDQT_SCHEME_NONE) return fail(MDQT_ESTATE, "per-trajectory ion counts need the 12-level scheme (or none)");
    if (h->nrows != h->N) return fail(MDQT_ESTATE, "per-trajectory ion counts on a row-decomposed handle");
    if (!h->items) return fail(MDQT_ESTATE, "per-trajectory ion counts need the item-walking force plan (n_ions <= 8192)");
    for (int b = 0; b < h->B; b++)
      if (n_ions[b] < 1 || n_ions[b] > h->N) return fail(MDQT_EINVAL, "ion count outside [1, n_ions]");
    if (!h->nb) CU(cudaMalloc((void**)&h->nb, sizeof(int) * (size_t)h->B));
    CU(cudaMemcpy(h->nb, n_ions, sizeof(int) * (size_t)h->B, cudaMemcpyHostToDevice));
    h->nb_host.assign(n_ions, n_ions + h->B);
  }
  // The chunk length of the item force kernel is a function of each trajectory's OWN ion count (plan_n == 0; a non-zero plan_n fixes one
  // length for all): a job sums its forces in the same order alone (n_ions = its N) and in any batch, and every job gets the plan
  // that fits its N (a nominal plan spills into a second round of items for the third of the jobs above N0 + 0.5 sigma).
  {
    const int old_nsplit = h->nsplit;
    if (h->jl) { cudaFree(h->jl); h->jl = nullptr; }
    plan_force(h);  // the uniform plan for N = n_ions (or plan_n)
    if (n_ions && h->p.plan_n == 0) {
      std::vector<int> jl(h->B);
      int jmax = 8, nsmax = 1;
      for (int b = 0; b < h->B; b++) {
        jl[b] = plan_items_jlen(n_ions[b]);
        jmax = std::max(jmax, jl[b]);
        nsmax = std::max(nsmax, (n_ions[b] + jl[b] - 1) / jl[b]);
      }
      CU(cudaMalloc((void**)&h->jl, sizeof(int) * (size_t)h->B));
      CU(cudaMemcpy(h->jl, jl.data(), sizeof(int) * (size_t)h->B, cudaMemcpyHostToDevice));
      h->jlen = jmax; h->nsplit = nsmax;  // tile capacity and chunk-slot capacity of the batch
      if (pdl_mode() < 0) h->pdl = (h->B == 1 && (long long)((n_ions[0] + 31) / 32) * h->nsplit <= 148LL * 2 * 8) ? 1 : 0;
    }
    // unequal ion counts leave ~8 % of the (trajectory, row group, chunk) slots empty, and a static walk over slots then gives the warps
    // 29-34 real items each: hand the kernel the packed list of the non-empty items (two rows per lane: the batch instantiations)
    if (h->ilist) { cudaFree(h->ilist); h->ilist = nullptr; h->icount = 0; }
    static const bool use_list = [] { const char* e = getenv("MDQT_K1_ILIST"); return !(e && e[0] == '0'); }();  // A/B knob
    if (n_ions && h->items && h->B > 1 && h->B < (1 << 14) && h->nsplit <= 1024 && h->N <= 64 * 256 && use_list) {
      std::vector<unsigned> list;
      list.reserve((size_t)h->B * ((h->N + 63) / 64) * h->nsplit);
      for (int b = 0; b < h->B; b++) {
        const int jlb = (h->p.plan_n == 0) ? plan_items_jlen(n_ions[b]) : h->jlen;
        const int groups = (n_ions[b] + 63) / 64, nch = (n_ions[b] + jlb - 1) / jlb;
        for (int g = 0; g < groups; g++)
          for (int ch = 0; ch < nch; ch++) list.push_back((unsigned)b << 18 | (unsigned)g << 10 | (unsigned)ch);
      }
      CU(cudaMalloc((void**)&h->ilist, sizeof(unsigned) * list.size()));
      CU(cudaMemcpy(h->ilist, list.data(), sizeof(unsigned) * list.size(), cudaMemcpyHostToDevice));
      h->icount = (int)list.size();
    }
    if (h->nsplit != old_nsplit) {  // the partial-sum buffers are sized by the number of chunk slots
      cudaFree(h->Fpart); cudaFree(h->epot_partials);
      h->Fpart = h->epot_partials = nullptr;
      const size_t n1 = std::max<size_t>(h->nsplit > 1 ? (size_t)h->nsplit * state_elems(h) : 1, 1);
      const size_t n2 = std::max<size_t>((size_t)h->itiles * h->nsplit * h->B, 1);
      CU(cudaMalloc((void**)&h->Fpart, n1 * sizeof(double)));
      CU(cudaMalloc((void**)&h->epot_partials, n2 * sizeof(double)));
      CU(cudaMemset(h->Fpart, 0, n1 * sizeof(double)));
      CU(cudaMemset(h->epot_partials, 0, n2 * sizeof(double)));
    }
  }
  for (GraphEntry& g : h->graphs) cudaGraphExecDestroy(g.exec);  // captured arguments carried the old pointer
  h->graphs.clear();
  return MDQT_OK;
}

int mdqt_set_traj_seeds(mdqt_handle* h, const uint64_t* seeds) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (!seeds) {
    if (h->seeds) { cudaFree(h->seeds); h->seeds = nullptr; }
  } else {
    if (!h->seeds) CU(cudaMalloc((void**)&h->seeds, sizeof(uint64_t) * (size_t)h->B));
    CU(cudaMemcpy(h->seeds, seeds, sizeof(uint64_t) * (size_t)h->B, cudaMemcpyHostToDevice));
  }
  for (GraphEntry& g : h->graphs) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
  return MDQT_OK;
}

// entry points whose kernels assume one ion count for the whole batch
#define NEED_UNIFORM_N(h) do { if ((h)->nb) return fail(MDQT_ESTATE, "not available with per-trajectory ion counts (mdqt_set_ion_counts)"); } while (0)
// entry points that advance positions more than once per call: on a row-decomposed handle the remote rows of R would be
// stale from the second force evaluation on (one force call per position exchange)
#define NEED_ALL_ROWS(h, what) do { if ((h)->nrows != (h)->N) return fail(MDQT_ESTATE, what ": a row-decomposed handle allows one force evaluation per position exchange (use mdqt_comm_init, or call mdqt_forces / mdqt_substeps and exchange R yourself)"); } while (0)

extern "C++" ForceArgs mdqt_force_args(mdqt_handle* h) {
  ForceArgs a;
  memset(&a, 0, sizeof(a));  // padding included: graph entries are compared bytewise
  a.R = h->R; a.F = h->F; a.Fpart = h->Fpart; a.counters = h->counters;
  a.N = h->N; a.ld = h->ld; a.B = h->B; a.row0 = h->row0; a.nrows = h->nrows;
  a.nsplit = h->nsplit; a.jlen = h->jlen; a.ipt = h->ipt; a.jsub = h->jsub; a.rg = h->rg; a.Rfix = h->Rfix;
  a.items = h->items; a.gcap = (h->nrows + 31) / 32; a.nb = h->nb; a.jl = h->jl; a.pdl = h->pdl; a.ilist = h->ilist; a.icount = h->icount;
  a.mg_chunk = ((1ULL << 40) + h->nsplit - 1) / h->nsplit; a.mg_gcap = ((1ULL << 40) + a.gcap - 1) / a.gcap;
  { const int g2 = (h->nrows + 63) / 64; a.mg_gcap2 = ((1ULL << 40) + g2 - 1) / g2; }
  a.L = h->p.L; a.halfL = h->p.L / 2.; a.invL = 1.0 / h->p.L; a.kappa = h->p.kappa; a.rc2 = h->p.rcut * h->p.rcut;
  a.invL_lo = fma(-a.invL, a.L, 1.0) * a.invL;  // 1/L - fl(1/L), to first order
  a.half_l = (h->p.rcut == h->p.L / 2.) ? 1 : 0;
  {
    const double u = a.L / 18446744073709551616.0;  // L / 2^64
    const double rc_u = sqrt(a.rc2) / u;
    a.inv_u = 1.0 / u;
    a.rc2_u = a.half_l ? 85070591730234615865843651857942052864.0 /* 2^126 = (L/2)^2 */ : rc_u * rc_u;
  }
  return a;
}

// the pair kernels read the fixed-point copy of R: refresh it if R was written from outside the engine's kernels
extern "C++" void mdqt_refresh_fixed(mdqt_handle* h, bool wait_comm) {
  if (wait_comm && h->comm) mdqt_comm_sync_pending(h);  // remote rows of Rfix may still be arriving on the communication stream
  if (!h->rfix_dirty) return;
  const double invL = 1.0 / h->p.L;
  launch_to_fixed(h->R, h->Rfix, state_elems(h), invL, fma(-invL, h->p.L, 1.0) * invL, h->stream);
  h->rfix_dirty = 0;
}

extern "C++" QTArgs mdqt_qt_args(mdqt_handle* h, int nsub, int do_step, int do_kick) {
  QTArgs a;
  memset(&a, 0, sizeof(a));
  const mdqt_params& p = h->p;
  a.R = h->R; a.V = h->V; a.F = h->F; a.psi = h->psi; a.tPart = h->tPart;
  a.Rfix = h->Rfix; a.invL = 1.0 / p.L; a.invL_lo = fma(-a.invL, p.L, 1.0) * a.invL;
  a.forced_u = h->forced_u ? h->forced_u + (size_t)h->forced_cursor * h->N * 5 : nullptr;
  a.N = h->N; a.ld = h->ld; a.B = h->B; a.row0 = h->row0; a.nrows = h->nrows; a.traj0 = p.traj0;
  a.nsub = nsub; a.do_step = do_step; a.do_kick = do_kick; a.do_tpart = do_kick;  // tPart lives where the kick does (SU, TS)
  a.scheme = h->S; a.S = h->S; a.renorm = p.renormalize; a.quad = p.quad;
  a.nb = h->nb; a.seeds = h->seeds;
  a.pdl = h->pdl;
  a.lanes = 0;  // lanes per ion by (N, B): the two- and four-lane kernels give the same bits (tests/test_gpu_variants.py)
  a.t0 = h->t; a.substep0 = h->substep; a.seed = p.seed;
  a.L = p.L; a.dtq = p.dtq;
  a.detuning = p.detuning; a.detuningDP = p.detuningDP; a.Om = p.Om; a.OmDP = p.OmDP; a.dR = p.dR; a.kRat = p.kRat;
  a.vKick = p.vKick; a.vKickDP = p.vKickDP; a.g2E = p.g2E; a.pv2qv = p.pv2qv;
  a.fracOfSig = p.fracOfSig; a.Te = p.Te; a.sig0 = p.sig0; a.density = p.density;
  return a;
}

static cudaEvent_t next_event(mdqt_handle* h) {
  if (h->ev_used == h->ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    h->ev.push_back(e);
  }
  return h->ev[h->ev_used++];
}

extern "C++" int mdqt_enqueue_substeps(mdqt_handle* h, int nsub, int do_step, int do_kick, bool forces_partial) {
  if (h->forced_u && h->forced_cursor + nsub > h->forced_nsub) return fail(MDQT_ESTATE, "forced uniforms exhausted");
  QTArgs a = qt_args(h, nsub, do_step, do_kick);
  if (forces_partial && forces_are_partial(force_args(h))) { a.fpart = h->Fpart; a.Fw = h->F; a.fp_jlen = h->jlen; a.jl = h->jl; }
  launch_substeps(a, h->qc, h->S, h->stream);
  if (h->forced_u) h->forced_cursor += nsub;
  h->substep += (uint64_t)nsub;
  if (do_step || h->S == MDQT_SCHEME_V3)
    for (int s = 0; s < nsub; s++) h->t += h->p.dtq;  // the same repeated addition as SU:716 / the kernel (TS:387)
  return MDQT_OK;
}

int mdqt_forces(mdqt_handle* h) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  refresh_fixed(h);
  launch_forces(force_args(h), h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_substeps(mdqt_handle* h, int nsub) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (h->S != MDQT_SCHEME_SR12) return fail(MDQT_ESTATE, "mdqt_substeps needs the 12-level scheme");
  if (nsub < 0) return fail(MDQT_EINVAL, "nsub < 0");
  if (nsub == 0) return MDQT_OK;
  CU(cudaSetDevice(h->p.device));
  int rc = enqueue_substeps(h, nsub, 1, 1);
  if (rc) return rc;
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_qsteps(mdqt_handle* h, int nsub) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (h->S != MDQT_SCHEME_SR7 && h->S != MDQT_SCHEME_CA5 && h->S != MDQT_SCHEME_V3)
    return fail(MDQT_ESTATE, "mdqt_qsteps needs the 7-, 5- or 3-level scheme");
  NEED_UNIFORM_N(h);
  if (nsub < 0) return fail(MDQT_EINVAL, "nsub < 0");
  if (nsub == 0) return MDQT_OK;
  CU(cudaSetDevice(h->p.device));
  // pump schemes: frozen velocities, no kick (MC408L:754, MC422L:722); 3-level test system: kick, no positions (TS:283)
  int rc = enqueue_substeps(h, nsub, 0, h->S == MDQT_SCHEME_V3 ? 1 : 0);
  if (rc) return rc;
  CU(cudaGetLastError());
  return MDQT_OK;
}

// nsteps MD steps as ONE replayed CUDA graph. Kernel-to-kernel dependencies inside a graph resolve without the ~2 us
// scheduling granularity seen between stream launches on B200 (61.5 -> 57.6 us per MD step at N = 3500). Kernel arguments
// are frozen at capture, so the clock is read from device memory (set by a tiny kernel before each replay, advanced by
// the force kernels inside the graph); a cached graph is reused while the arguments it froze are still current.
static bool graphs_enabled() {
  static const bool on = [] { const char* e = getenv("MDQT_GRAPH"); return !(e && e[0] == '0'); }();
  return on;
}
static int md_steps_graph(mdqt_handle* h, int nsteps) {
  const int ratio = h->p.substeps_per_md;
  refresh_fixed(h);
  ForceArgs fa = force_args(h);
  fa.clock = h->clock; fa.clock_dtq = h->p.dtq; fa.clock_advance = 0;
  QTArgs qa = qt_args(h, ratio, 1, 1);
  qa.clock = h->clock; qa.t0 = 0.0; qa.substep0 = 0;
  if (forces_are_partial(fa)) { qa.fpart = h->Fpart; qa.Fw = h->F; qa.fp_jlen = h->jlen; qa.jl = h->jl; }
  const bool stamp = h->timing == 2;
  if (stamp) {
    const size_t need = (size_t)nsteps * 2;
    if (h->stamps_cap < need) {
      if (h->stamps) cudaFree(h->stamps);
      h->stamps = nullptr; h->stamps_cap = 0;
      CU(cudaMalloc((void**)&h->stamps, need * 2 * sizeof(unsigned long long)));
      h->stamps_cap = need;
    }
    fa.stamp = h->stamps; qa.stamp = h->stamps + 2;  // per-launch slots are set at capture; these key the cached graph
  }
  cudaGraphExec_t exec = nullptr;
  for (GraphEntry& g : h->graphs)
    if (g.nsteps == nsteps && !memcmp(&g.fa, &fa, sizeof(fa)) && !memcmp(&g.qa, &qa, sizeof(qa))) { exec = g.exec; break; }
  if (!exec) {
    cudaGraph_t graph;
    CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    for (int k = 0; k < nsteps; k++) {
      ForceArgs fk = fa;
      fk.clock_advance = k ? ratio : 0;  // the clock is set for step 0 before the replay; step k-1's substeps are added here
      QTArgs qk = qa;
      if (stamp) { fk.stamp = h->stamps + (size_t)4 * k; qk.stamp = h->stamps + (size_t)4 * k + 2; }
      launch_forces(fk, h->stream, false);  // the substep kernel adds the item kernel's partial sums while it loads its ion
      launch_substeps(qk, h->qc, h->S, h->stream);
    }
    cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
    if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph capture: ") + cudaGetErrorString(e));
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph instantiate: ") + cudaGetErrorString(e));
    if (h->graphs.size() >= 4) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
    VVArgs v0;
    memset(&v0, 0, sizeof(v0));
    h->graphs.push_back(GraphEntry{nsteps, exec, fa, qa, v0});
  }
  k_set_clock<<<1, 1, 0, h->stream>>>(h->clock, h->t, (unsigned long long)h->substep, (unsigned long long)h->vv_step);
  if (stamp) k_init_stamps<<<(2 * nsteps + 127) / 128, 128, 0, h->stream>>>(h->stamps, 2 * nsteps);
  CU(cudaGraphLaunch(exec, h->stream));
  for (long long s = 0; s < (long long)nsteps * ratio; s++) h->t += h->p.dtq;  // host mirror: the same repeated addition
  h->substep += (uint64_t)nsteps * ratio;
  CU(cudaGetLastError());
  if (stamp) {  // per-kernel durations and the gaps between them INSIDE the replayed graph
    std::vector<unsigned long long> st((size_t)nsteps * 4);
    CU(cudaMemcpyAsync(st.data(), h->stamps, st.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < 4; k++) { h->time_ms[k] = 0; h->time_n[k] = 0; }
    for (int k = 0; k < nsteps; k++) {
      const unsigned long long f0 = st[4 * k], f1 = st[4 * k + 1], q0 = st[4 * k + 2], q1 = st[4 * k + 3];
      h->time_ms[0] += (double)(f1 - f0) * 1e-6; h->time_n[0]++;
      h->time_ms[1] += (double)(q1 - q0) * 1e-6; h->time_n[1]++;
      h->time_ms[2] += ((double)q0 - (double)f1) * 1e-6; h->time_n[2]++;
      if (k + 1 < nsteps) { h->time_ms[3] += ((double)st[4 * k + 4] - (double)q1) * 1e-6; h->time_n[3]++; }
    }
  }
  return MDQT_OK;
}

int mdqt_md_steps(mdqt_handle* h, int nsteps) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (h->S != MDQT_SCHEME_SR12) return fail(MDQT_ESTATE, "mdqt_md_steps needs the 12-level scheme");
  if (h->p.substeps_per_md < 1) return fail(MDQT_EINVAL, "substeps_per_md < 1");
  CU(cudaSetDevice(h->p.device));
  if (h->comm) {  // row-decomposed run with a communicator: the position all-gather is part of every MD step
    if (h->forced_u) return fail(MDQT_ESTATE, "forced uniforms on a communicating handle");
    int rc = mdqt_comm_md_steps(h, nsteps);
    if (rc) return rc;
    return MDQT_OK;
  }
  if (nsteps > 1) NEED_ALL_ROWS(h, "mdqt_md_steps(n > 1)");
  if (nsteps >= 2 && h->timing != 1 && !h->forced_u && graphs_enabled()) return md_steps_graph(h, nsteps);
  const bool timing = h->timing == 1;
  if (timing) h->ev_used = 0;
  for (int k = 0; k < nsteps; k++) {
    refresh_fixed(h);
    if (timing) CU(cudaEventRecord(next_event(h), h->stream));
    launch_forces(force_args(h), h->stream, false);
    if (timing) { CU(cudaEventRecord(next_event(h), h->stream)); CU(cudaEventRecord(next_event(h), h->stream)); }
    int rc = enqueue_substeps(h, h->p.substeps_per_md, 1, 1, /*forces_partial=*/true);
    if (rc) return rc;
    if (timing) CU(cudaEventRecord(next_event(h), h->stream));
  }
  CU(cudaGetLastError());
  if (timing) {
    CU(cudaStreamSynchronize(h->stream));
    h->time_ms[0] = h->time_ms[1] = 0; h->time_n[0] = h->time_n[1] = 0;
    for (size_t k = 0; k + 3 < h->ev_used; k += 4) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, h->ev[k], h->ev[k + 1]);
      cudaEventElapsedTime(&b, h->ev[k + 2], h->ev[k + 3]);
      h->time_ms[0] += a; h->time_ms[1] += b; h->time_n[0]++; h->time_n[1]++;
    }
  }
  return MDQT_OK;
}

int mdqt_md_steps_host(mdqt_handle* h, int nsteps, double* R, double* V, double* psi, double* tPart, int ld) {
  if (!h || !R || !V || !psi || !tPart) return fail(MDQT_EINVAL, "null argument");
  NEED_ALL_ROWS(h, "mdqt_md_steps_host");
  int rc = mdqt_upload_state(h, R, V, psi, tPart, ld);
  if (rc) return rc;
  rc = mdqt_md_steps(h, nsteps);
  if (rc) return rc;
  return mdqt_download_state(h, R, V, psi, tPart, ld);
}

int mdqt_epot(mdqt_handle* h, double* epot) {
  if (!h || !epot) return fail(MDQT_EINVAL, "null argument");
  CU(cudaSetDevice(h->p.device));
  refresh_fixed(h);
  launch_epot(force_args(h), h->epot_partials, h->scalars + (size_t)h->B * 8, h->stream);
  CU(cudaMemcpyAsync(epot, h->scalars + (size_t)h->B * 8, (size_t)h->B * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  if (h->comm) return mdqt_comm_allreduce(h, epot, 1);  // the own rows' share -> the whole system's energy on every rank
  return MDQT_OK;
}

int mdqt_download_rows(mdqt_handle* h, double* R, double* V, double* psi, double* tPart, int ld) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (ld < h->N) return fail(MDQT_EINVAL, "ld smaller than n_ions");
  if (h->B != 1) return fail(MDQT_ESTATE, "mdqt_download_rows needs n_traj == 1");
  CU(cudaSetDevice(h->p.device));
  const size_t r0 = (size_t)h->row0, nr = (size_t)h->nrows;
  if (R) CU(cudaMemcpy2DAsync(R + r0, (size_t)ld * 8, h->R + r0, (size_t)h->ld * 8, nr * 8, 3, cudaMemcpyDeviceToHost, h->stream));
  if (V) CU(cudaMemcpy2DAsync(V + r0, (size_t)ld * 8, h->V + r0, (size_t)h->ld * 8, nr * 8, 3, cudaMemcpyDeviceToHost, h->stream));
  if (psi) {
    if (!h->S) return fail(MDQT_ESTATE, "handle has no wavefunctions (scheme NONE)");
    launch_transpose_psi_out(h->psi, h->psi_stage, h->S, h->N, h->ld, h->B, h->stream);
    CU(cudaMemcpyAsync(psi + r0 * 2 * h->S, h->psi_stage + r0 * 2 * h->S, nr * 2 * h->S * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  if (tPart) CU(cudaMemcpyAsync(tPart + r0, h->tPart + r0, nr * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_diagnostics(mdqt_handle* h, mdqt_diag* out) {
  if (!h || !out) return fail(MDQT_EINVAL, "null argument");
  if (h->comm) {  // partial sums over the own rows, completed by two small all-reduces: the whole-system values on every rank
    CU(cudaSetDevice(h->p.device));
    double s[5] = {0, 0, 0, 0, 0};
    launch_diag_partial(h->V, h->row0, h->nrows, h->ld, 1, nullptr, h->scalars, h->stream);
    CU(cudaMemcpyAsync(s, h->scalars, 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    int rc = mdqt_comm_allreduce(h, s, 1);
    if (rc) return rc;
    const double mean = s[0] / (double)h->N;
    rc = mdqt_diag_partial(h, &mean, s);
    if (rc) return rc;
    rc = mdqt_comm_allreduce(h, s, 5);
    if (rc) return rc;
    out[0].t = h->t; out[0].vx_avg = mean; out[0].ekin_x = s[1] / (double)h->N; out[0].ekin_y = s[2] / (double)h->N;
    out[0].ekin_z = s[3] / (double)h->N; out[0].epot = s[4];
    return MDQT_OK;
  }
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "row-decomposed handle: use mdqt_diag_partial and all-reduce the sums");
  CU(cudaSetDevice(h->p.device));
  refresh_fixed(h);
  launch_diag(h->V, h->N, h->ld, h->B, h->nb, h->scalars, h->stream);
  launch_epot(force_args(h), h->epot_partials, h->scalars + (size_t)h->B * 8, h->stream);
  std::vector<double> s((size_t)h->B * 16);
  CU(cudaMemcpyAsync(s.data(), h->scalars, s.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  for (int b = 0; b < h->B; b++) {
    out[b].t = h->t; out[b].vx_avg = s[b * 8]; out[b].ekin_x = s[b * 8 + 1]; out[b].ekin_y = s[b * 8 + 2];
    out[b].ekin_z = s[b * 8 + 3]; out[b].epot = s[(size_t)h->B * 8 + b];
  }
  return MDQT_OK;
}

int mdqt_diag_partial(mdqt_handle* h, const double* vx_mean, double* sums) {
  if (!h || !sums) return fail(MDQT_EINVAL, "null argument");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  refresh_fixed(h);
  double* mean_dev = nullptr;
  if (vx_mean) {
    mean_dev = h->scalars + (size_t)h->B * 12;  // scratch behind the [B][8] sums and the [B] potential energies
    CU(cudaMemcpyAsync(mean_dev, vx_mean, (size_t)h->B * 8, cudaMemcpyHostToDevice, h->stream));
  }
  launch_diag_partial(h->V, h->row0, h->nrows, h->ld, h->B, mean_dev, h->scalars, h->stream);
  launch_epot(force_args(h), h->epot_partials, h->scalars + (size_t)h->B * 8, h->stream);  // owned rows x all j, already / N
  std::vector<double> s((size_t)h->B * 9);
  CU(cudaMemcpyAsync(s.data(), h->scalars, s.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  for (int b = 0; b < h->B; b++) {
    for (int k = 0; k < 4; k++) sums[b * 5 + k] = s[b * 8 + k];
    sums[b * 5 + 4] = s[(size_t)h->B * 8 + b];
  }
  return MDQT_OK;
}

int mdqt_vel_dist_partial(mdqt_handle* h, const double* vx_mean, double* pvel) {
  if (!h || !pvel || !vx_mean) return fail(MDQT_EINVAL, "null argument");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  std::vector<double> m((size_t)h->B * 8, 0.0);
  for (int b = 0; b < h->B; b++) m[(size_t)b * 8] = vx_mean[b];
  CU(cudaMemcpyAsync(h->scalars, m.data(), m.size() * 8, cudaMemcpyHostToDevice, h->stream));
  launch_vel_dist_rows(h->V, h->scalars, h->row0, h->nrows, h->ld, h->B, h->pvel, h->stream);
  CU(cudaMemcpyAsync(pvel, h->pvel, (size_t)h->B * 3 * kVelBins * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_vel_dist(mdqt_handle* h, double* pvel) {
  if (!h || !pvel) return fail(MDQT_EINVAL, "null argument");
  if (h->comm) {  // <v_x> over all ranks, the KDE of the own rows about it, then the sum of the bins over the ranks
    CU(cudaSetDevice(h->p.device));
    double s0 = 0;
    launch_diag_partial(h->V, h->row0, h->nrows, h->ld, 1, nullptr, h->scalars, h->stream);
    CU(cudaMemcpyAsync(&s0, h->scalars, 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    int rc = mdqt_comm_allreduce(h, &s0, 1);
    if (rc) return rc;
    const double mean = s0 / (double)h->N;
    rc = mdqt_vel_dist_partial(h, &mean, pvel);
    if (rc) return rc;
    return mdqt_comm_allreduce(h, pvel, 3 * kVelBins);
  }
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "row-decomposed handle: use mdqt_vel_dist_partial and all-reduce the bins");
  CU(cudaSetDevice(h->p.device));
  launch_diag(h->V, h->N, h->ld, h->B, h->nb, h->scalars, h->stream);
  launch_vel_dist(h->V, h->scalars, h->N, h->ld, h->B, h->nb, h->pvel, h->stream);
  CU(cudaMemcpyAsync(pvel, h->pvel, (size_t)h->B * 3 * kVelBins * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_populations(mdqt_handle* h, double* pops) {
  if (!h || !pops) return fail(MDQT_EINVAL, "null argument");
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_populations: a row-decomposed handle holds the wavefunctions of its own rows only (use mdqt_populations_rows)");
  if (!h->S) return fail(MDQT_ESTATE, "handle has no wavefunctions (scheme NONE)");
  CU(cudaSetDevice(h->p.device));
  launch_populations(h->psi, h->S, h->N, h->ld, h->B, h->pops, h->stream);
  CU(cudaMemcpyAsync(pops, h->pops, (size_t)h->B * h->N * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_populations_rows(mdqt_handle* h, double* pops) {
  if (!h || !pops) return fail(MDQT_EINVAL, "null argument");
  if (!h->S) return fail(MDQT_ESTATE, "handle has no wavefunctions (scheme NONE)");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  launch_populations(h->psi, h->S, h->N, h->ld, h->B, h->pops, h->stream);  // rows outside the block hold stale amplitudes: not copied
  CU(cudaMemcpy2DAsync(pops, (size_t)h->nrows * 24, h->pops + (size_t)h->row0 * 3, (size_t)h->N * 24, (size_t)h->nrows * 24, h->B,
                       cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

// nsteps x { qsteps x qstep(); MDStep() } as ONE replayed CUDA graph (see md_steps_graph): the MD-family loops
// MD:1081-1083 / 1107-1165 (qsteps = 0) and the pump stage MC408L:1227-1232 (qsteps = plasmaToQuantumTimestepRatio).
int mdqt_vv_steps(mdqt_handle* h, int nsteps, int qsteps, double dt, double collisionFreq, double sigma_v, int laser,
                  double laser_coeff) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!(dt > 0) || nsteps < 0 || qsteps < 0) return fail(MDQT_EINVAL, "dt must be > 0, nsteps and qsteps >= 0");
  if (qsteps > 0 && h->S != MDQT_SCHEME_SR7 && h->S != MDQT_SCHEME_CA5) return fail(MDQT_ESTATE, "pump sweeps need the 7- or 5-level scheme");
  NEED_UNIFORM_N(h);
  NEED_ALL_ROWS(h, "mdqt_vv_steps");
  CU(cudaSetDevice(h->p.device));
  const bool graph = nsteps >= 2 && h->timing != 1 && !h->forced_u && !h->forced_cu && graphs_enabled();
  if (!graph) {
    for (int k = 0; k < nsteps; k++) {
      if (qsteps > 0) { int rc = mdqt_qsteps(h, qsteps); if (rc) return rc; }
      int rc = mdqt_vv_step(h, dt, collisionFreq, sigma_v, laser, laser_coeff);
      if (rc) return rc;
    }
    return MDQT_OK;
  }
  refresh_fixed(h);
  ForceArgs fa = force_args(h);  // F / oldF alternate inside the graph: the entry is keyed on the pointers of step 0
  QTArgs qa = qt_args(h, qsteps, 0, 0);
  qa.clock = h->clock; qa.t0 = 0.0; qa.substep0 = 0;
  VVArgs va;
  memset(&va, 0, sizeof(va));
  va.R = h->R; va.V = h->V; va.A = h->F; va.oldA = h->oldF;
  va.N = h->N; va.ld = h->ld; va.B = h->B; va.row0 = h->row0; va.nrows = h->nrows; va.traj0 = h->p.traj0;
  va.L = h->p.L; va.dt = dt; va.collisionFreq = collisionFreq; va.sigma_v = sigma_v; va.laser_coeff = laser_coeff; va.laser = laser;
  va.seed = h->p.seed; va.Rfix = h->Rfix; va.invL = 1.0 / h->p.L; va.invL_lo = fma(-va.invL, h->p.L, 1.0) * va.invL;
  va.clock = h->clock; va.adv_sub = qsteps;
  cudaGraphExec_t exec = nullptr;
  for (GraphEntry& g : h->graphs)
    if (g.nsteps == -nsteps && !memcmp(&g.fa, &fa, sizeof(fa)) && !memcmp(&g.qa, &qa, sizeof(qa)) && !memcmp(&g.va, &va, sizeof(va))) { exec = g.exec; break; }
  if (!exec) {
    cudaGraph_t gr;
    CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    double *F = h->F, *oldF = h->oldF;
    for (int k = 0; k < nsteps; k++) {
      if (qsteps > 0) launch_substeps(qa, h->qc, h->S, h->stream);     // qstep() sweeps (MC408L:1228-1230)
      std::swap(F, oldF);                                              // oldA = A (MD:505-506)
      VVArgs vk = va;
      vk.A = oldF; vk.oldA = oldF; vk.adv_vv = k ? 1 : 0;
      launch_vv_positions(vk, h->stream);                              // stepPositions (MD:507); advances the counters
      ForceArgs fk = fa;
      fk.F = F;
      launch_forces(fk, h->stream);                                    // calculateAccelerations (MD:508)
      vk.A = F;
      launch_vv_velocities(vk, h->stream);                             // stepVelocities (MD:509)
    }
    cudaError_t e = cudaStreamEndCapture(h->stream, &gr);
    if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph capture: ") + cudaGetErrorString(e));
    e = cudaGraphInstantiate(&exec, gr, 0);
    cudaGraphDestroy(gr);
    if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph instantiate: ") + cudaGetErrorString(e));
    if (h->graphs.size() >= 4) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
    h->graphs.push_back(GraphEntry{-nsteps, exec, fa, qa, va});  // negative key: MD-family graphs
  }
  k_set_clock<<<1, 1, 0, h->stream>>>(h->clock, h->t, (unsigned long long)h->substep, (unsigned long long)h->vv_step);
  CU(cudaGraphLaunch(exec, h->stream));
  if (nsteps & 1) std::swap(h->F, h->oldF);
  h->substep += (uint64_t)nsteps * qsteps;
  h->vv_step += (uint64_t)nsteps;
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_vv_step(mdqt_handle* h, double dt, double collisionFreq, double sigma_v, int laser, double laser_coeff) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!(dt > 0)) return fail(MDQT_EINVAL, "dt must be > 0");
  NEED_UNIFORM_N(h);
  NEED_ALL_ROWS(h, "mdqt_vv_step");
  CU(cudaSetDevice(h->p.device));
  std::swap(h->F, h->oldF);  // oldA = A (MD:505-506)
  VVArgs a;
  memset(&a, 0, sizeof(a));
  a.R = h->R; a.V = h->V; a.A = h->oldF; a.oldA = h->oldF;
  a.N = h->N; a.ld = h->ld; a.B = h->B; a.row0 = h->row0; a.nrows = h->nrows; a.traj0 = h->p.traj0;
  a.L = h->p.L; a.dt = dt; a.collisionFreq = collisionFreq; a.sigma_v = sigma_v; a.laser_coeff = laser_coeff; a.laser = laser;
  a.step = h->vv_step; a.seed = h->p.seed; a.forced_u = h->forced_cu; a.forced_n = h->forced_cn;
  a.Rfix = h->Rfix; a.invL = 1.0 / h->p.L; a.invL_lo = fma(-a.invL, h->p.L, 1.0) * a.invL;
  refresh_fixed(h);
  launch_vv_positions(a, h->stream);    // stepPositions (MD:507)
  launch_forces(force_args(h), h->stream);  // calculateAccelerations (MD:508)
  a.A = h->F;
  launch_vv_velocities(a, h->stream);   // stepVelocities (MD:509)
  h->vv_step++;
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_leapfrog_step(mdqt_handle* h, double dt) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!(dt > 0)) return fail(MDQT_EINVAL, "dt must be > 0");
  NEED_UNIFORM_N(h);
  NEED_ALL_ROWS(h, "mdqt_leapfrog_step");
  CU(cudaSetDevice(h->p.device));
  LFArgs a;
  a.R = h->R; a.V = h->V; a.F = h->F; a.Rfix = h->Rfix;
  a.invL = 1.0 / h->p.L; a.invL_lo = fma(-a.invL, h->p.L, 1.0) * a.invL; a.L = h->p.L;
  a.N = h->N; a.ld = h->ld; a.B = h->B; a.row0 = h->row0; a.nrows = h->nrows;
  a.DT = 0.5 * dt; a.DTV = dt;
  const int first = !(h->t > 0);  // FZ408L:321: the 2nd-order start recomputes forces() inside step_R
  refresh_fixed(h);
  if (first) {
    launch_forces(force_args(h), h->stream);
    a.first = 1; a.kick = 0; a.drift = 1; launch_lf(a, h->stream);   // step_R(0.5 dt)
    launch_forces(force_args(h), h->stream);
    a.first = 0; a.kick = 1; a.drift = 0; launch_lf(a, h->stream);   // step_V(dt)
    launch_forces(force_args(h), h->stream);
    a.first = 1; a.kick = 0; a.drift = 1; launch_lf(a, h->stream);   // step_R(0.5 dt)
  } else {
    a.first = 0; a.kick = 0; a.drift = 1; launch_lf(a, h->stream);   // step_R(0.5 dt)
    launch_forces(force_args(h), h->stream);                         // step_V(dt): forces(); V += dt F
    a.kick = 1; launch_lf(a, h->stream);                             //   ... fused with the second step_R(0.5 dt)
  }
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_advance_time(mdqt_handle* h, int nsub) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  for (int s = 0; s < nsub; s++) h->t += h->p.dtq;  // FZ408L:1066: t += quantumTimestep outside the pump window
  return MDQT_OK;
}

int mdqt_tag_particles(mdqt_handle* h, int32_t* tagged, int32_t* n_tagged) {
  if (!h || !n_tagged) return fail(MDQT_EINVAL, "null argument");
  if (h->S != MDQT_SCHEME_SR7 && h->S != MDQT_SCHEME_CA5) return fail(MDQT_ESTATE, "tagging needs the 7- or 5-level scheme");
  NEED_UNIFORM_N(h);
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_tag_particles: a row-decomposed handle holds the wavefunctions of its own rows only");
  CU(cudaSetDevice(h->p.device));
  const size_t n = (size_t)h->B * h->N;
  if (!h->tagged) CU(cudaMalloc((void**)&h->tagged, sizeof(int) * (n + h->B)));
  launch_tag(h->psi, h->S, h->N, h->ld, h->B, h->p.traj0, h->p.seed, h->substep, h->forced_tag, h->tagged, h->tagged + n, h->stream);
  if (tagged) CU(cudaMemcpyAsync(tagged, h->tagged, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(n_tagged, h->tagged + n, sizeof(int) * h->B, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_set_forced_tag_uniforms(mdqt_handle* h, const double* u) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (h->forced_tag) { cudaFree(h->forced_tag); h->forced_tag = nullptr; }
  if (!u) return MDQT_OK;
  if (h->B != 1) return fail(MDQT_ESTATE, "forced uniforms need n_traj == 1");
  CU(cudaMalloc((void**)&h->forced_tag, (size_t)h->N * 16));
  CU(cudaMemcpy(h->forced_tag, u, (size_t)h->N * 16, cudaMemcpyHostToDevice));
  return MDQT_OK;
}

static int vaf_impl(mdqt_handle* h, int start, double* vaf, int squares) {
  if (!h || !vaf) return fail(MDQT_EINVAL, "null argument");
  NEED_UNIFORM_N(h);
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_vaf: a row-decomposed handle holds the velocities of its own rows only");
  CU(cudaSetDevice(h->p.device));
  if (!h->vhold) {
    if (!start) return fail(MDQT_ESTATE, "mdqt_vaf: no interval started");
    CU(cudaMalloc((void**)&h->vhold, (size_t)h->B * h->ld * 8));
  }
  if (start)  // Vholder[j] = V[0][j] (FZ408L:949-954)
    CU(cudaMemcpy2DAsync(h->vhold, (size_t)h->ld * 8, h->V, (size_t)3 * h->ld * 8, (size_t)h->ld * 8, h->B, cudaMemcpyDeviceToDevice, h->stream));
  launch_vaf(h->V, h->vhold, h->N, h->ld, h->B, h->scalars, h->stream, squares);
  CU(cudaMemcpyAsync(vaf, h->scalars, (size_t)h->B * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_vaf(mdqt_handle* h, int start, double* vaf) { return vaf_impl(h, start, vaf, 0); }
int mdqt_vsq_autocorr(mdqt_handle* h, int start, double* out) { return vaf_impl(h, start, out, 1); }

int mdqt_pair_correlation(mdqt_handle* h, double step, double rmax, int nbins, double* g, uint64_t* counts) {
  if (!h || (!g && !counts)) return fail(MDQT_EINVAL, "null argument");
  if (!(step > 0) || nbins != (int)(rmax / step) || nbins < 1 || nbins > gr_max_bins())
    return fail(MDQT_EINVAL, "nbins must equal (int)(rmax/step) and lie in [1, 2048]");
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "pair correlation needs a handle that owns all rows");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  if (!h->gr_counts) CU(cudaMalloc((void**)&h->gr_counts, sizeof(unsigned long long) * (size_t)h->B * gr_max_bins()));
  launch_gr(h->R, h->N, h->ld, h->B, h->p.L, step, nbins, h->gr_counts, h->stream);
  std::vector<unsigned long long> c((size_t)h->B * nbins);
  CU(cudaMemcpyAsync(c.data(), h->gr_counts, c.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  const int N = h->N;
  for (int b = 0; b < h->B; b++)
    for (int i = 0; i < nbins; i++) {
      const double cnt = (double)c[(size_t)b * nbins + i];
      if (counts) counts[(size_t)b * nbins + i] = c[(size_t)b * nbins + i];
      // the reference's normalisation, integer sub-expressions included (MD:627-635)
      if (g) g[(size_t)b * nbins + i] = (i == 0) ? cnt / (N * 4 / 3 * M_PI * step * step * step)
                                                  : cnt / (N * 3 * step * step * step * i * i);
    }
  return MDQT_OK;
}

int mdqt_vstore_begin(mdqt_handle* h, int T) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (T < 1 || T > 5000) return fail(MDQT_EINVAL, "T must lie in [1, 5000]");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  for (double** ptr : {&h->vstore, &h->ac_partials, &h->ac_out}) if (*ptr) { cudaFree(*ptr); *ptr = nullptr; }
  const size_t n = (size_t)h->B * 3 * h->N * T;
  CU(cudaMalloc((void**)&h->vstore, n * 8));
  CU(cudaMemsetAsync(h->vstore, 0, n * 8, h->stream));
  CU(cudaMalloc((void**)&h->ac_partials, (size_t)h->B * autocorr_chunks(3 * h->N) * 4 * T * 8));
  CU(cudaMalloc((void**)&h->ac_out, (size_t)h->B * 4 * T * 8));
  h->vstore_T = T;
  return MDQT_OK;
}

int mdqt_vstore_record(mdqt_handle* h, int tS) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!h->vstore) return fail(MDQT_ESTATE, "mdqt_vstore_begin not called");
  if (tS < 0 || tS >= h->vstore_T) return fail(MDQT_EINVAL, "time slot outside [0,T)");
  CU(cudaSetDevice(h->p.device));
  launch_vstore_record(h->V, h->vstore, h->N, h->ld, h->B, h->vstore_T, tS, h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_vstore_upload(mdqt_handle* h, const double* v) {
  if (!h || !v) return fail(MDQT_EINVAL, "null argument");
  if (!h->vstore) return fail(MDQT_ESTATE, "mdqt_vstore_begin not called");
  CU(cudaSetDevice(h->p.device));
  CU(cudaMemcpy(h->vstore, v, (size_t)h->B * 3 * h->N * h->vstore_T * 8, cudaMemcpyHostToDevice));
  return MDQT_OK;
}

int mdqt_autocorrelations(mdqt_handle* h, double Gamma, double* vaf, double* longvisc, double* vcube, double* vfourth) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!h->vstore) return fail(MDQT_ESTATE, "mdqt_vstore_begin not called");
  if (!(Gamma > 0)) return fail(MDQT_EINVAL, "Gamma must be > 0");
  CU(cudaSetDevice(h->p.device));
  const int T = h->vstore_T;
  // subtracted constants as the reference writes them (MD:710, 785)
  launch_autocorr(h->vstore, h->N, h->B, T, 3 / (Gamma * Gamma), 3 * 9 / (Gamma * Gamma * Gamma * Gamma), h->ac_partials,
                  h->ac_out, h->stream);
  std::vector<double> o((size_t)h->B * 4 * T);
  CU(cudaMemcpyAsync(o.data(), h->ac_out, o.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  double* dst[4] = {vaf, longvisc, vcube, vfourth};
  for (int b = 0; b < h->B; b++)
    for (int p = 0; p < 4; p++)
      if (dst[p]) memcpy(dst[p] + (size_t)b * T, o.data() + ((size_t)b * 4 + p) * T, (size_t)T * 8);
  return MDQT_OK;
}

int mdqt_set_tags(mdqt_handle* h, const uint8_t* tags) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (!tags) { if (h->tags) { cudaFree(h->tags); h->tags = nullptr; } return MDQT_OK; }
  const size_t n = (size_t)h->B * h->N;
  if (!h->tags) CU(cudaMalloc((void**)&h->tags, n));
  CU(cudaMemcpy(h->tags, tags, n, cudaMemcpyHostToDevice));
  return MDQT_OK;
}

int mdqt_moments_begin(mdqt_handle* h, int nslots) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (nslots < 1 || nslots > (1 << 22)) return fail(MDQT_EINVAL, "nslots outside [1, 2^22]");
  NEED_UNIFORM_N(h);
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_moments: a row-decomposed handle holds the velocities of its own rows only");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (h->moments) { cudaFree(h->moments); h->moments = nullptr; }
  CU(cudaMalloc((void**)&h->moments, sizeof(double) * (size_t)nslots * h->B * kMomentsPerRecord));
  CU(cudaMemsetAsync(h->moments, 0, sizeof(double) * (size_t)nslots * h->B * kMomentsPerRecord, h->stream));
  h->moments_slots = nslots;
  return MDQT_OK;
}

int mdqt_moments_record(mdqt_handle* h, int slot) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!h->moments) return fail(MDQT_ESTATE, "mdqt_moments_begin not called");
  if (slot < 0 || slot >= h->moments_slots) return fail(MDQT_EINVAL, "slot outside [0, nslots)");
  CU(cudaSetDevice(h->p.device));
  launch_moments(h->V, h->tags, h->N, h->ld, h->B, h->moments + (size_t)slot * h->B * kMomentsPerRecord, h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_moments_download(mdqt_handle* h, double* out, int nslots) {
  if (!h || !out) return fail(MDQT_EINVAL, "null argument");
  if (!h->moments) return fail(MDQT_ESTATE, "mdqt_moments_begin not called");
  if (nslots < 1 || nslots > h->moments_slots) return fail(MDQT_EINVAL, "nslots outside [1, slots recorded]");
  CU(cudaSetDevice(h->p.device));
  CU(cudaMemcpyAsync(out, h->moments, sizeof(double) * (size_t)nslots * h->B * kMomentsPerRecord, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

// ---- pressure tensor (virial stress) recorder ----
static int stress_handle_ok(mdqt_handle* h) {
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_stress: a row-decomposed handle holds the forces of its own rows only");
  if (h->comm) return fail(MDQT_ESTATE, "mdqt_stress: not available on a handle with a communicator (mdqt_comm_init)");
  return MDQT_OK;
}
// the pair pass writes one 6-vector per item slot / CTA; mdqt_set_ion_counts may re-plan the chunks after mdqt_stress_begin
static int stress_partials_fit(mdqt_handle* h) {
  const size_t need = (size_t)std::max(1, stress_partials_needed(force_args(h)));
  if (h->stress_partials && h->stress_partials_cap >= need) return MDQT_OK;
  CU(cudaStreamSynchronize(h->stream));
  if (h->stress_partials) { cudaFree(h->stress_partials); h->stress_partials = nullptr; h->stress_partials_cap = 0; }
  CU(cudaMalloc((void**)&h->stress_partials, need * sizeof(double)));
  h->stress_partials_cap = need;
  return MDQT_OK;
}

int mdqt_stress_begin(mdqt_handle* h, int nslots) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (nslots < 1 || nslots > (1 << 22)) return fail(MDQT_EINVAL, "nslots outside [1, 2^22]");
  if (int rc = stress_handle_ok(h)) return rc;
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  for (double** ptr : {&h->stress, &h->stress_series, &h->stress_ac_partials, &h->stress_ac_out}) if (*ptr) { cudaFree(*ptr); *ptr = nullptr; }
  h->stress_slots = 0;
  const size_t n = (size_t)h->B * kStressPerRecord * nslots;
  CU(cudaMalloc((void**)&h->stress, n * sizeof(double)));
  CU(cudaMemsetAsync(h->stress, 0, n * sizeof(double), h->stream));
  const int T = std::min(nslots, stress_autocorr_max_T());
  CU(cudaMalloc((void**)&h->stress_series, (size_t)h->B * 3 * T * sizeof(double)));
  CU(cudaMalloc((void**)&h->stress_ac_partials, (size_t)h->B * 4 * T * sizeof(double)));
  CU(cudaMalloc((void**)&h->stress_ac_out, (size_t)h->B * 4 * T * sizeof(double)));
  if (int rc = stress_partials_fit(h)) return rc;
  h->stress_slots = nslots; h->stress_ac_cap = T;
  return MDQT_OK;
}

int mdqt_stress_record(mdqt_handle* h, int slot) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!h->stress) return fail(MDQT_ESTATE, "mdqt_stress_begin not called");
  if (slot < 0 || slot >= h->stress_slots) return fail(MDQT_EINVAL, "slot outside [0, nslots)");
  if (int rc = stress_handle_ok(h)) return rc;
  CU(cudaSetDevice(h->p.device));
  if (int rc = stress_partials_fit(h)) return rc;
  refresh_fixed(h);
  launch_stress(force_args(h), h->stress_partials, h->V, h->stress, h->stress_slots, slot, h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_stress_download(mdqt_handle* h, double* out, int nslots) {
  if (!h || !out) return fail(MDQT_EINVAL, "null argument");
  if (!h->stress) return fail(MDQT_ESTATE, "mdqt_stress_begin not called");
  if (nslots < 1 || nslots > h->stress_slots) return fail(MDQT_EINVAL, "nslots outside [1, slots recorded]");
  CU(cudaSetDevice(h->p.device));
  // [B][12][stress_slots] on the device -> [B][12][nslots] on the host
  CU(cudaMemcpy2DAsync(out, (size_t)nslots * 8, h->stress, (size_t)h->stress_slots * 8, (size_t)nslots * 8, (size_t)h->B * kStressPerRecord,
                       cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_stress_autocorr(mdqt_handle* h, int nslots, double* acf) {
  if (!h || !acf) return fail(MDQT_EINVAL, "null argument");
  if (!h->stress) return fail(MDQT_ESTATE, "mdqt_stress_begin not called");
  if (nslots < 1 || nslots > h->stress_slots) return fail(MDQT_EINVAL, "nslots outside [1, slots recorded]");
  if (nslots > h->stress_ac_cap) return fail(MDQT_EINVAL, "nslots above the correlator's limit of " + std::to_string(stress_autocorr_max_T()) + " records");
  CU(cudaSetDevice(h->p.device));
  const int T = nslots;
  launch_stress_autocorr(h->stress, h->stress_slots, h->B, T, h->stress_series, h->stress_ac_partials, h->stress_ac_out, h->stream);
  CU(cudaMemcpy2DAsync(acf, (size_t)T * 8, h->stress_ac_out, (size_t)4 * T * 8, (size_t)T * 8, h->B, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

// ---- heat (energy) current recorder ----
static int heat_handle_ok(mdqt_handle* h) {
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_heat: a row-decomposed handle holds the sums of its own rows only");
  if (h->comm) return fail(MDQT_ESTATE, "mdqt_heat: not available on a handle with a communicator (mdqt_comm_init)");
  return MDQT_OK;
}
// the pair pass writes one 8-vector per item slot / CTA; mdqt_set_ion_counts may re-plan the chunks after mdqt_heat_begin
static int heat_partials_fit(mdqt_handle* h) {
  const size_t need = (size_t)std::max(1, heat_partials_needed(force_args(h)));
  if (h->heat_partials && h->heat_partials_cap >= need) return MDQT_OK;
  CU(cudaStreamSynchronize(h->stream));
  if (h->heat_partials) { cudaFree(h->heat_partials); h->heat_partials = nullptr; h->heat_partials_cap = 0; }
  CU(cudaMalloc((void**)&h->heat_partials, need * sizeof(double)));
  h->heat_partials_cap = need;
  return MDQT_OK;
}

int mdqt_heat_begin(mdqt_handle* h, int nslots) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (nslots < 1 || nslots > (1 << 22)) return fail(MDQT_EINVAL, "nslots outside [1, 2^22]");
  if (int rc = heat_handle_ok(h)) return rc;
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  for (double** ptr : {&h->heat, &h->heat_series, &h->heat_ac_partials, &h->heat_ac_out}) if (*ptr) { cudaFree(*ptr); *ptr = nullptr; }
  h->heat_slots = 0;
  const size_t n = (size_t)h->B * kHeatPerRecord * nslots;
  CU(cudaMalloc((void**)&h->heat, n * sizeof(double)));
  CU(cudaMemsetAsync(h->heat, 0, n * sizeof(double), h->stream));
  const int T = std::min(nslots, stress_autocorr_max_T());  // the same correlator as the shear stress
  CU(cudaMalloc((void**)&h->heat_series, (size_t)h->B * 3 * T * sizeof(double)));
  CU(cudaMalloc((void**)&h->heat_ac_partials, (size_t)h->B * 4 * T * sizeof(double)));
  CU(cudaMalloc((void**)&h->heat_ac_out, (size_t)h->B * 4 * T * sizeof(double)));
  if (int rc = heat_partials_fit(h)) return rc;
  h->heat_slots = nslots; h->heat_ac_cap = T;
  return MDQT_OK;
}

int mdqt_heat_record(mdqt_handle* h, int slot) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (!h->heat) return fail(MDQT_ESTATE, "mdqt_heat_begin not called");
  if (slot < 0 || slot >= h->heat_slots) return fail(MDQT_EINVAL, "slot outside [0, nslots)");
  if (int rc = heat_handle_ok(h)) return rc;
  CU(cudaSetDevice(h->p.device));
  if (int rc = heat_partials_fit(h)) return rc;
  refresh_fixed(h);
  launch_heat(force_args(h), h->heat_partials, h->V, h->heat, h->heat_slots, slot, h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_heat_download(mdqt_handle* h, double* out, int nslots) {
  if (!h || !out) return fail(MDQT_EINVAL, "null argument");
  if (!h->heat) return fail(MDQT_ESTATE, "mdqt_heat_begin not called");
  if (nslots < 1 || nslots > h->heat_slots) return fail(MDQT_EINVAL, "nslots outside [1, slots recorded]");
  CU(cudaSetDevice(h->p.device));
  // [B][15][heat_slots] on the device -> [B][15][nslots] on the host
  CU(cudaMemcpy2DAsync(out, (size_t)nslots * 8, h->heat, (size_t)h->heat_slots * 8, (size_t)nslots * 8, (size_t)h->B * kHeatPerRecord,
                       cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_heat_autocorr(mdqt_handle* h, int nslots, double* acf) {
  if (!h || !acf) return fail(MDQT_EINVAL, "null argument");
  if (!h->heat) return fail(MDQT_ESTATE, "mdqt_heat_begin not called");
  if (nslots < 1 || nslots > h->heat_slots) return fail(MDQT_EINVAL, "nslots outside [1, slots recorded]");
  if (nslots > h->heat_ac_cap) return fail(MDQT_EINVAL, "nslots above the correlator's limit of " + std::to_string(stress_autocorr_max_T()) + " records");
  CU(cudaSetDevice(h->p.device));
  const int T = nslots;
  launch_heat_autocorr(h->heat, h->heat_slots, h->B, T, h->N, h->nb, h->heat_series, h->heat_ac_partials, h->heat_ac_out, h->stream);
  CU(cudaMemcpy2DAsync(acf, (size_t)T * 8, h->heat_ac_out, (size_t)4 * T * 8, (size_t)T * 8, h->B, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_vel_dist_tagged(mdqt_handle* h, double* pv) {
  if (!h || !pv) return fail(MDQT_EINVAL, "null argument");
  if (!h->tags) return fail(MDQT_ESTATE, "mdqt_set_tags not called");
  NEED_UNIFORM_N(h);
  if (h->nrows != h->N) return fail(MDQT_ESTATE, "mdqt_vel_dist_tagged: a row-decomposed handle holds the velocities of its own rows only");
  CU(cudaSetDevice(h->p.device));
  if ((size_t)h->B * kTagBins > (size_t)h->B * 3 * kVelBins) return fail(MDQT_ESTATE, "internal: pvel scratch too small");
  launch_vel_dist_tagged(h->V, h->tags, h->N, h->ld, h->B, h->pvel, h->stream);  // 4001 <= 3 x 2001 doubles per trajectory
  CU(cudaMemcpyAsync(pv, h->pvel, (size_t)h->B * kTagBins * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_scale_velocities(mdqt_handle* h, double sx, double sy, double sz) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  NEED_UNIFORM_N(h);
  CU(cudaSetDevice(h->p.device));
  launch_scale_velocities(h->V, h->N, h->ld, h->B, sx, sy, sz, h->stream);
  CU(cudaGetLastError());
  return MDQT_OK;
}

int mdqt_set_forced_uniforms(mdqt_handle* h, const double* u, int nsub) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (h->forced_u) { cudaFree(h->forced_u); h->forced_u = nullptr; }
  h->forced_nsub = 0; h->forced_cursor = 0;
  if (!u) return MDQT_OK;
  if (h->B != 1) return fail(MDQT_ESTATE, "forced uniforms need n_traj == 1");
  if (nsub < 1) return fail(MDQT_EINVAL, "nsub < 1");
  size_t n = (size_t)nsub * h->N * 5;
  CU(cudaMalloc((void**)&h->forced_u, n * 8));
  CU(cudaMemcpy(h->forced_u, u, n * 8, cudaMemcpyHostToDevice));
  h->forced_nsub = nsub;
  return MDQT_OK;
}

int mdqt_set_forced_collisions(mdqt_handle* h, const double* u, const double* v) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  CU(cudaSetDevice(h->p.device));
  CU(cudaStreamSynchronize(h->stream));
  if (h->forced_cu) { cudaFree(h->forced_cu); h->forced_cu = nullptr; }
  if (h->forced_cn) { cudaFree(h->forced_cn); h->forced_cn = nullptr; }
  if (!u || !v) return MDQT_OK;
  if (h->B != 1) return fail(MDQT_ESTATE, "forced collisions need n_traj == 1");
  CU(cudaMalloc((void**)&h->forced_cu, (size_t)h->N * 8));
  CU(cudaMalloc((void**)&h->forced_cn, (size_t)h->N * 24));
  CU(cudaMemcpy(h->forced_cu, u, (size_t)h->N * 8, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->forced_cn, v, (size_t)h->N * 24, cudaMemcpyHostToDevice));
  return MDQT_OK;
}

// host replica of the device stream (same integer arithmetic): lets callers feed the oracle the very uniforms
// the kernel consumes
static void philox_host(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
static double u52_host(uint32_t hi, uint32_t lo) {
  uint64_t k = ((uint64_t)hi << 20) | (uint64_t)(lo >> 12);
  return ((double)k + 0.5) * 2.220446049250313080847263336181640625e-16;
}
int mdqt_philox_uniforms(uint64_t seed, uint32_t traj, uint32_t ion, uint64_t substep, double u[5]) {
  if (!u) return fail(MDQT_EINVAL, "null argument");
  for (uint32_t call = 0; call < 3; call++) {
    uint32_t c[4] = {(uint32_t)substep, (uint32_t)(substep >> 32), ion, (traj << 3) | call};
    philox_host(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    u[2 * call] = u52_host(c[0], c[1]);
    if (call < 2) u[2 * call + 1] = u52_host(c[2], c[3]);
  }
  return MDQT_OK;
}

void* mdqt_device_ptr(mdqt_handle* h, int which) {
  if (!h) return nullptr;
  return which == 0 ? (void*)h->R : which == 1 ? (void*)h->V : which == 2 ? (void*)h->F : nullptr;
}
int mdqt_device_ld(mdqt_handle* h) { return h ? h->ld : 0; }
void* mdqt_stream(mdqt_handle* h) { return h ? (void*)h->stream : nullptr; }

int mdqt_mark_wrapped(mdqt_handle* h, int wrapped) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  (void)wrapped;  // kept for ABI stability: the fixed-point pair kernel is exact for wrapped and unwrapped coordinates alike
  h->rfix_dirty = 1;
  return MDQT_OK;
}

int mdqt_force_plan(mdqt_handle* h, int* nsplit, int* jlen) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  if (nsplit) *nsplit = h->nsplit;
  if (jlen) *jlen = h->jlen;
  return MDQT_OK;
}

int mdqt_enable_timing(mdqt_handle* h, int on) {
  if (!h) return fail(MDQT_EINVAL, "null handle");
  h->timing = (on == 2) ? 2 : (on != 0);
  return MDQT_OK;
}
int mdqt_kernel_time_ms(mdqt_handle* h, int which, double* ms_per_launch, int* launches) {
  if (!h || which < 0 || which > 3) return fail(MDQT_EINVAL, "bad argument");
  if (ms_per_launch) *ms_per_launch = h->time_n[which] ? h->time_ms[which] / h->time_n[which] : 0.0;
  if (launches) *launches = h->time_n[which];
  return MDQT_OK;
}

int mdqt_time_forces(mdqt_handle* h, int reps, double* ms_per_launch) {
  if (!h || !ms_per_launch || reps < 1) return fail(MDQT_EINVAL, "bad argument");
  CU(cudaSetDevice(h->p.device));
  refresh_fixed(h);
  cudaGraph_t graph;
  cudaGraphExec_t exec = nullptr;
  CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  ForceArgs fa = force_args(h);
  fa.pdl = 0;  // plain stream order: with programmatic dependent launch successive force launches would overlap, and this is a kernel time
  for (int k = 0; k < reps; k++) launch_forces(fa, h->stream, false);  // the force kernel alone
  cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
  if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph capture: ") + cudaGetErrorString(e));
  e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("graph instantiate: ") + cudaGetErrorString(e));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaGraphLaunch(exec, h->stream);  // warm-up replay
  cudaEventRecord(e0, h->stream);
  cudaGraphLaunch(exec, h->stream);
  cudaEventRecord(e1, h->stream);
  e = cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaGraphExecDestroy(exec);
  if (e != cudaSuccess) return fail(MDQT_ECUDA, std::string("mdqt_time_forces: ") + cudaGetErrorString(e));
  *ms_per_launch = (double)ms / reps;
  return MDQT_OK;
}

int mdqt_fp64_peak(mdqt_handle* h, double* tflops) {
  if (!h || !tflops) return fail(MDQT_EINVAL, "null argument");
  CU(cudaSetDevice(h->p.device));
  double v = run_fp64_peak(h->stream);
  if (v <= 0) return fail(MDQT_ECUDA, "fp64 peak probe failed");
  *tflops = v;
  return MDQT_OK;
}

}  // extern "C"
