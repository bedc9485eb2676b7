// mdqt_handle.h -- the handle behind the C ABI (include/mdqt.h) and the helpers shared by the translation units that
// implement it (mdqt_capi.cu: single-GPU entry points; mdqt_comm.cu: the row-decomposed multi-GPU path over NCCL).
#pragma once
#include "../../include/mdqt.h"
#include "mdqt_internal.h"
#include "mdqt_qtconsts.h"
#include <string>
#include <vector>

int mdqt_fail(int code, const std::string& msg);
#define CU(call)                                                                                             \
  do {                                                                                                       \
    cudaError_t e_ = (call);                                                                                 \
    if (e_ != cudaSuccess)                                                                                   \
      return mdqt_fail(MDQT_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                      \
  } while (0)

// one instantiated CUDA graph of `nsteps` MD steps, valid while the kernel arguments it froze are still the handle's
struct GraphEntry { int nsteps; cudaGraphExec_t exec; mdqt::ForceArgs fa; mdqt::QTArgs qa; mdqt::VVArgs va; };
struct mdqt_comm;  // mdqt_comm.cu

struct mdqt_handle {
  mdqt_params p;
  int N, B, S, ld, row0, nrows;
  cudaStream_t stream;
  double *R, *V, *F, *oldF, *psi, *tPart, *Fpart, *psi_stage, *epot_partials, *scalars, *pvel, *pops, *vhold, *forced_tag;
  int* tagged;      // [B][N] spin tags + [B] counts (allocated on first use)
  unsigned long long* gr_counts;  // [B][gr_max_bins]
  double *vstore, *ac_partials, *ac_out; int vstore_T;  // vStore[B][3][N][T] and autocorrelation scratch
  unsigned* counters;
  long long* Rfix;  // periodic fixed-point copy of R (what the pair kernels read)
  int rfix_dirty;   // R was written by an upload / externally: refresh Rfix before the next pair kernel
  double* forced_u; int forced_nsub, forced_cursor;
  double *forced_cu, *forced_cn;
  mdqt::QTConsts qc;
  double t; uint64_t substep, vv_step;
  int nsplit, jlen, itiles, ipt, jsub, rg, items;
  int pdl;  // programmatic dependent launch between the force and substep kernels (plan_force)
  int* nb;              // [B] per-trajectory ion counts on the device (ensembles with unequal N) or null
  std::vector<int> nb_host;
  unsigned* ilist; int icount;  // compact item list of an unequal-N batch (ForceArgs.ilist) or null
  int* jl;              // [B] per-trajectory chunk length of the item force kernel (set with nb when plan_n == 0) or null
  uint64_t* seeds;      // [B] per-trajectory Philox keys or null
  int timing;  // 0 off; 1 = CUDA-event pair around every stream launch; 2 = %globaltimer stamps inside the replayed graph
  unsigned long long* stamps; size_t stamps_cap;  // [launch]{min start, max end} ns
  std::vector<cudaEvent_t> ev;  // [force_start, force_end, sub_start, sub_end] per MD step when timing
  size_t ev_used;
  double time_ms[4]; int time_n[4];  // force kernel, substep kernel, gap force->substep, gap substep->force
  double* clock;                    // device {t, substep index}: the simulation clock inside replayed graphs
  std::vector<GraphEntry> graphs;   // small cache keyed by nsteps
  unsigned char* tags;              // [B][N] four tag bits per ion (MD-family tagged-particle recorders) or null
  double* moments; int moments_slots;  // [slots][B][23] recorded sums (mdqt_moments_begin / _record / _download)
  // pressure-tensor recorder (mdqt_stress_begin / _record / _download / _autocorr): the log [B][12][stress_slots], the pair pass's
  // partial 6-vectors, and the correlator's scratch (series [B][3][T], partials [B][4][T], output [B][4][T] for T <= stress_ac_cap)
  double *stress, *stress_partials, *stress_series, *stress_ac_partials, *stress_ac_out;
  int stress_slots, stress_ac_cap; size_t stress_partials_cap;
  // heat-current recorder (mdqt_heat_*): the same layout with the log [B][15][heat_slots] and partial 8-vectors
  double *heat, *heat_partials, *heat_series, *heat_ac_partials, *heat_ac_out;
  int heat_slots, heat_ac_cap; size_t heat_partials_cap;
  mdqt_comm* comm;                  // row-decomposed runs: NCCL communicator and exchange buffers (mdqt_comm_init), or null
};

mdqt::ForceArgs mdqt_force_args(mdqt_handle* h);
mdqt::QTArgs mdqt_qt_args(mdqt_handle* h, int nsub, int do_step, int do_kick);
void mdqt_refresh_fixed(mdqt_handle* h, bool wait_comm = true);
int mdqt_enqueue_substeps(mdqt_handle* h, int nsub, int do_step, int do_kick, bool forces_partial = false);
// mdqt_comm.cu
int mdqt_comm_md_steps(mdqt_handle* h, int nsteps);
void mdqt_comm_release(mdqt_handle* h);
int mdqt_comm_rank_world(const mdqt_handle* h, int* rank, int* world);  // 0 when the handle has no communicator
int mdqt_comm_sync_pending(mdqt_handle* h);  // make the handle's stream wait for an exchange still in flight
extern "C" int mdqt_comm_allreduce(mdqt_handle* h, double* values, int n);
