#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native MDQT hot path (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            our arm   (one process per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU implementation of the path
    python bench.py ... --dump-outputs DIR                   also write the timed path's outputs of its last step to DIR/*.npy

Workload (BASELINE.json configs[1]): the MDQT laser-cooling thesis run, N0 = 3500 ions, detuning = -1,
detuningDP = +1, Om = OmDP = 1, density = 2, Ge = 0.1 -- synthetic random-start ions and random S-manifold
wavefunctions of that shape.  One bench "step" = one sampling interval of the reference's main loop (sampleFreq =
40 MD steps, SU:78) = 40 x { forces(); 25 x { step(); qstep(); } } = 1000 quantum substeps of every ion.

metric  = ion-steps/s  (one ion advanced by one quantum substep, forces included), whole job over all GPUs.
value   : state resident in HBM, device time (CUDA events on the engine's stream, max over ranks).
e2e     : the same through the C-ABI host call mdqt_md_steps_host: pinned host buffers in, host buffers out, every step.
roofline: dominant kernel = the all-pairs Yukawa force kernel (FP64-pipe bound; neither HBM nor tensor bound) --
          34 flop per ordered pair x N^2 pairs per launch / mean launch duration, against the FP64 DFMA peak measured
          live on this GPU by the engine's own probe kernel.
With N > 1 every rank advances its own trajectory of the ensemble (the SLURM --array replacement): weak scaling, no
collective on the data path.  The row-decomposed large-N path (NCCL all-gather of positions once per MD step) is
timed as the extra "large_n" block.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

MD_PER_STEP = 40          # sampleFreq (SU:78)
DUMP_LIMIT_BYTES = 60 << 20  # --dump-outputs writes at most this much over all ranks (+ .npy headers): < 64 MB however MB is counted
FLOP_PER_PAIR = 34        # SURVEY.md section 8(d)
BYTES_PER_ION_STEP = 520  # SURVEY.md section 8(d)
FLOP_PER_ION_STEP = 1700  # SURVEY.md section 8(d): ~1.7 kflop per no-jump 12-level ion-step (sparse H, 4 stages)
FP64_NOMINAL_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12  # 148 SMs x 64 FP64 lanes x 2 flop x 1.965 GHz = 37.2 (B200 nominal)
N0 = 3500


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, "/tmp/mdqt_clocks_%d_%d.csv" % (os.getpid(), index)

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()  # the exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        clocks, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clocks.append(float(parts[0])); mx = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if clocks:
            # the samples under load are the upper half (the first ones may precede the timed work)
            out.update(sm_mhz=float(np.median(sorted(clocks)[len(clocks) // 2:])), sm_max_mhz=mx, reasons=sorted(reasons),
                       samples=len(clocks))
        return out


def synthetic_state(n, L, job, n_traj=1):
    from mdqtplasmasims_b200 import synthetic
    R = np.stack([synthetic.random_positions(n, L, seed=12345 + job + b) for b in range(n_traj)])
    psi = np.stack([synthetic.random_s_state(n, 12, seed=12345 + job + b) for b in range(n_traj)])
    V = np.zeros((n_traj, 3, n))
    tp = np.zeros((n_traj, n))
    if n_traj == 1:
        return R[0], V[0], psi[0], tp[0]
    return R, V, psi, tp


def dump_outputs(out_dir, eng, suffix="", limit=DUMP_LIMIT_BYTES):
    """What a caller of the timed path receives after its last step -- the state R, V, psi, tPart, t and the forces F of the
    last MD step -- as float64 DIR/<name><suffix>.npy. Above `limit` bytes in all, the same seeded sample of ions is kept in
    every run, so that two builds can still be compared array for array."""
    s = eng.download()
    arrays = {"R": s["R"], "V": s["V"], "psi": s["psi"], "tPart": s["tPart"], "F": eng.download_forces(), "t": np.array(s["t"])}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        keep = np.sort(np.random.default_rng(0).choice(eng.N, eng.N * limit // total, replace=False))
        ion_axis = {"R": -1, "V": -1, "F": -1, "tPart": -1, "psi": -3}
        arrays = {k: np.take(a, keep, axis=ion_axis[k]) if k in ion_axis else a for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + suffix + ".npy"), a)


def pinned_like(torch, a):
    t = torch.empty(a.shape, dtype=torch.float64).pin_memory()
    v = t.numpy()
    v[...] = a
    return t, v


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mdqtplasmasims_b200 import Engine, su_params

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    K, W = args.steps, max(3, args.warmup)
    B = args.traj_per_gpu
    job = rank * B + 1
    p = su_params(n_ions=N0, N0=N0, n_traj=B, traj0=job, seed=12345, device=local)
    eng = Engine(p)
    R, V, psi, tp = synthetic_state(N0, p.L, job, B)
    eng.upload(R=R, V=V, psi=psi, tPart=tp, t=0.0, substep=0)
    stream = torch.cuda.ExternalStream(eng.lib.mdqt_stream(eng.h), device=torch.device("cuda", local))
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")  # > 126 MB L2

    fp64_peak = eng.fp64_peak_tflops()
    hbm_peak, peak_src = load_peaks()

    def one_step():
        eng.md_steps(MD_PER_STEP)

    # ---- resident timing: W warm-up steps (>= 0.5 s so the clocks ramp), then exactly K timed steps --------------------
    t0 = time.perf_counter()
    w = 0
    while w < W or time.perf_counter() - t0 < 0.5:
        one_step(); w += 1
        if w % 8 == 0:
            eng.sync()
    eng.sync()
    # the timed steps start from the seeded inputs however many warm-up steps the clock ramp took: same arguments, same outputs
    eng.upload(R=R, V=V, psi=psi, tPart=tp, t=0.0, substep=0)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.15)
    torch.cuda.synchronize(); barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for k in range(K):
        with torch.cuda.stream(stream):
            flush.fill_(float(k))          # L2 flush between timed iterations (outside the timed intervals)
        starts[k].record(stream)
        one_step()
        ends[k].record(stream)
    eng.sync(); torch.cuda.synchronize(); barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, "" if world == 1 else "_rank%d" % rank, DUMP_LIMIT_BYTES // world)
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    dev_ms = max_over_ranks(dev_ms)
    clocks = sampler.stop() if sampler else None
    ion_steps_per_step = float(N0) * B * 25 * MD_PER_STEP
    value = sum_over_ranks(ion_steps_per_step * K) / (dev_ms * 1e-3)

    # ---- per-kernel durations: second pass over the same K steps with a CUDA-event pair around every launch -------------
    eng.enable_timing(True)
    for k in range(min(K, 8)):
        one_step()
    k1_ms, k1_n = eng.kernel_time_ms(0)
    k2_ms, k2_n = eng.kernel_time_ms(1)
    eng.enable_timing(False)
    k1_pair_ms, k2_pair_ms = k1_ms, k2_ms      # CUDA-event pair around every single stream launch (includes launch latency)
    # the force kernel's average launch duration: CUDA events on the engine's stream around ONE replayed graph of back-to-back
    # launches (no per-launch event / launch-latency overhead) -- this is what `roofline.achieved` uses
    k1_ms = float(np.median([eng.time_forces(40) for _ in range(5)]))
    # inside the production graph: %globaltimer stamps written by the kernels (earliest CTA start .. latest CTA end)
    eng.enable_timing(2)
    one_step()
    g_k1, _ = eng.kernel_time_ms(0); g_k2, _ = eng.kernel_time_ms(1); g_gap12, _ = eng.kernel_time_ms(2); g_gap21, _ = eng.kernel_time_ms(3)
    eng.enable_timing(False)
    k2_ms = g_k2
    pairs_per_launch = float(N0) * N0 * B
    k1_tflops = FLOP_PER_PAIR * pairs_per_launch / (k1_ms * 1e-3) / 1e12
    k2_gbs = BYTES_PER_ION_STEP * (N0 * B * 25) / (k2_ms * 1e-3) / 1e9

    # ---- e2e: the host-buffer C-ABI call, pinned memory, H2D + compute + D2H every step ------------------------------------
    hR_t, hR = pinned_like(torch, R); hV_t, hV = pinned_like(torch, V)
    hP_t, hP = pinned_like(torch, psi); hT_t, hT = pinned_like(torch, tp)
    for _ in range(3):
        eng.md_steps_host(MD_PER_STEP, hR, hV, hP, hT)
    torch.cuda.synchronize(); barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        eng.md_steps_host(MD_PER_STEP, hR, hV, hP, hT)
    torch.cuda.synchronize(); barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = sum_over_ranks(ion_steps_per_step * K) / e2e_s
    io_bytes = int(hR.nbytes + hV.nbytes + hP.nbytes + hT.nbytes)

    extras = {}
    # ---- extra: ensemble throughput mode (config 4 shape: 64 trajectories batched per GPU) -----------------------------------
    if args.ensemble > 1:
        Be = args.ensemble
        # every reference job draws its own N ~ Binomial(729 N0, 1/729) (SU:299-337): unequal ion counts in one handle
        counts = np.random.default_rng(4321 + rank).binomial(729 * N0, 1.0 / 729, size=Be).astype(np.int32)
        cap = int(counts.max())
        pe = su_params(n_ions=cap, N0=N0, n_traj=Be, traj0=1000 + rank * Be, seed=12345, device=local, plan_n=0)
        ee = Engine(pe)
        ee.set_ion_counts(counts)
        ee.set_traj_seeds(np.arange(Be, dtype=np.uint64) + 777 + rank * Be)
        Re, Ve, Pe, Te_ = synthetic_state(cap, pe.L, 1000 + rank * Be, Be)
        ee.upload(R=Re, V=Ve, psi=Pe, tPart=Te_, t=0.0, substep=0)
        ions_e = float(counts.sum())
        pairs_e = float((counts.astype(np.float64) ** 2).sum())
        es = torch.cuda.ExternalStream(ee.lib.mdqt_stream(ee.h), device=torch.device("cuda", local))
        nmd = 4
        ee.md_steps(nmd); ee.md_steps(nmd); ee.sync()
        torch.cuda.synchronize(); barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(es); ee.md_steps(2 * nmd); b_.record(es)
        ee.sync(); torch.cuda.synchronize(); barrier()
        ms = max_over_ranks(a.elapsed_time(b_))
        ee.enable_timing(2)  # per-kernel split of the batched step (stamps inside the replayed graph)
        ee.md_steps(nmd)
        e1_ms, _ = ee.kernel_time_ms(0)
        e2_ms, _ = ee.kernel_time_ms(1)
        ee.enable_timing(False)
        extras["ensemble"] = {"traj_per_gpu": Be, "ion_counts": "N_b ~ Binomial(729*3500, 1/729): min %d, max %d (mdqt_set_ion_counts)" % (counts.min(), cap),
                              "ion_steps_per_s": sum_over_ranks(ions_e * 25 * 2 * nmd) / (ms * 1e-3),
                              "pair_interactions_per_s": sum_over_ranks(pairs_e * 2 * nmd) / (ms * 1e-3),
                              "ms_per_md_step": ms / (2 * nmd),
                              "k_pairs_ms": e1_ms, "k_pairs_fp64_frac": FLOP_PER_PAIR * pairs_e / (e1_ms * 1e-3) / 1e12 / fp64_peak,
                              "k_pairs_fp64_frac_nominal": FLOP_PER_PAIR * pairs_e / (e1_ms * 1e-3) / 1e12 / FP64_NOMINAL_TFLOPS,
                              "k_substeps_ms": e2_ms,
                              "k_substeps_fp64_frac": FLOP_PER_ION_STEP * ions_e * 25 / (e2_ms * 1e-3) / 1e12 / fp64_peak}
        ee.close()

    # ---- extra: large-N row decomposition with an NCCL all-gather of positions per MD step (config 5 shape) -----------------
    for key, n_large in (("large_n", args.large_n), ("large_n_1e6", args.large_n2)):
        if n_large <= 0:
            continue
        from mdqtplasmasims_b200 import sharding, synthetic
        NL = (n_large // world) * world
        row0, rows = sharding.row_block(NL, world, rank)
        pl = su_params(n_ions=NL, N0=NL, row0=row0, n_rows=rows, seed=777, device=local)
        el = Engine(pl)
        Rl = synthetic.random_positions(NL, pl.L, seed=777)
        el.upload(R=Rl, V=np.zeros((3, NL)), psi=synthetic.random_s_state(NL, 12, seed=777), tPart=np.zeros(NL), t=0.0, substep=0)
        ls = torch.cuda.ExternalStream(el.lib.mdqt_stream(el.h), device=torch.device("cuda", local))
        if world > 1:  # the communicator lives in the library: rank 0's NCCL id travels through torch.distributed
            box = [Engine.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            el.comm_init(box[0], rank, world)

        def md_step_large():
            # forces over the own rows x all j; 25 fused substeps of the own rows; with several ranks ONE in-place ncclAllGather of
            # the fixed-point positions on a communication stream, overlapped with the own-row j chunks of the next force call
            el.md_steps(1)

        md_step_large(); el.sync(); torch.cuda.synchronize(); barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nl = 6 if NL <= 400000 else 2  # the short step is timed over more repetitions: rank skew after the barrier is of the order of 1 ms
        a.record(ls)
        for _ in range(nl):
            md_step_large()
        b_.record(ls)
        el.sync(); torch.cuda.synchronize(); barrier()
        ms = max_over_ranks(a.elapsed_time(b_)) / nl
        # output() observables of the run (outside the timed region): one rank computes them directly, several ranks
        # all-reduce their partial sums -- the printed digits must not depend on the number of GPUs
        dd = el.diagnostics()  # several ranks: partial sums over the own rows + two small ncclAllReduce calls inside the library
        obs = {"epot_per_ion": repr(float(dd["epot"])), "ekin_x": repr(float(dd["ekin_x"])),
               "collective": "2 x ncclAllReduce (1 and 5 fp64)" if world > 1 else "none (1 GPU)"}
        extras[key] = {"n_ions": NL, "scaling": "strong", "rows_per_gpu": rows, "ms_per_md_step": ms, "md_steps_timed": nl, "observables": obs,
                       "pair_interactions_per_s": float(NL) * NL / (ms * 1e-3),
                       "ion_steps_per_s": float(NL) * 25 / (ms * 1e-3),
                       "fp64_frac": FLOP_PER_PAIR * float(NL) * NL / (ms * 1e-3) / 1e12 / (fp64_peak * world),
                       "fp64_frac_nominal": FLOP_PER_PAIR * float(NL) * NL / (ms * 1e-3) / 1e12 / (FP64_NOMINAL_TFLOPS * world),
                       "collective": ("one in-place ncclAllGather of a [3][N/G] int64 fixed-point block per rank and MD step, inside the "
                                      "library (mdqt_comm_init), overlapped with the own-row j chunks of the next force call")
                       if world > 1 else "none (1 GPU)"}
        el.close()

    # ---- extra: the MD-family shapes (BASELINE configs[0] and [2]): MDStep at N=4096 and the 7-level pump stage -------------
    if args.md_family and rank == 0:
        from mdqtplasmasims_b200 import SCHEME_NONE, SCHEME_SR7, md_params, synthetic

        def timed(fn, eng_, stream_, reps):
            fn(); eng_.sync()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream_)
            for _ in range(reps):
                fn()
            b_.record(stream_)
            eng_.sync(); torch.cuda.synchronize()
            return a.elapsed_time(b_) / reps

        nm = 4096
        pm = md_params(scheme=SCHEME_NONE, n_ions=nm, kappa=0.5, density=0.4, device=local)
        em = Engine(pm)
        em.upload(R=synthetic.random_positions(nm, pm.L, seed=3), V=synthetic.maxwellian(nm, np.sqrt(1 / 3.), seed=3))
        em.forces()
        sm = torch.cuda.ExternalStream(em.lib.mdqt_stream(em.h), device=torch.device("cuda", local))
        for _ in range(5):
            em.MDSteps(40, dt=0.005, collisionFreq=0.25, sigma_v=np.sqrt(1 / 3.))
        ms = timed(lambda: em.MDSteps(40, dt=0.005, collisionFreq=0.25, sigma_v=np.sqrt(1 / 3.)), em, sm, 10) / 40
        extras["md_only_N4096"] = {"workload": "MDStep(): velocity Verlet + Andersen collisions, kappa=0.5 (MD:66-88, 504-511)",
                                   "ms_per_md_step": ms, "pair_interactions_per_s": float(nm) * nm / (ms * 1e-3)}
        em.close()
        p7 = md_params(scheme=SCHEME_SR7, n_ions=nm, kappa=0.5, density=2.0, device=local)
        e7 = Engine(p7)
        e7.upload(R=synthetic.random_positions(nm, p7.L, seed=4), V=synthetic.maxwellian(nm, np.sqrt(1 / 3.), seed=4),
                  psi=synthetic.random_s_state(nm, 7, seed=4))
        e7.forces()
        s7 = torch.cuda.ExternalStream(e7.lib.mdqt_stream(e7.h), device=torch.device("cuda", local))

        def pump_steps():  # 20 x { for l < plasmaToQuantumTimestepRatio: qstep(); MDStep(k) }  (MC408L:1227-1232)
            e7.MDSteps(20, dt=0.005, qsteps=p7.substeps_per_md)

        for _ in range(3):
            pump_steps()
        ms = timed(pump_steps, e7, s7, 5) / 20
        extras["qt_tagging_408_N4096"] = {"workload": "pump stage: 62 x 7-level qstep() + MDStep() per MD step (MC408L:1227-1232)",
                                          "ms_per_md_step": ms, "ion_steps_per_s": float(nm) * p7.substeps_per_md / (ms * 1e-3)}
        e7.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_block()

    if rank == 0:
        traffic = None
        tp_path = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp_path):
            try:
                traffic = json.load(open(tp_path)).get("k_pairs_dram_bytes_per_launch")
            except Exception:
                traffic = None
        line = {
            "metric": "ion-steps/s (MDQT) & Yukawa pair-interactions/s", "value": value, "unit": "ion-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "warmup_steps_run": w, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "mdqt_thesis_N0_3500 (BASELINE configs[1]): 12-level Sr+ MDQT, detuning=-1, detuningDP=+1, "
                                   "Om=OmDP=1, density=2, Ge=0.1; one trajectory per GPU",
                       "n_ions": N0, "traj_per_gpu": B, "md_steps_per_step": MD_PER_STEP, "substeps_per_md_step": 25,
                       "l2": "flushed between timed steps (256 MB fill); the 1 MB state is L2-resident within a step by nature",
                       "parallelism": "ensemble: one independent trajectory per GPU, no collective" if world > 1 else "1 GPU"},
            "pair_interactions_per_s": value / 25.0 * N0,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "ion-steps/s", "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes,
                    "api": "mdqt_md_steps_host (C ABI), pinned host buffers"},
            "gpu_launches": K * MD_PER_STEP * 2,
            "fp64_tflops_probe": fp64_peak, "fp64_tflops_nominal": FP64_NOMINAL_TFLOPS,
            "in_graph_us": {"k_pairs": g_k1 * 1e3, "k_substeps": g_k2 * 1e3, "gap_pairs_to_substeps": g_gap12 * 1e3,
                            "gap_substeps_to_pairs": g_gap21 * 1e3,
                            "how": "%globaltimer stamps written by the kernels inside the replayed production graph "
                                   "(earliest CTA start to latest CTA end per launch), mean over one bench step"},
            "roofline": {"bound": "fp64", "kernel": "k_pairs_items (all-pairs Yukawa force)", "achieved": k1_tflops, "peak": fp64_peak,
                         "unit": "TFLOP/s", "frac": k1_tflops / fp64_peak, "frac_nominal": k1_tflops / FP64_NOMINAL_TFLOPS,
                         "frac_in_md_graph": FLOP_PER_PAIR * pairs_per_launch / (g_k1 * 1e-3) / 1e12 / fp64_peak,
                         "launch_ms_event_pair_per_stream_launch": k1_pair_ms, "traffic": traffic,
                         "peak_source": "measured live: DFMA-chain probe kernel (mdqt_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
                         "flop_per_pair": FLOP_PER_PAIR, "pairs_per_launch": pairs_per_launch, "launch_ms": k1_ms, "launches_timed": k1_n,
                         "timing": "CUDA-event pair on the engine's stream around one replayed graph of 40 back-to-back launches, median of 5 "
                                   "(launch_ms_event_pair_per_stream_launch = the round-1 method, which adds launch latency to every launch)",
                         "note": "HBM/tensor do not bound this kernel. Per ordered pair the inner loop issues 23 FP64-pipe + ~20.5 other "
                                 "instructions (cuobjdump; exp and rsqrt expand). An FP64 warp instruction holds the sub-partition's issue "
                                 "port 2 cycles on sm_100, so the issue-bound ceiling is 34 flop x 32 lanes / (2*23+20.5 cycles) = 0.51 of "
                                 "the nominal DFMA rate (0.56 of the measured probe); large N reaches 0.51-0.53 of the probe (large_n.fp64_frac). "
                                 "At N=3500 one launch holds only ~24 us of issue work for the whole chip and ~9 us of launch latency, CTA "
                                 "prologue/epilogue and in-SM tail are exposed (per-CTA phase trace in profiles/)"},
            "roofline_substeps": {"bound": "hbm", "kernel": "k_substeps (25 fused step()+qstep())", "achieved": k2_gbs, "peak": hbm_peak,
                                  "unit": "GB/s", "frac": k2_gbs / hbm_peak, "peak_source": peak_src, "launch_ms": k2_ms,
                                  "launch_ms_event_pair_per_stream_launch": k2_pair_ms, "timing": "in-graph %globaltimer stamps",
                                  "flop_per_ion_step": FLOP_PER_ION_STEP,
                                  "fp64_tflops": FLOP_PER_ION_STEP * (N0 * B * 25) / (k2_ms * 1e-3) / 1e12,
                                  "fp64_frac": FLOP_PER_ION_STEP * (N0 * B * 25) / (k2_ms * 1e-3) / 1e12 / fp64_peak,
                                  "note": "effective bandwidth at 520 B per ion-substep; fused, so state crosses HBM once per 25 substeps "
                                          "(actual DRAM traffic: profiles/traffic.json). The kernel is not HBM-bound: one trajectory of 3500 ions is "
                                          "220 warps, one per SM sub-partition, bound by its own in-order instruction stream (fp64_frac at ~1.7 kflop "
                                          "per ion-step); batched trajectories fill the machine (ensemble.k_substeps_fp64_frac)"},
            "cpu_baseline": cpu,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------------------
# the reference's own CPU implementation of the path (oracle/_ref = unmodified reference sources; else the oracle port)
# ------------------------------------------------------------------------------------------------------------------------------
_CPU_CHILD = r"""
import json, os, sys, time
sys.path.insert(0, %(root)r)
import numpy as np
from oracle import pyoracle as po
budget, steps, md_max = float(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
kind = "reference" if po.ref_available("su") else "port"
if kind == "reference":
    ref = po.RefSU()
    N = ref.init(12345)          # the reference's own init(): random frozen start, N ~ Binomial around N0 = 3500
    def forces(): ref.forces()
    def substep(): ref.step(); ref.qstep()
else:
    orc = po.Oracle()
    p, ratio = po.su_params()
    N = 3500
    L = (3500 * 4 * np.pi / 3) ** 0.333333333
    rng = np.random.default_rng(12345)
    st = dict(R=rng.uniform(0, L, (3, N)), V=np.zeros((3, N)), psi=np.zeros((N, 12, 2)), tp=np.zeros(N), t=0.0, F=None)
    st["psi"][:, 0, 0] = 1
    def forces(): st["F"] = orc.forces_su(st["R"], L, 1 / np.sqrt(0.3))
    def substep():
        orc.step_su(st["R"], st["V"], st["F"], L, p.dtq, st["t"]); Vx = st["V"][0].copy()
        st["t"], _ = orc.qstep12(st["psi"], Vx, st["tp"], st["t"], p, rng.uniform(size=(N, 5))); st["V"][0] = Vx
# calibration: one forces() and two substeps -> how many whole MD steps of a 40-step sampling interval fit the budget
t0 = time.perf_counter(); forces(); tf = time.perf_counter() - t0
t0 = time.perf_counter(); substep(); substep(); ts = (time.perf_counter() - t0) / 2
m = int(max(1, min(md_max, budget / max(1, steps) / (tf + 25 * ts))))
res = []
for k in range(steps):
    t0 = time.perf_counter()
    for _ in range(m):
        forces()
        for _ in range(25):
            substep()
    res.append(time.perf_counter() - t0)
print(json.dumps({"kind": kind, "N": int(N), "md_steps_per_step": m, "step_s": res, "forces_s": tf, "substep_s": ts}))
"""


def cpu_reference_run(threads, budget_s, steps, md_max=MD_PER_STEP):
    """Run the reference's CPU path for REAL: `steps` steps of m whole MD steps each (m <= 40 sized to the budget), every MD
    step = forces() + 25 x { step(); qstep(); } (SU:1369-1378). Returns the child's record (wall seconds per step)."""
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, "-c", _CPU_CHILD % {"root": ROOT}, str(budget_s), str(steps), str(md_max)], env=env,
                         capture_output=True, text=True, timeout=900)
    return json.loads(out.stdout.strip().splitlines()[-1])


REF_LABEL = ("unmodified reference sources (oracle/_ref: laserCoolingPlusExpansionMDQTSpeedUp.cpp compiled g++ -std=c++11 -fopenmp -O3) "
             "with the from-scratch Armadillo shim for the 12x12 algebra (real Armadillo is not installable here)")


def cpu_baseline_block(budget_s=18.0):
    """cpu_baseline of our arm's line: the reference on the host cores at OMP_NUM_THREADS = 1 (the only race-free setting,
    SURVEY App. C Q1), 4 (as shipped, slurm:7) and all cores; each a bounded sample of whole MD steps."""
    ncpu = os.cpu_count() or 1
    by = {}
    kind, N = "unavailable", None
    for thr, share in ((1, 0.45), (4, 0.25), (ncpu, 0.30)):
        if str(thr) in by:
            continue
        try:
            d = cpu_reference_run(thr, budget_s * share, steps=1)
        except Exception as e:  # pragma: no cover
            by[str(thr)] = {"value": None, "error": repr(e)}
            continue
        kind, N = d["kind"], d["N"]
        t = d["step_s"][0]
        by[str(thr)] = {"value": d["N"] * 25.0 * d["md_steps_per_step"] / t, "md_steps_run": d["md_steps_per_step"], "wall_s": t,
                        "forces_s": d["forces_s"], "substep_s": d["substep_s"],
                        "pair_interactions_per_s_ordered_equiv": d["N"] * (d["N"] - 1.0) / d["forces_s"]}
    allv = by.get(str(ncpu), {})
    return {"value": allv.get("value"), "unit": "ion-steps/s", "cores": ncpu if kind == "reference" else 1, "kind": kind,
            "sample": "N=%s; whole MD steps (forces() + 25 x {step(); qstep();}) run for real, %s MD step(s) at all %d threads; %s; "
                      "multi-thread values are 'as shipped': the OpenMP force loop races (SURVEY App. C Q1), 1 thread is the correct one"
                      % (N, allv.get("md_steps_run"), ncpu, REF_LABEL if kind == "reference" else "oracle restatement (scalar C), 1 thread"),
            "by_threads": by}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm; the others exit 0 without work
    threads = os.cpu_count() or 1
    K, W = args.steps, max(1, min(args.warmup, 3))
    # every step is m whole MD steps run for real (m <= 40, sized so that the K + W steps end within ~2.5 minutes); the line
    # reports what was run: ms_per_step is the measured wall time of a step of m MD steps, value = N x 25 x m / that
    t0 = time.perf_counter()
    try:
        d = cpu_reference_run(threads, budget_s=float(os.environ.get("MDQT_REF_BUDGET_S", "150")), steps=K + W)
    except Exception as e:  # pragma: no cover
        print(json.dumps({"impl": "reference", "unavailable": "CPU reference run failed: %r" % (e,)}), flush=True)
        return
    wall = time.perf_counter() - t0
    m, N = d["md_steps_per_step"], d["N"]
    timed = d["step_s"][W:]
    step_s = float(np.mean(timed))
    value = N * 25.0 * m * len(timed) / float(np.sum(timed))
    cpu = {"value": value, "unit": "ion-steps/s", "cores": threads if d["kind"] == "reference" else 1, "kind": d["kind"],
           "sample": "N=%d; %d timed steps of %d whole MD steps each (of the 40 of a sampling interval), every MD step = forces() + 25 x "
                     "{step(); qstep();} run for real; %s; OMP_NUM_THREADS=%d as shipped -- its OpenMP force loop races (SURVEY App. C Q1)"
                     % (N, len(timed), m, REF_LABEL if d["kind"] == "reference" else "oracle restatement (scalar C), 1 thread", threads)}
    line = {"impl": "reference", "metric": "ion-steps/s (MDQT) & Yukawa pair-interactions/s", "value": value, "unit": "ion-steps/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": step_s * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "mdqt_thesis_N0_3500 (BASELINE configs[1]): 12-level Sr+ MDQT, detuning=-1, detuningDP=+1, "
                                   "Om=OmDP=1, density=2, Ge=0.1; one trajectory per GPU",
                       "n_ions": N, "md_steps_per_step": m, "substeps_per_md_step": 25, "host_threads": threads,
                       "note": "the reference's forces()/step()/qstep() on the host CPU; a step is %d of the 40 MD steps of a sampling "
                               "interval when the host is too slow for all 40 within the run budget" % m},
            "cpu_baseline": cpu, "wall_s": wall,
            "e2e": {"value": value, "unit": "ion-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--traj-per-gpu", type=int, default=1)
    ap.add_argument("--ensemble", type=int, default=64, help="extra pass: trajectories batched per GPU (0/1 = skip)")
    ap.add_argument("--large-n", type=int, default=200000, help="extra pass: row-decomposed large-N MD step (0 = skip)")
    ap.add_argument("--large-n2", type=int, default=1000000, help="second large-N pass: BASELINE configs[4], N = 10^6 (0 = skip)")
    ap.add_argument("--no-md-family", dest="md_family", action="store_false", help="skip the MD-only / 7-level pump extras")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state and forces after the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none to write")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
