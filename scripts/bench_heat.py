"""Cost of the heat-current record against the force kernel, and of `mdqt_run --program md --heat 1` (developer aid).

For each (N, B): the time of one mdqt_heat_record (host clock around `reps` back-to-back records ending in mdqt_sync, after a
warm-up) beside mdqt_time_forces of the same handle (CUDA events around a replayed graph of force launches), and their ratio.
Then the wall time of the md program at its defaults, without and with --heat 1 (alternated, --runs each).
Writes one JSON document (stdout, or --out) with the card's name, power limit and maximum SM clock read in the same run.
Usage: python scripts/bench_heat.py [--out file.json] [--runs 2] [--shapes "4096x1,3500x1,3500x64,20000x1,100000x1"]"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from mdqtplasmasims_b200 import Engine, SCHEME_NONE, load_library, md_params  # noqa: E402

DRIVER = os.path.join(ROOT, "mdqtplasmasims_b200", "mdqt_run")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except FileNotFoundError:
        raise SystemExit("bench_heat: no GPU (nvidia-smi not found)")
    if q.returncode != 0 or not q.stdout.strip():
        raise SystemExit("bench_heat: no GPU (nvidia-smi: %s)" % (q.stderr.strip() or "no output"))
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def time_shape(N, B, min_seconds=0.5):
    p = md_params(scheme=SCHEME_NONE, n_ions=N, n_traj=B)
    rng = np.random.default_rng(N + B)
    lead = (B,) if B > 1 else ()
    e = Engine(p)
    e.upload(R=rng.uniform(0, p.L, size=lead + (3, N)), V=rng.normal(size=lead + (3, N)) * 0.6)
    force_ms = min(e.time_forces(reps=20) for _ in range(3))
    # records: warm-up, then enough back-to-back records for min_seconds
    e.heat_begin(1)
    e.heat_record(0)
    e.sync()
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < 0.1:
        e.heat_record(0)
        n += 1
    e.sync()
    per = (time.perf_counter() - t0) / n
    reps = max(10, int(min_seconds / per))
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        for _ in range(reps):
            e.heat_record(0)
        e.sync()
        dt = (time.perf_counter() - t0) / reps
        best = dt if best is None else min(best, dt)
    nsplit, jlen = e.force_plan()
    e.close()
    rec_ms = best * 1e3
    return {"N": N, "B": B, "plan": {"nsplit": nsplit, "jlen": jlen}, "heat_record_ms": rec_ms, "time_forces_ms": force_ms,
            "ratio": rec_ms / force_ms, "record_ordered_pairs_per_s": float(N) * N * B / best, "record_reps": reps}


def time_program(heat, save):
    cmd = [DRIVER, "--program", "md", "1", "--seed", "1", "--saveDirectory", save + "/"] + (["--heat", "1"] if heat else [])
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        raise SystemExit("mdqt_run failed: %s" % r.stderr[-2000:])
    m = re.search(r"MD steps in ([0-9.]+) s", r.stderr)
    return {"heat": int(heat), "process_wall_s": wall, "program_wall_s": float(m.group(1)) if m else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--shapes", default="4096x1,3500x1,3500x64,20000x1,100000x1")
    args = ap.parse_args()
    info = gpu_info()
    if load_library().mdqt_device_count() < 1:
        raise SystemExit("bench_heat: no CUDA device")
    shapes = []
    for s in args.shapes.split(","):
        N, B = (int(x) for x in s.split("x"))
        shapes.append(time_shape(N, B))
        print("N=%6d B=%3d  record %.4f ms  forces %.4f ms  ratio %.3f" % (N, B, shapes[-1]["heat_record_ms"],
              shapes[-1]["time_forces_ms"], shapes[-1]["ratio"]), file=sys.stderr, flush=True)
    programs = []
    with tempfile.TemporaryDirectory() as tmp:
        for k in range(args.runs):
            for heat in (0, 1):
                programs.append(time_program(heat, os.path.join(tmp, "r%d_%d" % (k, heat))))
                print("md program --heat %d: %.3f s (in-program %.3f s)" % (heat, programs[-1]["process_wall_s"],
                      programs[-1]["program_wall_s"] or -1), file=sys.stderr, flush=True)
    doc = {"gpu": info, "shapes": shapes, "md_program_defaults": programs,
           "max_ratio": max(s["ratio"] for s in shapes),
           "method": "heat_record_ms: host clock around back-to-back mdqt_heat_record calls ending in mdqt_sync (best of 3); "
                     "time_forces_ms: mdqt_time_forces (CUDA events around a replayed graph of 20 force launches, best of 3)"}
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
