#!/bin/bash
# A/B of the pair-once force tiles against a library built from the parent commit (developer aid).
# Usage: scripts/ab_pair_once.sh PARENT_LIB OUT_DIR -- runs bench.py alternately with PARENT_LIB and the tree's library (twice each),
# dumps both after 1 and 20 bench steps, and compares the first forces after upload at N = 3500.
set -u
PARENT=$1; OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/card.txt"
B="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline"
for r in 1 2; do
  MDQT_LIB_PATH=$PARENT $B > "$OUT/bench_parent_$r.json" 2> "$OUT/bench_parent_$r.err"; echo "parent $r: $(tail -c 300 $OUT/bench_parent_$r.json)"
  $B > "$OUT/bench_new_$r.json" 2> "$OUT/bench_new_$r.err"; echo "new $r: $(tail -c 300 $OUT/bench_new_$r.json)"
done
for s in 1 20; do
  MDQT_LIB_PATH=$PARENT python bench.py --gpus 1 --steps $s --warmup 0 --no-cpu-baseline --ensemble 0 --large-n 0 --large-n2 0 --no-md-family --dump-outputs "$OUT/dump_parent_$s" > /dev/null 2>&1
  python bench.py --gpus 1 --steps $s --warmup 0 --no-cpu-baseline --ensemble 0 --large-n 0 --large-n2 0 --no-md-family --dump-outputs "$OUT/dump_new_$s" > /dev/null 2>&1
done
MDQT_LIB_PATH=$PARENT python scripts/first_forces.py "$OUT/F_parent.npy"
python scripts/first_forces.py "$OUT/F_new.npy"
python scripts/first_forces.py --compare "$OUT"
