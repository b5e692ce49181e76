#!/bin/bash
# NeighborhoodHash measurement (tools/bench_nh.py): device pass with stage times, end-to-end fit_transform, the
# reference's pairs/s on a prefix; card name and power limit are read in the same run.
#   bash tools/run_r04_nh.sh [output directory, default profiles]  ->  <dir>/r04_nh_bench.json
cd "$(dirname "$0")/.."
OUT=${1:-profiles}
mkdir -p "$OUT"
timeout 1200 python tools/bench_nh.py --out "$OUT/r04_nh_bench.json" 2> "$OUT/r04_nh_bench.err"
echo "bench_nh rc=$?"
