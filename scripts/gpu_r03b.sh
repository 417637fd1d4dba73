#!/bin/bash
# r03b: weighted graphs on the GPU (DESIGN.md K3, "per-row alias tables on the device") at C3
# (R-MAT 10 M / 200 M with log-normal weights): weighted ingest, the load split by
# B2E_LOAD_TIMING (device edge alias build, longest row), the host oracle's sequential Vose loop
# on the same graph and the bitwise comparison with it, weighted second-order walk steps/s; the
# GPU model and power limit of the same run.
# Usage: scripts/gpu_r03b.sh [output directory, default r03b_out]
out="${1:-r03b_out}"
mkdir -p "$out"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm --format=csv > "$out/r03b_gpus.txt"
cat "$out/r03b_gpus.txt"
B2E_LOAD_TIMING=1 timeout 540 python scripts/weighted_graphs.py --shape c3 --out "$out/r03b_weighted_c3.json" \
  2> "$out/r03b_weighted_c3_stderr.txt"
echo "c3 rc=$?"
