#!/bin/bash
# r03a: GloVe with the centre ids sharded over the GPUs (DESIGN.md K7) at the reference's GloVe
# defaults, on R-MAT 1 M / 16 M and on C3 (R-MAT 10 M / 200 M): seconds per epoch and the phase
# split on 1 GPU and on every GPU of the machine; the GPU model and power limit of the same run.
# Usage: scripts/gpu_r03a.sh [output directory, default r03a_out]
out="${1:-r03a_out}"
mkdir -p "$out"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm --format=csv > "$out/r03a_gpus.txt"
cat "$out/r03a_gpus.txt"
count=$(python -c "import torch; print(torch.cuda.device_count())")
worlds="1"
if [ "$count" -gt 1 ]; then worlds="1 $count"; fi
for graph in rmat1m c3; do
  for world in $worlds; do
    timeout 1200 python scripts/glove_sharded_scaling.py --graph $graph --world $world --epochs 2 \
      --out "$out/r03a_glove_sharded_${graph}_${world}gpu.json" 2> "$out/r03a_glove_sharded_${graph}_${world}gpu.err"
    echo "$graph world=$world rc=$?"
  done
done
