#!/bin/bash
# r02d: CBOW ring v2 + address math (C4, C3), bit-exact SGD tests,
# traffic captures (C3, C4), then the headline shape (C5) on our arm with the pinned-buffer fix
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_sgns.py tests/test_gpu_fuzz.py tests/test_golden.py tests/test_gpu_exchange.py -m gpu -q --maxfail=8 > gpurun_out/r02d_pytest_gpu.txt 2>&1
echo "pytest rc=$?"; tail -5 gpurun_out/r02d_pytest_gpu.txt
timeout 900 python bench.py --config C4 --steps 5 --warmup 3 --no-cpu-baseline --no-e2e > gpurun_out/r02d_bench_c4.json 2> gpurun_out/r02d_bench_c4.err
timeout 900 python bench.py --config C3 --steps 5 --warmup 3 --no-cpu-baseline --no-e2e > gpurun_out/r02d_bench_c3.json 2> gpurun_out/r02d_bench_c3.err
timeout 900 python bench.py --config C2 --steps 5 --warmup 3 --no-cpu-baseline --no-e2e > gpurun_out/r02d_bench_c2.json 2> gpurun_out/r02d_bench_c2.err
bash scripts/prof_train.sh r02d_c4 C4
bash scripts/prof_train.sh r02d_c3 C3
bash scripts/prof_walk.sh r02d_c3 C3
for t in prof_train_r02d_c4 prof_train_r02d_c3 prof_walk_r02d_c3; do python profiles/summarize.py gpurun_out/$t.ncu-rep > gpurun_out/$t.txt 2>&1; done
python - <<'PY'
import json
for f in ("r02d_bench_c4", "r02d_bench_c3", "r02d_bench_c2"):
    try:
        d = json.load(open(f"gpurun_out/{f}.json"))
        print(f, "value %.4g" % d["value"], "frac %.3f" % d["roofline"]["frac"], "walk %.4g steps/s %.2f ms" % (d["walk"]["steps_per_s_alone"], d["walk"]["avg_launch_ms"]), "loss", d["mean_pair_loss"])
    except Exception as e:
        print(f, "failed", e)
PY
grep -E "duration|dram__bytes_(read|write).sum  |inst_executed.sum|issue_active|warps_active|registers" gpurun_out/prof_train_r02d_c4.txt gpurun_out/prof_train_r02d_c3.txt
free -g | head -2
( time timeout 1800 python bench.py --steps 5 --warmup 2 > gpurun_out/r02d_bench_c5.json 2> gpurun_out/r02d_bench_c5.err ) 2> gpurun_out/r02d_bench_c5.time
echo "ours rc=$?"; tail -3 gpurun_out/r02d_bench_c5.time; tail -3 gpurun_out/r02d_bench_c5.err; head -c 5000 gpurun_out/r02d_bench_c5.json; echo
free -g | head -2
