#!/bin/bash
# r02c: tests, CBOW ring (C4), ncu of both kernels, then the
# headline shape (C5) on both arms
mkdir -p gpurun_out
timeout 1500 python -m pytest tests -m gpu -q --maxfail=8 > gpurun_out/r02c_pytest_gpu.txt 2>&1
echo "pytest rc=$?" | tee -a gpurun_out/r02c_pytest_gpu.txt
tail -25 gpurun_out/r02c_pytest_gpu.txt
timeout 600 python -m pytest tests/test_quality.py -m gpu -q -s 2>&1 | grep -E "AUROC|oracle|passed|failed" > gpurun_out/r02c_quality.txt
cat gpurun_out/r02c_quality.txt
timeout 900 python bench.py --config C4 --steps 5 --warmup 3 --no-cpu-baseline > gpurun_out/r02c_bench_c4.json 2> gpurun_out/r02c_bench_c4.err
echo "C4 rc=$?"; tail -2 gpurun_out/r02c_bench_c4.err
bash scripts/prof_walk.sh r02c_c3 C3
bash scripts/prof_train.sh r02c_c4 C4
python profiles/summarize.py gpurun_out/prof_walk_r02c_c3.ncu-rep > gpurun_out/r02c_walk_kernel_c3.txt 2>&1
python profiles/summarize.py gpurun_out/prof_train_r02c_c4.ncu-rep > gpurun_out/r02c_cbow_pipe_kernel_c4.txt 2>&1
python - <<'PY'
import json
for f in ("r02c_bench_c4",):
    try:
        d = json.load(open(f"gpurun_out/{f}.json"))
        print(f, "value %.4g" % d["value"], "frac %.3f" % d["roofline"]["frac"], "walk %.4g steps/s %.2f ms" % (d["walk"]["steps_per_s_alone"], d["walk"]["avg_launch_ms"]), "e2e", (d.get("e2e") or {}).get("value"), "loss", d["mean_pair_loss"])
    except Exception as e:
        print(f, "failed", e)
PY
# ---- the headline shape, both arms, as the driver will run them (fewer steps) ----
free -g | head -2
( time timeout 1200 python bench.py --impl reference --steps 5 --warmup 2 > gpurun_out/r02c_ref_c5.json 2> gpurun_out/r02c_ref_c5.err ) 2> gpurun_out/r02c_ref_c5.time
echo "ref rc=$?"; cat gpurun_out/r02c_ref_c5.time | tail -3; tail -2 gpurun_out/r02c_ref_c5.err; cat gpurun_out/r02c_ref_c5.json | head -c 1500; echo
free -g | head -2
( time timeout 1500 python bench.py --steps 5 --warmup 2 > gpurun_out/r02c_bench_c5.json 2> gpurun_out/r02c_bench_c5.err ) 2> gpurun_out/r02c_bench_c5.time
echo "ours rc=$?"; cat gpurun_out/r02c_bench_c5.time | tail -3; tail -3 gpurun_out/r02c_bench_c5.err; cat gpurun_out/r02c_bench_c5.json | head -c 4000; echo
free -g | head -2
