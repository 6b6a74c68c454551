#!/bin/bash
# kNN + plan tests, then the headline bench
set -u
mkdir -p gpurun_out
python -c "import __graft_entry__ as g; g.build()" > gpurun_out/build.log 2>&1; echo "build rc=$?"
timeout 900 python -m pytest tests/test_gpu_knn.py tests/test_gpu_plan.py tests/test_umap_small_data_golden.py -m gpu -q -x 2>&1 | tail -25 > gpurun_out/pytest_knn.log; echo "knn rc=${PIPESTATUS[0]}"
tail -25 gpurun_out/pytest_knn.log
timeout 600 python bench.py --steps 20 --warmup 3 --no-cpu-baseline > gpurun_out/bench.log 2> gpurun_out/bench.err; echo "bench rc=$?"
python - <<PY
import json
try:
    d=json.loads(open("gpurun_out/bench.log").read().strip().split("\n")[-1])
    print(round(d["value"]), "contigs/s", round(d["ms_per_step"],3), "ms", d["stage_ms"], "K4 TF", round(d["roofline"]["achieved"],1), "K1 GB/s", round(d["roofline_count"]["achieved"],1), "e2e", d.get("e2e"), d.get("neighbors15"), d.get("error"), d.get("traceback"))
except Exception as e:
    print("failed", e); print(open("gpurun_out/bench.err").read()[-2500:])
PY
