#!/bin/bash
# Reverse mode of the wrench, single-GPU validation: build + smoke(), the new GPU tests, the
# throughput probe (tools/wrench_vjp_probe.py), bench.py, then the whole GPU suite.
#   bash tools/gpu_wrench_vjp.sh <out-dir>
set -u
mkdir -p "${1:?usage: bash tools/gpu_wrench_vjp.sh <out-dir>}"
OUT=$(cd "$1" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem,driver_version --format=csv > "$OUT/gpu.csv"
cat "$OUT/gpu.csv"

python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.log" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/smoke.log"

python -m pytest -q -rs tests/test_gpu_wrench_grad.py -s > "$OUT/pytest_wrench_grad.log" 2>&1
echo "new tests rc=$?"
tail -5 "$OUT/pytest_wrench_grad.log"

python tools/wrench_vjp_probe.py --log "$OUT/wrench_vjp_probe.log" > /dev/null 2> "$OUT/probe.err"
echo "probe rc=$?"
cat "$OUT/wrench_vjp_probe.log"

python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"
echo "bench rc=$?"
tail -c 600 "$OUT/bench.json"; echo

python -m pytest -m gpu -q -rs tests > "$OUT/pytest_gpu.log" 2>&1
echo "pytest rc=$?"
tail -5 "$OUT/pytest_gpu.log"
