#!/bin/bash
# Reverse mode of the fused rollout, single-GPU validation: build + smoke(), the new GPU tests, the
# throughput probe (tools/rollout_vjp_probe.py), bench.py, then the whole GPU suite.
#   bash tools/gpu_rollout_vjp.sh <out-dir>
set -u
mkdir -p "${1:?usage: bash tools/gpu_rollout_vjp.sh <out-dir>}"
OUT=$(cd "$1" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem,driver_version --format=csv > "$OUT/gpu.csv"
cat "$OUT/gpu.csv"

python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.log" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/smoke.log"

python -m pytest -q -rs -x tests/test_gpu_rollout_grad.py > "$OUT/pytest_rollout_grad.log" 2>&1
echo "new tests rc=$?"
tail -25 "$OUT/pytest_rollout_grad.log"

python tools/rollout_vjp_probe.py --log "$OUT/rollout_vjp_probe.log" > /dev/null 2> "$OUT/probe.err"
echo "probe rc=$?"
cat "$OUT/rollout_vjp_probe.log"; tail -5 "$OUT/probe.err"

python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"
echo "bench rc=$?"
tail -c 600 "$OUT/bench.json"; echo

python -m pytest -m gpu -q -rs tests > "$OUT/pytest_gpu.log" 2>&1
echo "pytest rc=$?"
tail -5 "$OUT/pytest_gpu.log"
