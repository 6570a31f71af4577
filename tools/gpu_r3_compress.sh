#!/bin/bash
# Compressible control-matrix outputs, single-GPU validation: smoke(), bench.py alternated three times
# against a build of the parent commit (its tree in $BASE, default _base), --dump-outputs of both
# compared file for file, then the whole GPU suite.   BASE=<parent tree> bash tools/gpu_r3_compress.sh <out-dir>
set -u
mkdir -p "${1:?usage: BASE=<parent tree> bash tools/gpu_r3_compress.sh <out-dir>}"
OUT=$(cd "$1" && pwd)
BASE=${BASE:-_base}
DUMPS=$(mktemp -d)   # the two --dump-outputs sets (34 MB each) are compared here, then removed
trap 'rm -rf "$DUMPS"' EXIT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem,driver_version --format=csv > "$OUT/gpu.csv"
cat "$OUT/gpu.csv"

python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.log" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/smoke.log"

for i in 1 2 3; do
    d_base="" d_new=""
    if [ "$i" = 1 ]; then d_base="--dump-outputs $DUMPS/base"; d_new="--dump-outputs $DUMPS/new"; fi
    t0=$(date +%s)
    (cd "$BASE" && python bench.py --gpus 1 --steps 20 --warmup 5 $d_base) > "$OUT/bench_base_$i.json" 2> "$OUT/bench_base_$i.err"
    t1=$(date +%s)
    python bench.py --gpus 1 --steps 20 --warmup 5 $d_new > "$OUT/bench_new_$i.json" 2> "$OUT/bench_new_$i.err"
    t2=$(date +%s)
    echo "round $i: base $((t1 - t0)) s, new $((t2 - t1)) s"
done
for f in "$DUMPS"/base/*.npy; do
    cmp -s "$f" "$DUMPS/new/$(basename "$f")" && echo "dump identical: $(basename "$f")" || echo "dump DIFFERS: $(basename "$f")"
done

python - "$OUT" <<'EOF'
import json, statistics, sys, glob, os
out = sys.argv[1]
rows = {}
for arm in ("base", "new"):
    rows[arm] = []
    for i in (1, 2, 3):
        try:
            d = json.loads(open(os.path.join(out, f"bench_{arm}_{i}.json")).read().strip().splitlines()[-1])
        except Exception as e:
            print(arm, i, "no result:", e); continue
        c3 = d.get("configs3_het64m", {})
        c2 = d.get("configs2", {})
        rows[arm].append(d["value"])
        print(f"{arm} {i}: value {d['value']:.4e} ms/step {d['ms_per_step']:.3f} windows {d['output_windows']} "
              f"parity.ok {d['parity']['ok']} zeros {d['parity']['structural_zeros_exact']} "
              f"frac {d['roofline']['frac']:.3f} | configs3 {c3.get('value', 0):.4e} ms {c3.get('ms_per_step', 0):.3f} "
              f"| configs2 {json.dumps({k: v.get('value') for k, v in c2.items() if isinstance(v, dict) and 'value' in v})} "
              f"{c2.get('value')} | clocks {json.dumps(d.get('clocks'))[:300]}")
if rows["base"] and rows["new"]:
    mb, mn = statistics.median(rows["base"]), statistics.median(rows["new"])
    sp = lambda v: (max(v) - min(v)) / statistics.median(v)
    print(f"median value base {mb:.4e} new {mn:.4e} gain {mn / mb:.4f}; spread base {100 * sp(rows['base']):.2f} % "
          f"new {100 * sp(rows['new']):.2f} %")
EOF

python -m pytest -m gpu -q -rs tests > "$OUT/pytest_gpu.log" 2>&1
echo "pytest rc=$?"
tail -5 "$OUT/pytest_gpu.log"
