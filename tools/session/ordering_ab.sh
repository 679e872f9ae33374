#!/bin/bash
# Subdomain elimination order of solve_kernel_v2, before / after on one GPU:
#   tools/session/ordering_ab.sh OUT_DIR PARENT_TREE [DEV_PARENT_TREE DEV_TREE]
# PARENT_TREE: a checkout of the previous commit with its library built; DEV_*: checkouts of the previous / this commit built
# with LRBMS_DEVTOOLS=1 (per-column cycle counters, tools/solve_timing.py).  Bench lines, output dumps, their comparison and
# the counters go to OUT_DIR.
set -u
USAGE="usage: $0 OUT_DIR PARENT_TREE [DEV_PARENT_TREE DEV_TREE]"
mkdir -p "${1:?$USAGE}"
OUT=$(cd "$1" && pwd)
PARENT=$(cd "${2:?$USAGE}" && pwd)
shift
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > "$OUT/gpu.csv" 2>&1
run() {   # run TAG TREE ARGS...
  local tag=$1 tree=$2; shift 2
  (cd "$tree" && timeout 900 python bench.py --gpus 1 "$@") > "$OUT/$tag.json" 2> "$OUT/$tag.err"
  echo "$tag rc=$? $(grep -o '"value": [0-9.]*' "$OUT/$tag.json" | head -1)"
}
# C2, alternating parent / this tree; the first pair also dumps the outputs of the last step
run c2_parent_1 "$PARENT" --steps 10 --warmup 3 --dump-outputs "$OUT/dump_parent"
run c2_branch_1 . --steps 10 --warmup 3 --dump-outputs "$OUT/dump_branch"
python tools/compare_dumps.py "$OUT/dump_branch" "$OUT/dump_parent" > "$OUT/compare_dumps.json"; echo "compare rc=$?"
for r in 2 3; do
  run c2_parent_$r "$PARENT" --steps 10 --warmup 3 --no-cpu-baseline --no-c5
  run c2_branch_$r . --steps 10 --warmup 3 --no-cpu-baseline --no-c5
done
for c in c3 c4; do
  run ${c}_parent "$PARENT" --config $c --steps 10 --warmup 3 --no-cpu-baseline
  run ${c}_branch . --config $c --steps 10 --warmup 3 --no-cpu-baseline
done
if [ $# -ge 3 ]; then
  for t in parent:$2 branch:$3; do
    (cd "${t#*:}" && timeout 600 python tools/solve_timing.py) > "$OUT/timing_solve_v2_${t%%:*}.txt" 2>&1
    echo "timing ${t%%:*} rc=$?"
  done
fi
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv >> "$OUT/gpu.csv" 2>&1
