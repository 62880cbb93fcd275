#!/bin/bash
# usage: scripts/ab_compare.sh BASE_TREE OUT_DIR [REPS]
# A/B of this tree against BASE_TREE (another built checkout, e.g. the parent commit), one GPU:
#  1. outputs: bench.py --dump-outputs on configs 4, 2, 5, 3 and 1 in both trees, compared array by array
#     (scripts/compare_outputs.py);
#  2. speed: the default bench line (config 4, configs 2 and 5 under "extra") alternating between the trees REPS times.
# Writes the GPU's name and power limit, the bench lines, a summary and the dumps that differ under OUT_DIR.  Exit
# status 1 when an output differs.
set -u
BASE=$(cd "$1" && pwd)
NEW=$(cd "$(dirname "$0")/.." && pwd)
mkdir -p "$2"
OUT=$(cd "$2" && pwd)
REPS=${3:-3}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
rc=0
for w in config4 config2 config5 config3 config1; do
  for side in base new; do
    tree=$BASE; [ $side = new ] && tree=$NEW
    (cd "$tree" && python bench.py --workload $w --steps 10 --warmup 3 --no-cpu-baseline --no-extra \
       --dump-outputs "$OUT/dump_${side}_$w") > "$OUT/dump_${side}_$w.json" 2> "$OUT/dump_${side}_$w.err"
  done
  echo "== outputs $w"
  if python "$NEW/scripts/compare_outputs.py" "$OUT/dump_base_$w" "$OUT/dump_new_$w"; then
    rm -rf "$OUT/dump_base_$w" "$OUT/dump_new_$w"  # up to 64 MB each: kept only when they differ
  else
    rc=1
  fi
done
for i in $(seq "$REPS"); do
  for side in base new; do
    tree=$BASE; [ $side = new ] && tree=$NEW
    (cd "$tree" && python bench.py --no-cpu-baseline) > "$OUT/bench_${side}_$i.json" 2> "$OUT/bench_${side}_$i.err"
  done
done
python - "$OUT" "$REPS" <<'EOF' | tee "$OUT/summary.txt"
import json, sys
out, reps = sys.argv[1], int(sys.argv[2])
for side in ("base", "new"):
    for i in range(1, reps + 1):
        f = f"{out}/bench_{side}_{i}.json"
        try:
            d = json.loads(open(f).read().strip().splitlines()[-1])
        except Exception as e:
            print(side, i, "no bench line:", e)
            continue
        pk = {k: round(v, 3) for k, v in d["roofline"]["per_kernel_ms"].items()}
        ex = {n: (round(e["value"], 1), round(e["ms_per_step"], 4)) for n, e in d["extra"].items()}
        print(side, i, "config4", round(d["value"], 3), "iter/s", round(d["ms_per_step"], 3), "ms/step", pk, "extra", ex)
EOF
exit $rc
