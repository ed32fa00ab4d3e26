#!/bin/bash
# round 3: the chains beside the fits (rcmarl_overlap_split).  CTA-budget sweep of both phases alone and together
# (tools/prof_overlap.py), then the C2 bench of the parent commit's tree (built in ./_ab_head) and of this tree alternated
# three times each, both dumps (--dump-outputs) compared array by array, the GPU suite and smoke.
#   bash tools/calls/r03_call1_overlap.sh OUT_DIR        (run from the repository root; results go to OUT_DIR)
OUT=${1:?usage: r03_call1_overlap.sh OUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem --format=csv
echo "== CTA-budget sweep"
timeout 600 python tools/prof_overlap.py 2>&1 | tee "$OUT/r03_overlap_sweep.jsonl" | tail -16
echo "== C2 bench, parent (A) and branch (B) alternated"
for i in 1 2 3; do
  (cd _ab_head && timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3) > "$OUT/r03_bench_A$i.json" 2> "$OUT/r03_bench_A$i.err"
  timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT/r03_bench_B$i.json" 2> "$OUT/r03_bench_B$i.err"
done
OUT="$OUT" python - <<'PY'
import json, os
out = os.environ["OUT"]
for ab in "AB":
    for i in (1, 2, 3):
        try:
            d = json.load(open(f"{out}/r03_bench_{ab}{i}.json"))
            print(ab, i, d["value"], d["ms_per_step"], d.get("clocks"), d["breakdown_ms"])
        except Exception as ex:
            print(ab, i, "failed", ex)
PY
echo "== dumps"
(cd _ab_head && timeout 600 python bench.py --gpus 1 --steps 2 --warmup 1 --no-cpu-baseline --no-e2e --no-consensus --dump-outputs "$OUT/r03_dump_A") > /dev/null 2>&1
timeout 600 python bench.py --gpus 1 --steps 2 --warmup 1 --no-cpu-baseline --no-e2e --no-consensus --dump-outputs "$OUT/r03_dump_B" > /dev/null 2>&1
OUT="$OUT" python - <<'PY'
import glob, os
import numpy as np
out = os.environ["OUT"]
for fa in sorted(glob.glob(f"{out}/r03_dump_A/*.npy")):
    n = os.path.basename(fa)
    a, b = np.load(fa).astype(np.float64), np.load(f"{out}/r03_dump_B/{n}").astype(np.float64)
    d = np.abs(a - b)
    print(f"{n:24s} identical={np.array_equal(a, b)} max_abs={d.max():.3e} max_rel={(d / (np.abs(a) + 1e-30)).max():.3e} "
          f"max_abs/(1e-5+1e-3|a|)={(d / (1e-5 + 1e-3 * np.abs(a))).max():.3f}")
PY
echo "== pytest -m gpu"
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -8
echo "== smoke"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
