#!/bin/bash
# The r09 evidence in one GPU call: ranking suites then the whole GPU suite, smoke(), bit-identity of every ranking
# output against the parent commit, rank_bench.py of both alternated twice, bench.py step time of both alternated.
#   profiles/gpu_r09_rankfold.sh PARENT OUT
# PARENT: a built checkout of the parent commit; OUT: the output directory.
set -u
P=$(cd "$1" && pwd)
OUT=$(mkdir -p "$2" && cd "$2" && pwd)
ROOT=$(cd "$(dirname "$0")/.." && pwd)
cd "$ROOT"
SMI="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader"
$SMI > "$OUT/smi.txt"

python -m pytest tests/test_gpu_ranking.py tests/test_gpu_relation_ranking.py tests/test_gpu_pair_ranking.py \
    tests/test_gpu_pair_ranker.py -q -m gpu > "$OUT/pytest_rank.txt" 2>&1
echo "ranking suites rc=$?" | tee -a "$OUT/status.txt"
python -m pytest tests -q -m gpu > "$OUT/pytest_gpu.txt" 2>&1
echo "gpu suite rc=$?" | tee -a "$OUT/status.txt"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.txt" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/status.txt"

python profiles/rank_parity.py --other "$P" --out "$OUT" > "$OUT/parity_stdout.txt" 2>&1
echo "parity rc=$?" | tee -a "$OUT/status.txt"

for i in 1 2; do
  (cd "$P" && python profiles/rank_bench.py --out "$OUT/bench_parent_$i" > /dev/null 2>&1)
  echo "bench parent $i rc=$?" | tee -a "$OUT/status.txt"
  python profiles/rank_bench.py --out "$OUT/bench_change_$i" > /dev/null 2>&1
  echo "bench change $i rc=$?" | tee -a "$OUT/status.txt"
done
$SMI >> "$OUT/smi.txt"

STEP="bench.py --gpus 1 --steps 200 --warmup 10 --no-cpu-baseline --no-train-epoch --no-config5 --no-loss-check"
for i in 1 2 3; do
  if [ $((i % 2)) = 1 ]; then order="parent change"; else order="change parent"; fi
  for arm in $order; do
    dir=$ROOT; [ $arm = parent ] && dir=$P
    (cd "$dir" && python $STEP 2>/dev/null | tail -1) > "$OUT/step_${arm}_$i.json"
  done
done
for arm in parent change; do
  dir=$ROOT; [ $arm = parent ] && dir=$P
  (cd "$dir" && python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu-baseline --no-train-epoch --no-config5 \
      --no-loss-check --dump-outputs "$OUT/dump_$arm" > /dev/null 2>&1)
done
python - "$OUT" <<'EOF'
import os, sys, numpy as np
out = sys.argv[1]
a, b = os.path.join(out, "dump_parent"), os.path.join(out, "dump_change")
names = sorted(f for f in os.listdir(a) if f.endswith(".npy")) if os.path.isdir(a) else []
same = [n for n in names if os.path.isfile(os.path.join(b, n)) and
        np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print(f"dump-outputs: {len(same)} of {len(names)} arrays np.array_equal")
EOF
$SMI >> "$OUT/smi.txt"
