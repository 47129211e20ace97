#!/bin/bash
# The r10 evidence in one GPU call: the decoder suite at this commit and at the parent (which lacks the fixes), the
# whole GPU suite, smoke(), bit-identity of bench.py's outputs and gradients against the parent, and pose-0 / pose-2
# step times of both alternated.
#   profiles/gpu_r10_decoder.sh PARENT OUT
# PARENT: a built checkout of the parent commit; OUT: the output directory.
set -u
P=$(cd "$1" && pwd)
OUT=$(mkdir -p "$2" && cd "$2" && pwd)
ROOT=$(cd "$(dirname "$0")/.." && pwd)
cd "$ROOT"
SMI="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader"
$SMI > "$OUT/smi.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.txt" 2>&1
echo "build rc=$?" | tee -a "$OUT/status.txt"

python -m pytest tests/test_gpu_decoder.py -q -m gpu --durations=15 > "$OUT/pytest_decoder.txt" 2>&1
echo "decoder suite rc=$?" | tee -a "$OUT/status.txt"
cp tests/test_gpu_decoder.py "$P/tests/test_gpu_decoder.py"
(cd "$P" && python -m pytest tests/test_gpu_decoder.py -q -m gpu -rf > "$OUT/pytest_decoder_on_parent.txt" 2>&1)
echo "decoder suite on the parent rc=$?" | tee -a "$OUT/status.txt"
rm -f "$P/tests/test_gpu_decoder.py"
python -m pytest tests -q -m gpu > "$OUT/pytest_gpu.txt" 2>&1
echo "gpu suite rc=$?" | tee -a "$OUT/status.txt"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.txt" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/status.txt"

for arm in parent change; do
  dir=$ROOT; [ $arm = parent ] && dir=$P
  (cd "$dir" && python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu-baseline --no-train-epoch --no-config5 \
      --no-loss-check --dump-outputs "$OUT/dump_$arm" > /dev/null 2>&1)
done
python - "$OUT" <<'EOF' | tee -a "$OUT/status.txt"
import os, sys, numpy as np
out = sys.argv[1]
a, b = os.path.join(out, "dump_parent"), os.path.join(out, "dump_change")
names = sorted(f for f in os.listdir(a) if f.endswith(".npy")) if os.path.isdir(a) else []
same = [n for n in names if os.path.isfile(os.path.join(b, n)) and
        np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print(f"dump-outputs: {len(same)} of {len(names)} arrays np.array_equal; differ: {sorted(set(names) - set(same))}")
EOF

STEP="bench.py --gpus 1 --steps 200 --warmup 10 --no-cpu-baseline --no-train-epoch --no-config5 --no-loss-check"
for i in 1 2 3; do
  if [ $((i % 2)) = 1 ]; then order="parent change"; else order="change parent"; fi
  for wl in pose pose2; do
    for arm in $order; do
      dir=$ROOT; [ $arm = parent ] && dir=$P
      (cd "$dir" && python $STEP --workload $wl 2>/dev/null | tail -1) > "$OUT/step_${wl}_${arm}_$i.json"
    done
  done
done
$SMI >> "$OUT/smi.txt"
