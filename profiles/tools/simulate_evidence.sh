#!/bin/bash
# Evidence of the forward-simulation change on one GPU: card, GPU suite, smoke(), simulate_bench.py, then parent and
# new builds alternated on bench.py's headline and --dump-outputs of all seven workloads.
# Usage: profiles/tools/simulate_evidence.sh PARENT_TREE OUT   (PARENT_TREE: a built checkout of the parent commit)
set -u
PARENT=$1
OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/card.csv"
python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu.log" 2>&1; echo "rc=$?" >> "$OUT/pytest_gpu.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "rc=$?" >> "$OUT/smoke.log"
python profiles/tools/simulate_bench.py --out "$OUT" --profile > "$OUT/simulate_bench.log" 2>&1; echo "rc=$?" >> "$OUT/simulate_bench.log"
for i in 1 2; do
  (cd "$PARENT" && python bench.py --gpus 1 --steps 20 --warmup 3 --no-others --no-cpu) > "$OUT/headline_parent_$i.json" 2>/dev/null
  python bench.py --gpus 1 --steps 20 --warmup 3 --no-others --no-cpu > "$OUT/headline_new_$i.json" 2>/dev/null
done
TMP=$(mktemp -d)
: > "$OUT/outputs_compare.txt"
for w in c2 c2s c3 c3l c4 c5 c5s; do
  (cd "$PARENT" && python bench.py --workload $w --steps 2 --warmup 1 --no-others --no-cpu --dump-outputs "$TMP/parent_$w") > /dev/null 2>&1
  python bench.py --workload $w --steps 2 --warmup 1 --no-others --no-cpu --dump-outputs "$TMP/new_$w" > /dev/null 2>&1
  n=$(ls "$TMP/new_$w" 2>/dev/null | wc -l)
  if [ "$n" -gt 0 ] && diff -rq "$TMP/parent_$w" "$TMP/new_$w" > /dev/null; then
    echo "$w: $n files, byte-identical" >> "$OUT/outputs_compare.txt"
  else
    echo "$w: DIFFERENT or missing ($n files)" >> "$OUT/outputs_compare.txt"
  fi
done
rm -rf "$TMP"
