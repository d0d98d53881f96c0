#!/bin/bash
# uniqueness and novelty on a B200: build, the new GPU tests, the timing run, scratch/structure_match_time.py on the
# parent tree (exported to scratch/ab_base with git archive) and on this tree alternately; with "full" also smoke,
# bench.py on both trees alternately and the whole suite
# usage: bash scratch/gpu_unique_novel.sh [full] [output directory, default out/unique_novel]
MODE=${1:-new}
OUT=${2:-out/unique_novel}
mkdir -p "$OUT" && OUT=$(cd "$OUT" && pwd)      # absolute: the A/B runs write from the other tree
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
grep -A2 -E "structure_match_kernel" arreau_b200/lib/build.log > "$OUT/ptxas.txt"
timeout 1200 python -m pytest -q -s -m gpu tests/test_gpu_unique_novel.py -p no:cacheprovider > "$OUT/new_tests.txt" 2>&1
tail -30 "$OUT/new_tests.txt"
timeout 900 python scratch/unique_novel_time.py 2>&1 | tee "$OUT/unique_novel_time.txt"
if [ -d scratch/ab_base ]; then
  (cd scratch/ab_base && python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -1)
  for r in 1 2; do
    for tree in scratch/ab_base .; do
      echo "== $tree" | tee -a "$OUT/structure_match_ab.txt"
      (cd $tree && timeout 600 python scratch/structure_match_time.py 2>&1 | tee -a "$OUT/structure_match_ab.txt")
    done
  done
fi
if [ "$MODE" = full ]; then
  python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
  for r in 1 2; do
    for tree in scratch/ab_base .; do
      [ -d $tree ] || continue
      echo "== $tree" >> "$OUT/bench.jsonl"
      (cd $tree && python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -1 | tee -a "$OUT/bench.jsonl")
    done
  done
  timeout 2400 python -m pytest -q -p no:cacheprovider --ignore=tests/test_gpu_unique_novel.py \
    --ignore=scratch 2>&1 | tail -15 | tee "$OUT/suite.txt"
fi
