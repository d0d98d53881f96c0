#!/bin/bash
# structure matcher on a B200: build, the new GPU tests, the timing run; with "full" also the whole GPU suite, smoke and
# bench.py twice
# usage: bash scratch/gpu_structure_match.sh [full] [output directory, default out/structure_match]
MODE=${1:-new}
OUT=${2:-out/structure_match}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
grep -A2 -E "structure_match_kernel" arreau_b200/lib/build.log > "$OUT/ptxas.txt"
timeout 900 python -m pytest -q -m gpu tests/test_gpu_structure_match.py -p no:cacheprovider > "$OUT/new_tests.txt" 2>&1
tail -30 "$OUT/new_tests.txt"
timeout 900 python scratch/structure_match_time.py 2>&1 | tee "$OUT/structure_match_time.txt"
if [ "$MODE" = full ]; then
  python -m pytest -q -p no:cacheprovider --ignore=tests/test_gpu_structure_match.py 2>&1 | tail -15 | tee "$OUT/suite.txt"
  python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
  for r in 1 2; do python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -1 | tee -a "$OUT/bench.jsonl"; done
fi
