#!/bin/bash
# structure-conditioned sampling on a B200: new tests, timings, bench against the parent tree (scratch/ab_base, a copy
# of the parent commit with its library built), the whole GPU suite and smoke
# usage: bash scratch/gpu_structure.sh [output directory, default out/gpu_structure]
OUT=${1:-out/gpu_structure}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
grep -A1 -E "reverse_kernel" arreau_b200/lib/build.log > "$OUT/ptxas.txt"
python -m pytest -q -m gpu tests/test_gpu_structure_conditioning.py -p no:cacheprovider > "$OUT/new_tests.txt" 2>&1
tail -30 "$OUT/new_tests.txt"
python scratch/structure_time.py 3 2>&1 | tee "$OUT/structure_time.txt"
for r in 1 2 3; do
  for tree in base new; do
    if [ $tree = base ]; then dir=scratch/ab_base; else dir=.; fi
    (cd $dir && python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -1) | tee -a "$OUT/bench_$tree.jsonl"
  done
done
python -m pytest -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_structure_conditioning.py 2>&1 | tail -15 | tee "$OUT/gpu_suite.txt"
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
