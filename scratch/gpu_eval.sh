#!/bin/bash
# evaluation path on a B200: new tests, the whole GPU suite, smoke, bench, throughput measurement
# usage: bash scratch/gpu_eval.sh [output directory, default out/gpu_eval]
OUT=${1:-out/gpu_eval}
mkdir -p "$OUT"
python -m pytest -q -m gpu tests/test_gpu_eval.py -s -p no:cacheprovider 2>&1 | tail -40 | tee "$OUT/eval_tests.txt"
python -m pytest -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_eval.py 2>&1 | tail -15 | tee "$OUT/gpu_suite.txt"
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -3 | tee "$OUT/bench.txt"
python scratch/eval_throughput.py 2>&1 | tee "$OUT/eval_throughput.txt"
