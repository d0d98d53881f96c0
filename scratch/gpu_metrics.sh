#!/bin/bash
# crystal metrics on a B200: new tests, the whole GPU suite, smoke, bench, kernel timings
# usage: bash scratch/gpu_metrics.sh [output directory, default out/gpu_metrics] [quick: the new tests only]
OUT=${1:-out/gpu_metrics}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
grep -A3 crystal_metrics arreau_b200/lib/build.log | tee "$OUT/ptxas.txt"
python -m pytest -q -m gpu tests/test_crystal_metrics.py -s -p no:cacheprovider > "$OUT/metrics_tests.txt" 2>&1
grep -E "extended|sampler:|passed|failed|Error|assert" "$OUT/metrics_tests.txt" | tail -40
python scratch/crystal_metrics_time.py 2>&1 | tee "$OUT/crystal_metrics_time.txt"
if [ "$2" = "quick" ]; then exit 0; fi
python -m pytest -q -m gpu -p no:cacheprovider --ignore=tests/test_crystal_metrics.py 2>&1 | tail -15 | tee "$OUT/gpu_suite.txt"
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -3 | tee "$OUT/bench.txt"
