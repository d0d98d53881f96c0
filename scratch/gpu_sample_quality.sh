#!/bin/bash
# keyed sampling noise + sample-quality monitoring on a B200: new tests, timings, the whole GPU suite, smoke, bench
# usage: bash scratch/gpu_sample_quality.sh [output directory, default out/gpu_sample_quality] [quick: new tests + timings]
OUT=${1:-out/gpu_sample_quality}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
grep -B1 -A3 "noise\|sample_init" arreau_b200/lib/build.log > "$OUT/ptxas.txt"
python -m pytest -q -m gpu tests/test_gpu_keyed_sampling.py -s -p no:cacheprovider > "$OUT/keyed_tests.txt" 2>&1
grep -E "sample quality|passed|failed|Error|assert" "$OUT/keyed_tests.txt" | tail -40
python scratch/sample_quality_time.py 2>&1 | tee "$OUT/sample_quality_time.txt"
if [ "$2" = "quick" ]; then exit 0; fi
python -m pytest -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_keyed_sampling.py 2>&1 | tail -15 | tee "$OUT/gpu_suite.txt"
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -3 | tee "$OUT/bench.txt"
