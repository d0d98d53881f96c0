#!/bin/bash
# resume + EMA on a B200: new tests, the whole GPU suite, smoke, bench, throughput with / without EMA alternated
# usage: bash scratch/gpu_resume.sh [output directory, default out/gpu_resume] [quick: the new tests only]
OUT=${1:-out/gpu_resume}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv 2>&1 | tee "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -2
python -m pytest -q -m gpu tests/test_gpu_resume.py -s -p no:cacheprovider > "$OUT/resume_tests.txt" 2>&1; grep -E "EMA vs|capacity|restored|passed|failed|Error" "$OUT/resume_tests.txt" | tail -40
if [ "$2" = "quick" ]; then exit 0; fi
python scratch/adam_ema_time.py 2>&1 | tee "$OUT/adam_ema_time.txt"
for r in 1 2; do
  python scratch/fit_throughput.py 8100 270 3 2>&1 | tee -a "$OUT/fit_throughput.txt"
  python scratch/fit_throughput.py 8100 270 3 0.999 2>&1 | tee -a "$OUT/fit_throughput.txt"
done
python -m pytest -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_resume.py 2>&1 | tail -15 | tee "$OUT/gpu_suite.txt"
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee "$OUT/smoke.txt"
python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -3 | tee "$OUT/bench.txt"
