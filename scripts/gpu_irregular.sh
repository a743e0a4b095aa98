#!/bin/bash
# irregular co-visibility round: build, the new GPU tests (measured errors and pivot ratios printed), the covariance tests, the
# whole GPU suite, smoke, bench.py lines of cfg3ref and cfg5
set -u
OUT="${1:?usage: scripts/gpu_irregular.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 || { tail -30 "$OUT"/build.log; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/device.txt 2>&1
timeout 1200 python -m pytest -q -s -m gpu tests/test_gpu_irregular_covisibility.py -p no:cacheprovider > "$OUT"/irregular_tests.log 2>&1
echo "irregular tests rc=$?"; grep -E "passed|failed|FAILED|Error" "$OUT"/irregular_tests.log | tail -30
timeout 600 python -m pytest -q -s -m gpu tests/test_gpu_covariance.py -p no:cacheprovider > "$OUT"/cov_tests.log 2>&1
echo "cov tests rc=$?"; grep -E "smallest|passed|failed|FAILED" "$OUT"/cov_tests.log | tail -20
if [ "${FULL:-1}" = 1 ]; then
  timeout 1500 python -m pytest -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_covariance.py \
    --deselect tests/test_gpu_irregular_covisibility.py > "$OUT"/gpu_suite.log 2>&1
  echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
  timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -2 "$OUT"/smoke.log | cut -c1-300
  for w in cfg3ref cfg5; do
    timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 --workload $w > "$OUT"/bench_$w.log 2>&1; echo "bench $w rc=$?"
    tail -1 "$OUT"/bench_$w.log | cut -c1-700
  done
fi
