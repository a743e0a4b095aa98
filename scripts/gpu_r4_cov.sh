#!/bin/bash
# covariance round: build, the new GPU tests (measured errors printed), the covariance benchmark, the whole GPU suite, smoke,
# bench.py lines of cfg3ref and cfg5
set -u
OUT="${1:?usage: scripts/gpu_r4_cov.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 || { tail -30 "$OUT"/build.log; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/device.txt 2>&1
timeout 1200 python -m pytest -q -s -m gpu tests/test_gpu_covariance.py -p no:cacheprovider > "$OUT"/cov_tests.log 2>&1
echo "cov tests rc=$?"; grep -E "covariance max|passed|failed|Error |error:" "$OUT"/cov_tests.log | tail -40
timeout 600 python scripts/covariance_bench.py --out "$OUT"/cov_bench.jsonl > "$OUT"/cov_bench.log 2>&1
echo "cov bench rc=$?"; cut -c1-400 "$OUT"/cov_bench.log | tail -5
if [ "${FULL:-1}" = 1 ]; then
  timeout 1500 python -m pytest -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_covariance.py > "$OUT"/gpu_suite.log 2>&1
  echo "gpu suite rc=$?"; tail -4 "$OUT"/gpu_suite.log
  timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -2 "$OUT"/smoke.log | cut -c1-300
  for w in cfg3ref cfg5; do
    timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 --workload $w > "$OUT"/bench_$w.log 2>&1; echo "bench $w rc=$?"
    tail -1 "$OUT"/bench_$w.log | cut -c1-700
  done
fi
