#!/bin/bash
# covariance-blocks round: (build), the new GPU tests (measured errors printed), the covariance tests it shares code with, the
# benchmark of scripts/covariance_blocks_bench.py; FULL=1: the whole GPU suite, smoke, bench.py
set -u
OUT="${1:?usage: scripts/gpu_r9_covblocks.sh OUTPUT_DIR}"
mkdir -p "$OUT"
if [ "${BUILD:-1}" = 1 ]; then
  python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 || { tail -30 "$OUT"/build.log; exit 1; }
fi
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/device.txt 2>&1
timeout 1500 python -m pytest -q -s -m gpu tests/test_gpu_covariance_blocks.py tests/test_gpu_covariance.py \
  tests/test_gpu_irregular_covisibility.py -k "blocks or covariance or rank_deficient_rejected" -p no:cacheprovider > "$OUT"/cov_tests.log 2>&1
echo "cov tests rc=$?"; grep -E "max relative|against ba_gpu|passed|failed|Error |error:|FAILED" "$OUT"/cov_tests.log | cut -c1-300 | tail -60
timeout 900 python scripts/covariance_blocks_bench.py --repeats 5 --sizes "${SIZES:-3000,10000}" --out "$OUT"/covblocks_bench.jsonl > "$OUT"/covblocks_bench.log 2>&1
echo "bench rc=$?"; cut -c1-900 "$OUT"/covblocks_bench.log | tail -5
if [ "${FULL:-0}" = 1 ]; then
  timeout 1800 python -m pytest -q -m gpu -p no:cacheprovider > "$OUT"/gpu_suite.log 2>&1
  echo "gpu suite rc=$?"; tail -4 "$OUT"/gpu_suite.log
  timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -2 "$OUT"/smoke.log | cut -c1-300
  timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT"/bench.log 2>&1; echo "bench.py rc=$?"; tail -1 "$OUT"/bench.log | cut -c1-700
fi
