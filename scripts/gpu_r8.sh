#!/bin/bash
# Removal of the superseded kernels and their switches: build this tree and the parent's (in .head/), the changed tests,
# the whole GPU suite, the outputs of both trees at cfg5 and cfg3ref compared bit for bit, bench.py alternated parent / this
# tree (cfg5 three times, cfg3ref, cfg2 and cfg1 once each), smoke.
# Before the call: mkdir .head && git archive <parent commit> | tar -x -C .head
set -u
OUT="${1:?usage: scripts/gpu_r8.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
tail -n 2 "$OUT"/build.log "$OUT"/build_head.log | cut -c1-200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
timeout 900 python -m pytest -q -s -m gpu -p no:cacheprovider tests/test_gpu_schur_values.py \
  "tests/test_gpu_parity.py::test_solve_explicit_blocked_cholesky_ref" tests/test_gpu_parity.py::test_blocked_cholesky_schedules_are_bit_identical \
  tests/test_gpu_spchol_border.py::test_other_tree_agrees tests/test_gpu_irregular_covisibility.py::test_covariance_other_tree_agrees \
  > "$OUT"/changed_tests.log 2>&1
echo "changed tests rc=$?"; grep -E "passed|failed|FAILED|Error|assert" "$OUT"/changed_tests.log | tail -20
timeout 1800 python -m pytest -q -m gpu tests -p no:cacheprovider > "$OUT"/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
D=$(mktemp -d)
for w in cfg5 cfg3ref; do
  (cd .head && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w --dump-outputs "$D"/head_$w) > "$OUT"/dump_${w}_head.log 2>&1
  echo "dump $w head rc=$?"
  timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w --dump-outputs "$D"/branch_$w > "$OUT"/dump_${w}_branch.log 2>&1
  echo "dump $w branch rc=$?"
done
python - "$D" <<'EOF' | tee "$OUT"/dump_compare.txt
import glob, os, sys
import numpy as np
d = sys.argv[1]
for w in ("cfg5", "cfg3ref"):
    files = sorted(glob.glob(os.path.join(d, "head_" + w, "*.npy")))
    print(f"{w}: {len(files)} arrays")
    for f in files:
        k = os.path.basename(f)[:-4]
        a, b = np.load(f), np.load(os.path.join(d, "branch_" + w, k + ".npy"))
        print(f"  {k}: shape {a.shape} bit-identical {a.shape == b.shape and np.array_equal(a, b)}")
EOF
rm -rf "$D"
summary() {
  tail -1 "$1" | python -c 'import json,sys; d=json.loads(sys.stdin.read()); print(round(d["value"],2), d.get("final_cost"), d.get("parity_vs_n1"))' 2>&1 | cut -c1-300
}
for w in cfg5 cfg5 cfg5 cfg3ref cfg2 cfg1; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    n=$(ls "$OUT"/bench_${w}_${t}_*.log 2>/dev/null | wc -l)
    (cd $d && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w) > "$OUT"/bench_${w}_${t}_$((n + 1)).log 2>&1
    echo "bench $w $t $((n + 1)) rc=$?"; summary "$OUT"/bench_${w}_${t}_$((n + 1)).log
  done
done
timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -3 "$OUT"/smoke.log | cut -c1-300
