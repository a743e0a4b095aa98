#!/bin/bash
# Step evaluation in one point-major pass: build this tree and the parent's (in .head/), the new test file on both trees
# (the parent's errors against the oracle are the baseline of its tolerances), the whole GPU suite, bench.py alternated
# parent / this tree (cfg5, cfg4 and cfg3 three times each, cfg1, cfg2 and cfg3ref once) with the phase times, smoke.
# The outputs of both trees are compared by scripts/gpu_r10_check.sh.
# Before the call: mkdir .head && git archive <parent commit> | tar -x -C .head
set -u
OUT="${1:?usage: scripts/gpu_r10.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
tail -n 2 "$OUT"/build.log "$OUT"/build_head.log | cut -c1-200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
timeout 600 python -m pytest -q -s -m gpu -p no:cacheprovider tests/test_gpu_step_evaluation.py > "$OUT"/step_eval_tests.log 2>&1
echo "step evaluation tests rc=$?"; grep -E "^(cfg|wide)|passed|failed|FAILED|Error" "$OUT"/step_eval_tests.log | tail -20
cp tests/test_gpu_step_evaluation.py .head/tests/
(cd .head && timeout 600 python -m pytest -q -s -m gpu -p no:cacheprovider tests/test_gpu_step_evaluation.py) > "$OUT"/step_eval_tests_head.log 2>&1
echo "step evaluation tests on the parent rc=$?"; grep -E "^(cfg|wide)|passed|failed" "$OUT"/step_eval_tests_head.log | tail -20
timeout 1800 python -m pytest -q -m gpu tests -p no:cacheprovider > "$OUT"/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
summary() {
  tail -1 "$1" | python -c '
import json, sys
d = json.loads(sys.stdin.read())
ph = d.get("phase_ms_per_step") or {}
print(round(d["value"], 2), d.get("final_cost"), (d.get("parity_vs_n1") or {}).get("ok") if isinstance(d.get("parity_vs_n1"), dict) else d.get("parity_vs_n1"))
print("   ", {k: round(v, 4) for k, v in ph.items()} if isinstance(ph, dict) else ph)' 2>&1 | cut -c1-600
}
for w in cfg5 cfg5 cfg5 cfg4 cfg4 cfg4 cfg3 cfg3 cfg3 cfg3ref cfg2 cfg1; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    n=$(ls "$OUT"/bench_${w}_${t}_*.log 2>/dev/null | wc -l)
    (cd $d && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w) > "$OUT"/bench_${w}_${t}_$((n + 1)).log 2>&1
    echo "bench $w $t $((n + 1)) rc=$?"; summary "$OUT"/bench_${w}_${t}_$((n + 1)).log
  done
done
timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -3 "$OUT"/smoke.log | cut -c1-300
