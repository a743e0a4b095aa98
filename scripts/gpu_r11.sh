#!/bin/bash
# The solve plan decided once per upload: build this tree and the parent's (in .head/), the grown test_auto_policy on both,
# scripts/plan_trace.py on both and --compare, bench.py --dump-outputs at cfg5 and cfg3ref compared array by array, bench.py
# alternated parent / this tree (cfg5, cfg4 and cfg3 three times each, cfg3ref, cfg2 and cfg1 once), the GPU suite, the
# two-GPU tests when the machine has two GPUs, smoke.
# Before the call: mkdir .head && git archive <parent commit> | tar -x -C .head
set -u
OUT="${1:?usage: scripts/gpu_r11.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
tail -n 2 "$OUT"/build.log "$OUT"/build_head.log | cut -c1-200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
cp tests/test_gpu_edge_cases.py .head/tests/
cp scripts/plan_trace.py .head/scripts/
for t in branch head; do
  if [ $t = head ]; then d=.head; else d=.; fi
  (cd $d && timeout 900 python -m pytest -q -m gpu -p no:cacheprovider "tests/test_gpu_edge_cases.py::test_auto_policy") > "$OUT"/auto_policy_$t.log 2>&1
  echo "test_auto_policy $t rc=$?"; tail -n 3 "$OUT"/auto_policy_$t.log | cut -c1-300
done
P=$(mktemp -d)
for t in head branch; do
  if [ $t = head ]; then d=.head; else d=.; fi
  (cd $d && timeout 900 python scripts/plan_trace.py "$P"/$t) > "$OUT"/plan_trace_$t.log 2>&1
  echo "plan_trace $t rc=$?"
done
python scripts/plan_trace.py --compare "$P"/head "$P"/branch | tee "$OUT"/plan_trace_compare.txt
cp "$P"/branch/plan_trace.json "$OUT"/plan_trace_branch.json
rm -rf "$P"
D=$(mktemp -d)
for w in cfg5 cfg3ref; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    (cd $d && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w --dump-outputs "$D"/${t}_$w) > "$OUT"/dump_${w}_$t.log 2>&1
    echo "dump $w $t rc=$?"
  done
done
python - "$D" <<'PY' | tee "$OUT"/dump_compare.txt
import glob, os, sys
import numpy as np
d = sys.argv[1]
print("# bench.py --dump-outputs, parent commit vs this state")
for w in ("cfg5", "cfg3ref"):
    files = sorted(glob.glob(os.path.join(d, f"head_{w}", "*.npy")))
    print(f"{w}: {len(files)} arrays")
    for f in files:
        n = os.path.basename(f)[:-4]
        a, b = np.load(f), np.load(os.path.join(d, f"branch_{w}", n + ".npy"))
        print(f"  {n}: shape {a.shape} bit-identical {np.array_equal(a, b)}")
PY
rm -rf "$D"
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
timeout 1800 python -m pytest -q -m gpu tests -p no:cacheprovider > "$OUT"/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
if [ "$(nvidia-smi -L | wc -l)" -ge 2 ]; then
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    (cd $d && timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_multi.py) > "$OUT"/multi_$t.log 2>&1
    echo "multi-GPU tests $t rc=$?"; tail -n 2 "$OUT"/multi_$t.log
  done
else
  echo "one GPU: tests/test_gpu_multi.py not run"
fi
timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -3 "$OUT"/smoke.log | cut -c1-300
