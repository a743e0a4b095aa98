#!/bin/bash
# Point-major linearisation without a record plane, 32-byte g records: build this tree and the parent's (in .head/), the new
# tests, bench.py cfg5 alternated parent / this tree three times, cfg4 and cfg3 once each, the outputs of both trees at cfg5
# compared, the whole GPU suite, smoke.
# Before the call: mkdir .head && git archive <parent commit> | tar -x -C .head
set -u
OUT="${1:?usage: scripts/gpu_r7.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
tail -2 "$OUT"/build.log "$OUT"/build_head.log | cut -c1-200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
timeout 600 python -m pytest -q -s -m gpu tests/test_gpu_fused_linearize.py -p no:cacheprovider > "$OUT"/new_tests.log 2>&1
echo "new tests rc=$?"; grep -E "passed|failed|FAILED|Error|assert" "$OUT"/new_tests.log | tail -20
summary() {
  tail -1 "$1" | python -c 'import json,sys; d=json.loads(sys.stdin.read()); print(round(d["value"],2), d.get("final_cost"), d.get("parity_vs_n1"), {k: round(v,3) for k,v in d.get("phase_ms_per_step",{}).items()})' 2>&1 | cut -c1-700
}
for i in 1 2 3; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    (cd $d && timeout 600 python bench.py --gpus 1 --no-cpu-baseline) > "$OUT"/bench_cfg5_${t}_$i.log 2>&1; echo "bench cfg5 $t $i rc=$?"
    summary "$OUT"/bench_cfg5_${t}_$i.log
  done
done
for w in cfg4 cfg3; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    (cd $d && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w) > "$OUT"/bench_${w}_${t}.log 2>&1; echo "bench $w $t rc=$?"
    summary "$OUT"/bench_${w}_${t}.log
  done
done
D=$(mktemp -d)
(cd .head && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --dump-outputs "$D"/head) > "$OUT"/dump_head.log 2>&1; echo "dump head rc=$?"
timeout 600 python bench.py --gpus 1 --no-cpu-baseline --dump-outputs "$D"/branch > "$OUT"/dump_branch.log 2>&1; echo "dump branch rc=$?"
python - "$D" <<'EOF' | tee "$OUT"/dump_compare.txt
import glob, os, sys
import numpy as np
d = sys.argv[1]
for f in sorted(glob.glob(os.path.join(d, "head", "*.npy"))):
    k = os.path.basename(f)[:-4]
    a, b = np.load(f), np.load(os.path.join(d, "branch", k + ".npy"))
    same = a.shape == b.shape and np.array_equal(a, b)
    rel = float(np.max(np.abs(a - b)) / max(np.max(np.abs(a)), 1e-300)) if a.shape == b.shape and a.size else float("nan")
    print(f"{k}: shape {a.shape} bit-identical {same} max rel diff {rel:.3e}")
EOF
rm -rf "$D"
timeout 1800 python -m pytest -q -m gpu tests -p no:cacheprovider --deselect tests/test_gpu_fused_linearize.py > "$OUT"/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -3 "$OUT"/smoke.log | cut -c1-300
