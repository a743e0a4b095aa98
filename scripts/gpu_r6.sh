#!/bin/bash
# DMMA values-of-S round: build this tree and the parent's (in .head/), the new tests, bench.py cfg5 alternated parent /
# this tree, the SIMT / DMMA A/B on cfg5, cfg4, cfg3, the whole GPU suite, smoke.
# Before the call: mkdir .head && git archive <parent commit> | tar -x -C .head
set -u
OUT="${1:?usage: scripts/gpu_r6.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
tail -3 "$OUT"/build.log "$OUT"/build_head.log | cut -c1-200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
timeout 900 python -m pytest -q -s -m gpu tests/test_gpu_schur_values.py -p no:cacheprovider > "$OUT"/new_tests.log 2>&1
echo "new tests rc=$?"; grep -E "passed|failed|FAILED|Error|assert" "$OUT"/new_tests.log | tail -20
for i in 1 2 3; do
  for t in head branch; do
    if [ $t = head ]; then d=.head; else d=.; fi
    (cd $d && timeout 600 python bench.py --gpus 1) > "$OUT"/bench_cfg5_${t}_$i.log 2>&1; echo "bench $t $i rc=$?"
    tail -1 "$OUT"/bench_cfg5_${t}_$i.log | python -c 'import json,sys; d=json.loads(sys.stdin.read()); print(d["value"], d.get("final_cost"), d.get("parity_vs_n1"), {k: round(v,3) for k,v in d.get("phase_ms_per_step",{}).items()})' 2>&1 | cut -c1-600
  done
done
timeout 1500 python scripts/sp_schur_ab.py --out "$OUT"/r06_sp_schur_ab.jsonl > "$OUT"/ab.log 2>&1; echo "ab rc=$?"
python -c '
import json,sys
for l in open(sys.argv[1]):
    d=json.loads(l)
    print({k: (round(v,4) if isinstance(v,float) else v) for k,v in d.items() if k!="phase_ms_per_step"})' "$OUT"/r06_sp_schur_ab.jsonl | cut -c1-400
timeout 1800 python -m pytest -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_schur_values.py > "$OUT"/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|FAILED" "$OUT"/gpu_suite.log | tail -8
timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT"/smoke.log 2>&1; echo "smoke rc=$?"; tail -3 "$OUT"/smoke.log | cut -c1-300
