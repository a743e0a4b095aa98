#!/bin/bash
# Second call of the step-evaluation change: the new test file with its tolerances set from the first call's measurements,
# and bench.py --dump-outputs of the parent (.head/) and this tree at cfg5 and cfg3 after one LM iteration (the state is
# then the first candidate: y and x+ are to keep their bits) and after the default ten, compared array by array as the
# largest difference over the largest magnitude.
set -u
OUT="${1:?usage: scripts/gpu_r10_check.sh OUTPUT_DIR}"
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT"/build.log 2>&1 &
(cd .head && python -c 'import __graft_entry__ as g; g.build()') > "$OUT"/build_head.log 2>&1 &
wait
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/device.txt
timeout 600 python -m pytest -q -s -m gpu -p no:cacheprovider tests/test_gpu_step_evaluation.py > "$OUT"/step_eval_tests.log 2>&1
echo "step evaluation tests rc=$?"; grep -E "^(cfg|wide)|passed|failed|FAILED|Error" "$OUT"/step_eval_tests.log | tail -20
D=$(mktemp -d)
for w in cfg5 cfg3; do
  for k in 1 10; do
    (cd .head && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w --steps $k --dump-outputs "$D"/head_${w}_$k) > "$OUT"/dump_${w}_${k}_head.log 2>&1
    echo "dump $w $k head rc=$?"
    timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w --steps $k --dump-outputs "$D"/branch_${w}_$k > "$OUT"/dump_${w}_${k}_branch.log 2>&1
    echo "dump $w $k branch rc=$?"
  done
done
python - "$D" <<'PY' | tee "$OUT"/dump_compare.txt
import glob, os, sys
import numpy as np
d = sys.argv[1]
print("# bench.py --dump-outputs, parent commit vs this state; difference = max |a - b| / max |a| per array")
for w in ("cfg5", "cfg3"):
    for k in (1, 10):
        files = sorted(glob.glob(os.path.join(d, f"head_{w}_{k}", "*.npy")))
        print(f"{w}, {k} LM iteration(s): {len(files)} arrays")
        for f in files:
            n = os.path.basename(f)[:-4]
            a, b = np.load(f), np.load(os.path.join(d, f"branch_{w}_{k}", n + ".npy"))
            rel = float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(a))), 1e-300))
            line = f"  {n}: shape {a.shape} bit-identical {np.array_equal(a, b)} difference {rel:.3e}"
            if n == "cost_per_iteration":
                line += f", per iteration {float(np.max(np.abs(a - b) / np.abs(a))):.3e} relative"
                line += f", accept sequence equal {np.array_equal(np.diff(a) < 0, np.diff(b) < 0)}"
            print(line)
PY
rm -rf "$D"
