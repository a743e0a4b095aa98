#!/bin/bash
# N ranks on one box: multi-GPU parity tests, then the cfg5 bench line with the distributed factorisation
cd "$GRAFT_REPO_ROOT" || exit 1
mkdir -p gpurun_out
N=$(nvidia-smi -L | wc -l)
timeout 400 python -m pytest tests/test_gpu_multi.py -m gpu -x -q -k "${MULTI_K:-sparse or auto or implicit}" > gpurun_out/r2_multi_tests_n${N}.log 2>&1; echo rc=$? >> gpurun_out/r2_multi_tests_n${N}.log
tail -n 5 gpurun_out/r2_multi_tests_n${N}.log
for mode in ${MODES:-dist}; do
  BA_SPCHOL_DEBUG=1 timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 2954$N bench.py --gpus $N --steps 20 --warmup 5 > gpurun_out/r2_bench_cfg5_n${N}_$mode.log 2>&1
  echo "N=$N $mode rc=$?"
  grep "^\[spchol\]" gpurun_out/r2_bench_cfg5_n${N}_$mode.log | head -n 2
  python - gpurun_out/r2_bench_cfg5_n${N}_$mode.log <<'PY'
import json,sys
for l in open(sys.argv[1]):
    if l.startswith('{'):
        d=json.loads(l); print(d["n_gpus"], d["value"], d["ms_per_step"], "e2e", d["e2e"]["value"], d["detail"]["solver"][:40], d["final_cost"], d.get("parity_vs_n1"))
        print({k: round(v,3) for k,v in d.get("phase_ms_per_step",{}).items()})
PY
done
