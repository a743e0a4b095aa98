#!/bin/bash
# partitioned sparse Cholesky on one GPU: bit-identity tests, then the linear solve with N parts run one after the other
cd "$GRAFT_REPO_ROOT" || exit 1
mkdir -p gpurun_out
timeout 300 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "spchol" > gpurun_out/r2_parts_tests.log 2>&1; echo rc=$? >> gpurun_out/r2_parts_tests.log
tail -n 4 gpurun_out/r2_parts_tests.log
{
for n in 2 4 8; do
  echo "parts $n (all parts on this GPU)"; BA_SPCHOL_DEBUG=1 BA_SPCHOL_PARTS=$n timeout 120 python scripts/phase_probe.py 5 10 4 2>&1 | tail -n 2
done
} > gpurun_out/r2_parts_probe.log 2>&1
cat gpurun_out/r2_parts_probe.log
