"""Values of the block-sparse S: the fp64 DMMA kernel (k_sp_schur) against the per-lane-accumulator kernel it replaced
(k_sp_schur_simt, BA_SPS_SIMT=1), alternated in one process on the bench's workloads and options.

    python scripts/sp_schur_ab.py [--workloads cfg5,cfg4,cfg3] [--repeats 3] [--steps 20] [--warmup 5] [--out FILE]

Each repeat creates one solver per kernel (the switch is read at create) and runs them one after the other: W warm-up LM
iterations, then K timed ones on a fresh upload.  Per run it prints and appends a JSON line: LM it/s, the schur_complement
phase in ms per LM iteration, the final cost, and for the DMMA run the largest pose difference against the SIMT run of
the same repeat.  The first line names the device and its power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ba_b200  # noqa: E402
from bench import SOLVERS, WORKLOADS  # noqa: E402


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": q[0] if q else "unknown"}


def run(problem, mode, simt, K, W):
    if simt:
        os.environ["BA_SPS_SIMT"] = "1"
    else:
        os.environ.pop("BA_SPS_SIMT", None)
    opts = dict(use_depth_prior=mode[0], optimize_intrinsics=mode[1], function_tolerance=0.0, parameter_tolerance=0.0,
                gradient_tolerance=0.0, solver=SOLVERS["auto"])
    s = ba_b200.GpuSolver(max_num_iterations=W, **opts)
    os.environ.pop("BA_SPS_SIMT", None)
    try:
        s.upload(problem)
        s.solve()
        s.set_options(max_num_iterations=K)
        s.upload(problem)
        summ = s.solve()
        ph = s.phase_times()
        pose, _, _ = s.download()
        n = max(summ.num_iterations, 1)
        return dict(it_s=summ.num_iterations / (summ.solve_ms * 1e-3), schur_ms=ph.get("schur_complement", 0.0) / n,
                    phase_ms_per_step={k: v / n for k, v in ph.items()}, final_cost=summ.final_cost,
                    iterations=summ.num_iterations, solver_used=summ.solver_used), pose
    finally:
        s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg5,cfg4,cfg3")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_sp_schur_ab.jsonl"))
    a = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        def emit(d):
            line = json.dumps(d)
            print(line, flush=True)
            f.write(line + "\n")

        emit(device_line())
        for wl in a.workloads.split(","):
            w = WORKLOADS[wl]
            problem = ba_b200.synthetic.make_config(w["cfg"], scale=a.scale)
            for rep in range(a.repeats):
                ref_pose = None
                for simt in (True, False):
                    res, pose = run(problem, w["mode"], simt, a.steps, a.warmup)
                    res.update(workload=wl, repeat=rep, kernel="simt" if simt else "dmma")
                    if ref_pose is None:
                        ref_pose, ref_cost = pose, res["final_cost"]
                    else:
                        res["max_pose_diff_vs_simt"] = float(np.max(np.abs(pose - ref_pose)))
                        res["final_cost_rel_diff_vs_simt"] = abs(res["final_cost"] - ref_cost) / ref_cost
                    emit(res)


if __name__ == "__main__":
    main()
