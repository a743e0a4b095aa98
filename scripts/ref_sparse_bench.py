"""REF cost (depth prior + free intrinsics): the dense explicit solver against the sparse Cholesky with the intrinsics border.

bench.py's method on one GPU: a fixed LM iteration count with the tolerances disabled, a warm-up solve, LM it/s from
summary.solve_ms.  Prints JSON lines:
  * device name and power limit (nvidia-smi query, same command);
  * cfg3ref at full size (800 keyframes), dense (solver 1) and sparse (solver 4) alternated three times each in this process:
    LM it/s, ms per step, the sparse path's phase times, final cost and pose differences between the two paths;
  * REF sequences of 3,000 and 10,000 keyframes, sparse only (beyond the dense path's 16,384 unknowns): LM it/s, upload ms,
    symbolic ms, tree depth, device memory in use after the upload.
Usage: python scripts/ref_sparse_bench.py [--steps 20] [--warmup 5] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ba_b200  # noqa: E402

syn = ba_b200.synthetic
OUT = None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if OUT:
        with open(OUT, "a") as f:
            f.write(line + "\n")


def cfg3ref(scale=1.0):
    c3 = syn.CONFIGS[3]
    n_kf = max(4, int(round(c3["n_kf"] * scale)))
    seq = syn.make_tum_sequence(n_kf, max(8, int(round(c3["n_lm"] * scale))), max(24, int(round(c3["n_obs"] * scale))),
                                syn.SEED_BASE + 3)
    return syn.window_problem(seq, 0, n_kf - 1).problem


def long_sequence(n_kf):
    # cfg3ref's density per keyframe: 75 landmarks and 500 observations per keyframe
    seq = syn.make_tum_sequence(n_kf, 75 * n_kf, 500 * n_kf, syn.SEED_BASE + 7)
    return syn.window_problem(seq, 0, n_kf - 1).problem


def timed_solve(p, solver, steps, warmup):
    import torch
    s = ba_b200.GpuSolver(use_depth_prior=1, optimize_intrinsics=1, solver=solver, max_num_iterations=warmup,
                          function_tolerance=0.0, gradient_tolerance=0.0, parameter_tolerance=0.0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.upload(p)
    torch.cuda.synchronize()
    upload_ms = (time.perf_counter() - t0) * 1e3
    free, total = torch.cuda.mem_get_info()
    if warmup > 0:
        s.solve()
    s.set_options(max_num_iterations=steps)
    s.upload(p)
    summ = s.solve()
    pose = s.download()[0].copy()
    out = dict(solver_used=int(summ.solver_used), lm_iterations=int(summ.num_iterations),
               lm_it_per_s=summ.num_iterations / (summ.solve_ms * 1e-3), ms_per_step=summ.solve_ms / max(summ.num_iterations, 1),
               final_cost=summ.final_cost, initial_cost=summ.initial_cost, upload_ms=upload_ms,
               device_mem_used_after_upload_GB=(total - free) / 1e9, phase_ms_per_step=None, spchol=None)
    if summ.solver_used == ba_b200.capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY:
        out["phase_ms_per_step"] = {k: v / max(summ.num_iterations, 1) for k, v in s.phase_times().items()}
        info = s.spchol_info()
        out["spchol"] = dict(nodes=info["nodes"], levels=info["levels"], max_own=info["max_own"], max_border=info["max_border"],
                             symbolic_ms=info["symbolic_us"] / 1e3, gflop_per_factorisation=info["flops"] / 1e9)
    s.close()
    return out, pose


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sizes", default="3000,10000")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    OUT = a.out
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:  # (reported, not fatal)
        smi = "nvidia-smi unavailable: %s" % e
    emit(dict(what="device", nvidia_smi=smi))

    p = cfg3ref()
    runs = {1: [], 4: []}
    poses = {}
    for r in range(a.repeats):
        for solver in (1, 4):
            o, pose = timed_solve(p, solver, a.steps, a.warmup)
            runs[solver].append(o)
            poses[solver] = pose
            emit(dict(what="cfg3ref", repeat=r, solver=solver, n_cam=p.n_cam, n_obs=p.n_obs, reduced_dim=6 * (p.n_cam - 1) + 4, **o))
    d, s_ = runs[1][-1], runs[4][-1]
    drot = ba_b200.se3.rot_angle(poses[1][:, :4], poses[4][:, :4])
    emit(dict(what="cfg3ref_summary", steps=a.steps,
              dense_lm_it_per_s_median=float(np.median([x["lm_it_per_s"] for x in runs[1]])),
              sparse_lm_it_per_s_median=float(np.median([x["lm_it_per_s"] for x in runs[4]])),
              dense_ms_per_step_median=float(np.median([x["ms_per_step"] for x in runs[1]])),
              sparse_ms_per_step_median=float(np.median([x["ms_per_step"] for x in runs[4]])),
              final_cost_dense=d["final_cost"], final_cost_sparse=s_["final_cost"],
              final_cost_rel_diff=abs(d["final_cost"] - s_["final_cost"]) / d["final_cost"],
              max_translation_diff=float(np.max(np.linalg.norm(poses[1][:, 4:] - poses[4][:, 4:], axis=1))),
              max_rotation_diff_rad=float(np.max(drot))))
    for n_kf in [int(x) for x in a.sizes.split(",") if x]:
        q = long_sequence(n_kf)
        o, _ = timed_solve(q, 0, a.steps, a.warmup)  # AUTO: beyond the dense limit -> the sparse Cholesky
        emit(dict(what="long_ref_sequence", n_kf=n_kf, n_pt=q.n_pt, n_obs=q.n_obs, reduced_dim=6 * (q.n_cam - 1) + 4, **o))


if __name__ == "__main__":
    main()
