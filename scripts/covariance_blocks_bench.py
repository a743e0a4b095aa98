"""Time of the covariance of chosen blocks (ba_gpu_covariance_blocks) on the REF problems of scripts/ref_sparse_bench.py:
cfg3ref (800 keyframes) and the long REF sequences of 3,000 and 10,000 keyframes, through the sparse Cholesky with the
intrinsics border (solver 4), next to ba_gpu_covariance and an LM step in the same process.

Per problem: an LM solve of --steps exact steps (tolerances disabled) gives the ms per LM step; then, at the solved state, each
case is warmed up and timed --repeats times with a host clock around the call (it returns after a device synchronisation and
the copy of its outputs):
    far_pair   one camera pair that shares no point (the first free camera and the last camera)
    row        one camera (the middle one) against every camera
    cam_pt     1,000 seeded camera-point blocks
    pt_pt      1,000 seeded point-point blocks
    n0         no request: the shared prologue (relinearisation, values of S, factorisation, X, T^-1) alone
    covariance ba_gpu_covariance with the points (the selected inversion)
Prints JSON lines (device name and power limit first, from nvidia-smi in the same process).
Usage: python scripts/covariance_blocks_bench.py [--steps 10] [--repeats 5] [--sizes 3000,10000] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import ba_b200  # noqa: E402
from ref_sparse_bench import cfg3ref, long_sequence  # noqa: E402

OUT = None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if OUT:
        with open(OUT, "a") as f:
            f.write(line + "\n")


def timed(fn, repeats):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return dict(median=float(np.median(ts)), min=float(np.min(ts)), all=ts)


def bench(name, p, steps, repeats):
    s = ba_b200.GpuSolver(use_depth_prior=1, optimize_intrinsics=1, solver=4, max_num_iterations=steps, function_tolerance=0.0,
                          gradient_tolerance=0.0, parameter_tolerance=0.0)
    s.upload(p)
    s.solve()  # (warm-up)
    s.upload(p)
    summ = s.solve()
    out = dict(what="covariance_blocks", problem=name, n_cam=p.n_cam, n_pt=p.n_pt, n_obs=p.n_obs,
               lm_iterations=int(summ.num_iterations), lm_ms_per_step=summ.solve_ms / max(summ.num_iterations, 1),
               spchol=s.spchol_info())
    rng = np.random.default_rng(0)
    free = [c for c in range(p.n_cam) if c != p.fixed_cam]
    mid = free[len(free) // 2]
    cases = dict(
        far_pair=[(("cam", free[0]), ("cam", p.n_cam - 1))],
        row=[(("cam", mid), ("cam", c)) for c in range(p.n_cam)],
        cam_pt=[(("cam", int(c)), ("pt", int(q))) for c, q in zip(rng.integers(0, p.n_cam, 1000), rng.integers(0, p.n_pt, 1000))],
        pt_pt=[(("pt", int(a)), ("pt", int(b))) for a, b in zip(rng.integers(0, p.n_pt, 1000), rng.integers(0, p.n_pt, 1000))],
        n0=[])
    for case, req in cases.items():
        out[case + "_ms"] = timed(lambda: s.covariance_blocks(req), repeats)
    out["covariance_ms"] = timed(lambda: s.covariance(points=True), repeats)
    out["far_pair_trace"] = float(np.trace(s.covariance_blocks(cases["far_pair"])[0]))
    s.close()
    emit(out)


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
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
    bench("cfg3ref", cfg3ref(), a.steps, a.repeats)
    for n_kf in [int(x) for x in a.sizes.split(",") if x]:
        bench("ref_sequence_%d" % n_kf, long_sequence(n_kf), a.steps, a.repeats)


if __name__ == "__main__":
    main()
