"""Time of the covariance (ba_gpu_covariance) on the REF problems of scripts/ref_sparse_bench.py: cfg3ref (800 keyframes) and
the long REF sequences of 3,000 and 10,000 keyframes, through the sparse Cholesky with the intrinsics border (solver 4).

Per problem, in one process: an LM solve of --steps exact steps (tolerances disabled) gives the ms per LM step; then the
covariance call at the solved state, warmed up, timed --repeats times with a host clock around the call (it returns after a
device synchronisation and the copies of its outputs) in two variants: cameras + intrinsics only, and with the points.
Prints JSON lines (device name and power limit first, from nvidia-smi in the same process).
--dump DIR also writes every output to DIR/<problem>.npz, for a bitwise comparison of two builds: both covariance variants,
camera pairs, and ba_gpu_covariance_blocks with every kind of pair (far camera pairs, camera-point, point-point and the
intrinsics against each).  --closures adds the 120-camera loop-closure problems of tests/irregular_problems.py.
Usage: python scripts/covariance_bench.py [--steps 10] [--repeats 5] [--sizes 3000,10000] [--out FILE] [--dump DIR] [--closures]"""
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
DUMP = None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if OUT:
        with open(OUT, "a") as f:
            f.write(line + "\n")


def requests(p, rng):
    """Camera pairs that share a point (for covariance(pairs=)) and pairs of every kind (for covariance_blocks)."""
    order = np.argsort(p.pt_idx, kind="stable")
    cam, pt = p.cam_idx[order], p.pt_idx[order]
    same = (pt[1:] == pt[:-1]) & (cam[1:] != cam[:-1])
    co = np.unique(np.sort(np.stack([cam[:-1][same], cam[1:][same]], axis=1), axis=1), axis=0)
    pairs = co[rng.choice(len(co), size=min(200, len(co)), replace=False)]
    cams, pts = rng.integers(0, p.n_cam, 12), rng.integers(0, p.n_pt, 12)
    blocks = [(("cam", 1), ("cam", p.n_cam - 1)), (("cam", 0), ("cam", p.n_cam // 2)), (("intr", 0), ("intr", 0))]
    blocks += [(("cam", int(a)), ("cam", int(b))) for a, b in zip(cams[:6], cams[6:])]
    blocks += [(("cam", int(a)), ("pt", int(b))) for a, b in zip(cams, pts)]
    blocks += [(("pt", int(a)), ("pt", int(b))) for a, b in zip(pts[:6], pts[6:])]
    blocks += [(("intr", 0), ("cam", int(a))) for a in cams[:4]] + [(("pt", int(a)), ("intr", 0)) for a in pts[:4]]
    return pairs, blocks


def dump(name, s, p):
    pairs, blocks = requests(p, np.random.default_rng(7))
    c = s.covariance(points=True, pairs=pairs)
    out = {k: v for k, v in c.items() if v is not None}
    out["cameras_intrinsics_cam"] = s.covariance(points=False)["cam"]
    out["blocks"] = np.concatenate([b.reshape(-1) for b in s.covariance_blocks(blocks)])
    os.makedirs(DUMP, exist_ok=True)
    np.savez(os.path.join(DUMP, name + ".npz"), **out)


def bench(name, p, steps, repeats):
    s = ba_b200.GpuSolver(use_depth_prior=1, optimize_intrinsics=1, solver=4, max_num_iterations=steps, function_tolerance=0.0,
                          gradient_tolerance=0.0, parameter_tolerance=0.0)
    s.upload(p)
    s.solve()  # (warm-up)
    s.upload(p)
    summ = s.solve()
    out = dict(what="covariance", problem=name, n_cam=p.n_cam, n_pt=p.n_pt, n_obs=p.n_obs, lm_iterations=int(summ.num_iterations),
               lm_ms_per_step=summ.solve_ms / max(summ.num_iterations, 1), spchol=s.spchol_info())
    for variant, points in (("cameras_intrinsics", False), ("with_points", True)):
        for _ in range(2):
            s.covariance(points=points)
        ts = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            c = s.covariance(points=points)
            ts.append((time.perf_counter() - t0) * 1e3)
        out[variant + "_ms"] = dict(median=float(np.median(ts)), min=float(np.min(ts)), all=ts)
    if DUMP:
        dump(name, s, p)
    out["cov_intr_diag"] = np.diag(c["intr"]).tolist()
    out["cov_cam_trace_median"] = float(np.median(np.trace(c["cam"], axis1=1, axis2=2)))
    s.close()
    emit(out)


def main():
    global OUT, DUMP
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--sizes", default="3000,10000")
    ap.add_argument("--out", default=None)
    ap.add_argument("--dump", metavar="DIR", default=None)
    ap.add_argument("--closures", action="store_true")
    a = ap.parse_args()
    OUT, DUMP = a.out, a.dump
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:  # (reported, not fatal)
        smi = "nvidia-smi unavailable: %s" % e
    emit(dict(what="device", nvidia_smi=smi))
    bench("cfg3ref", cfg3ref(), a.steps, a.repeats)
    if a.closures:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import irregular_problems
        for case in "abc":
            bench("closure_" + case, irregular_problems.closure_problem(case), a.steps, a.repeats)
    for n_kf in [int(x) for x in a.sizes.split(",") if x]:
        bench("ref_sequence_%d" % n_kf, long_sequence(n_kf), a.steps, a.repeats)


if __name__ == "__main__":
    main()
