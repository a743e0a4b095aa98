"""What each solve path launches and computes, for comparing two builds of the library bit for bit.

    python scripts/plan_trace.py OUT            # run every case, write OUT/plan_trace.json and OUT/<case>.npz
    python scripts/plan_trace.py --compare A B  # per case: same plan, launches, kernel sequence per stream, output bits

Every case uploads one seeded problem, solves a fixed number of LM iterations with every tolerance 0, then calls the
covariance entry points and the Schur hooks where its cost mode allows them.  A second pass runs the same cases under
torch.profiler (CUDA activities) and records, per CUDA stream, the ordered kernels with their grid, block and shared memory.
Streams are numbered per case in the order they first run a kernel."""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import ba_b200, mode_opts  # noqa: E402
from test_gpu_edge_cases import _wide_covisibility  # noqa: E402

syn = ba_b200.synthetic
ITERS = 3


def _with_depth(p):
    q = p.copy()
    q.depth = syn.camera_point(q.pose7[q.cam_idx], q.pt3[q.pt_idx])[:, 2].copy()
    return q


def cases():
    """(name, problem, gpu options, environment, calls) for one or more cases per solve path."""
    cfg1 = syn.make_config(1)
    seq = _with_depth(syn.make_config(3, scale=0.05))
    wide = _wide_covisibility()
    cov = ("covariance",)
    out = [
        ("cfg1_ref_windowed", cfg1, mode_opts("REF")[0], {}, cov),
        ("seq_ref_blocked_dense", seq, mode_opts("REF")[0], {}, cov),
        ("seq_ref_bordered", seq, mode_opts("REF", solver=4)[0], {}, cov),
        ("seq_depth_bordered", seq, mode_opts("DEPTH", solver=4)[0], {}, cov),
        ("seq_ns_sparse_chol", seq, mode_opts("NS", solver=4)[0], {}, ("schur",)),
        ("seq_ns_sparse_chol_2parts", seq, mode_opts("NS", solver=4)[0], {"BA_SPCHOL_PARTS": "2"}, ("schur",)),
        ("seq_ns_pcg_steps", seq, dict(mode_opts("NS", solver=3)[0], persistent_pcg=0), {}, ("schur",)),
        ("seq_ns_pcg_persistent", seq, dict(mode_opts("NS", solver=3)[0], persistent_pcg=1), {}, ("schur",)),
        ("wide_ns_auto_pcg_fallback", wide, mode_opts("NS")[0], {}, ("schur",)),
    ]
    for store, name in ((0, "tiled"), (2, "factored"), (1, "planes")):
        out.append((f"seq_ns_implicit_{name}", seq, mode_opts("NS", solver=2, jacobian_store=store)[0], {}, ("schur",)))
    out.append(("seq_depth_implicit", seq, mode_opts("DEPTH", solver=2)[0], {}, ("schur",)))
    return out


def run_case(p, opts, env, calls):
    """-> (record, arrays)"""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    s = ba_b200.GpuSolver(max_num_iterations=ITERS, function_tolerance=0.0, gradient_tolerance=0.0, parameter_tolerance=0.0,
                          **opts)
    try:
        s.upload(p)
        summ = s.solve()
        pose, pt, intr = s.download()
        arrays = dict(pose=pose, pt=pt, intr=intr, cost=np.array([summ.initial_cost, summ.final_cost]),
                      trace=np.array([[float(v) for v in r.values()] for r in s.trace()]))
        rec = dict(solver_used=int(summ.solver_used), jacobian_store_used=s.jacobian_store_used(),
                   kernel_launches=int(summ.kernel_launches), num_iterations=int(summ.num_iterations),
                   sparse_blocks=s.sparse_stats()[1], tree_nodes=s.spchol_info().get("nodes", 0))
        rng = np.random.default_rng(0)
        if "schur" in calls:
            x = rng.normal(size=6 * p.n_cam)
            arrays["schur_matvec"] = s.schur_matvec(1e4, x)
            if rec["tree_nodes"]:
                arrays["schur_solve"] = s.schur_solve(1e4, x)
        if "covariance" in calls:
            pairs = np.array([[1, 1], [1, 2], [2, 3]], dtype=np.int32)
            c = s.covariance(points=True, pairs=pairs)
            arrays.update({"cov_" + k: v for k, v in c.items() if v is not None})
            far = p.n_cam - 1
            blocks = s.covariance_blocks([(("cam", 1), ("cam", far)), (("cam", 2), ("pt", 5)), (("pt", 3), ("pt", 7)),
                                          (("intr", 0), ("cam", 3))])
            arrays.update({f"covblock_{i}": b for i, b in enumerate(blocks)})
            rec["launches_after_covariance"] = int(s.lib.ba_gpu_launch_count(s._ctx))
        return rec, arrays
    finally:
        s.close()
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def kernel_sequences(p, opts, env, calls):
    """Ordered kernels per stream of one case, under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_case(p, opts, env, calls)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, "trace.json")
        prof.export_chrome_trace(f)
        with open(f) as fh:
            ev = json.load(fh)["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    streams, seq = {}, {}
    for e in kern:
        a = e.get("args", {})
        sid = streams.setdefault(a.get("stream", e.get("tid")), len(streams))
        seq.setdefault(str(sid), []).append([e["name"], a.get("grid"), a.get("block"), a.get("shared memory")])
    return seq


def run_all(out):
    os.makedirs(out, exist_ok=True)
    result = {}
    all_cases = cases()
    for name, p, opts, env, calls in all_cases:
        rec, arrays = run_case(p, opts, env, calls)
        np.savez(os.path.join(out, name + ".npz"), **arrays)
        result[name] = rec
        print(name, json.dumps(rec), flush=True)
    for name, p, opts, env, calls in all_cases:
        seq = kernel_sequences(p, opts, env, calls)
        result[name]["streams"] = seq
        print(name, "kernels per stream:", {k: len(v) for k, v in seq.items()}, flush=True)
    with open(os.path.join(out, "plan_trace.json"), "w") as fh:
        json.dump(result, fh, indent=1)


def compare(a, b):
    ra = json.load(open(os.path.join(a, "plan_trace.json")))
    rb = json.load(open(os.path.join(b, "plan_trace.json")))
    ok_all = True
    for name in ra:
        x, y = ra[name], rb.get(name)
        if y is None:
            print(f"{name}: missing in {b}")
            ok_all = False
            continue
        plan = all(x[k] == y[k] for k in x if k != "streams")
        seq = x["streams"] == y["streams"]
        na, nb = np.load(os.path.join(a, name + ".npz")), np.load(os.path.join(b, name + ".npz"))
        bits = sorted(na.files) == sorted(nb.files) and all(np.array_equal(na[k], nb[k]) for k in na.files)
        n_k = sum(len(v) for v in x["streams"].values())
        print(f"{name}: solver {x['solver_used']} store {x['jacobian_store_used']} launches {x['kernel_launches']} | "
              f"same plan and launches {plan}, same kernel sequence {seq} ({len(x['streams'])} streams, {n_k} kernels), "
              f"same bits {bits} ({len(na.files)} arrays)")
        ok_all &= plan and seq and bits
    print("ALL SAME" if ok_all else "DIFFERENCES")
    return 0 if ok_all else 1


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    run_all(args.out)
