#!/usr/bin/env python
"""bench.py -- LM iterations/s (and Jacobian-eval observations/s) of the B200 BA
solver on BASELINE.json's synthetic configs, with the kernel roofline and the
CPU baseline beside it.

  python bench.py --gpus N --steps K --warmup W [--workload cfg5] [--impl reference] [--dump-outputs DIR]

A "step" is one Levenberg-Marquardt iteration (linearisation + Schur linear
solve + step evaluation) of the fixed-iteration-count solve on the workload.
--dump-outputs DIR writes what the timed solve returned (poses, points,
intrinsics, cost per iteration) as DIR/<name>.npy; the synthetic inputs are
seeded, so two builds run with the same arguments can be compared array by
array.
Default workload: cfg5 of BASELINE.json (10k cameras, 2M points, 8M
observations, reprojection only, implicit-Schur PCG) -- the config the metric's
"1/2/4/8 B200" refers to; it fits one GPU.  With N > 1 (torchrun, one rank per
GPU) the points and their observations are sharded across ranks and the
camera-sized partial vectors are combined with NCCL all-reduce: total work is
fixed => "scaling": "strong".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg1": dict(cfg=1, mode=(1, 1), desc="7-keyframe TUM-shaped window, 500 landmarks, 3000 obs, REF cost, explicit Schur + Cholesky"),
    "cfg2": dict(cfg=2, mode=(1, 1), desc="sliding 20-keyframe windows over 800 keyframes, REF cost, explicit Schur + Cholesky"),
    "cfg3": dict(cfg=3, mode=(0, 0), desc="global BA 800 keyframes, 60k landmarks, 400k obs, NS cost; linear solver in force: detail.solver (BASELINE.json names implicit-Schur PCG for this config: --solver implicit)"),
    "cfg3ref": dict(cfg=3, mode=(1, 1), desc="the reference's global optimisation: 800 keyframes, 60k landmarks, 400k obs, REF cost (depth prior + "
                                             "free intrinsics), dense explicit Schur + blocked Cholesky (exact LM step)"),
    "cfg4": dict(cfg=4, mode=(0, 0), desc="BAL-shaped loop 1723 cameras, 156k points, 680k obs, NS cost; linear solver in force: detail.solver (BASELINE.json names implicit-Schur PCG for this config: --solver implicit)"),
    "cfg5": dict(cfg=5, mode=(0, 0), desc="large synthetic 10k cameras, 2M points, 8M obs, NS cost; linear solver in force: detail.solver (BASELINE.json names implicit-Schur PCG for this config: --solver implicit)"),
}
# Algorithmic bytes per launch (DESIGN.md section 4): NS mode, fp64, int32 indices.
# (per observation, per point, per camera) for every Jacobian store; the dominant
# kernel's figure is what roofline.achieved is computed from.
BYTES = {
    # materialised planes: r 16 + Jc 96 + Jp 48 written, uv 16 + idx 8 + point 24 read
    "planes": {"linearize": (208, 0, 0), "pass1": (148, 72, 48), "pass2": (172, 0, 96)},
    # factored store: r 16 + g 32 written; passes read g 32 + idx 4 (+ 32 B gather of t in pass 2)
    "factored": {"linearize": (96, 0, 0), "pass1": (36, 108, 0), "pass2": (68, 0, 96)},
    # tile-fused single pass: g 32 + packed idx 4 per obs, Vs 48 + rowptr 4 per point
    "tiled": {"linearize": (96, 0, 0), "fused": (36, 52, 0)},
}
STORE_NAME = {1: "planes", 2: "factored", 3: "tiled"}
SOLVERS = {"auto": 0, "implicit": 2, "sparse": 3, "cholesky": 4}
SOLVER_NAME = {1: "dense explicit Schur + Cholesky", 2: "implicit-Schur PCG", 3: "block-sparse explicit Schur + persistent PCG",
               4: "block-sparse explicit Schur + exact sparse Cholesky (supernodal multifrontal, nested dissection)"}
# DRAM traffic per launch from the committed `ncu --set full` captures (dram__bytes_read.sum + dram__bytes_write.sum),
# cfg5 only; (substring of the roofline kernel name) -> (bytes per launch, source)
NCU_TRAFFIC_CFG5 = {
    "block-CSR product": (1.36e6, "profiles/r01_ncu_full_kernels_cfg5.csv: k_pcg_sparse_persistent moved 52.8 MB read + 1.4 MB written "
                                  "over 40 PCG iterations: S (45 MB) is L2-resident (L2 hit rate 96.0 %)"),
    "linearize (factored": (567.3e6, "profiles/r01_ncu_full_linearize_cfg5.csv: 240.6 MB read + 326.7 MB written (the 24 B/obs point "
                                     "gathers hit L2)"),
    "linearize (tiled": (567.3e6, "profiles/r01_ncu_full_linearize_cfg5.csv (same kernel as the factored store)"),
    "kt_schur_fused": (408.3e6, "profiles/r01_ncu_full_kernels_cfg5.csv: 398.7 MB read + 9.6 MB written (algorithmic 392 MB)"),
    "schur_pass1 (two-pass, factored": (492.4e6, "profiles/r01_ncu_full_kernels_cfg5.csv: 444.1 MB read + 48.3 MB written"),
    "schur_pass2 (two-pass, factored": (366.6e6, "profiles/r01_ncu_full_kernels_cfg5.csv: 361.8 MB read + 4.8 MB written (the t_p gather hits L2)"),
    "schur_pass1 (two-pass, planes": (1347e6, "profiles/r01_ncu_full_schur_cfg5.csv"),
    "schur_pass2 (two-pass, planes": (1313e6, "profiles/r01_ncu_full_schur_cfg5.csv"),
}


def ncu_traffic(workload, kernel_name):
    if workload != "cfg5":
        return None, None
    for key, (b, src) in NCU_TRAFFIC_CFG5.items():
        if key in kernel_name:
            return b, src
    return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def oracle_problem(problem):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ora
    return ora, ora.Problem(problem.pose7, problem.pt3, problem.cam_idx, problem.pt_idx, problem.uv2, problem.depth, problem.intr,
                            problem.intr_prior, problem.fixed_cam)


def cpu_reference_run(problem, mode, iters, threads, warmup=0):
    """RUNS the CPU oracle (oracle/ba_oracle.c: the restatement of the reference's cost functors + Ceres 2.0.0 LM) on the
    same problem for `iters` LM iterations with the reference's own linear solver setting -- SPARSE_SCHUR
    (headers/BundleAdjustmentConfig.h:62): explicit reduced camera matrix in envelope storage + sparse Cholesky, exact
    step -- on `threads` OpenMP threads, tolerances disabled.  Nothing is extrapolated: value = iterations / wall seconds
    of that solve.  `warmup` > 0 runs that many iterations on a copy first (untimed)."""
    ora, op = oracle_problem(problem)
    kw = dict(use_depth_prior=mode[0], optimize_intrinsics=mode[1], solver=2, num_threads=threads, function_tolerance=0.0,
              parameter_tolerance=0.0, gradient_tolerance=0.0)
    if warmup > 0:
        ora.solve(op.copy(), ora.default_options(max_num_iterations=warmup, **kw))
    t0 = time.time()
    rc, s, tr = ora.solve(op, ora.default_options(max_num_iterations=iters, **kw), trace_cap=iters + 8)
    wall = time.time() - t0
    n = max(1, int(s.num_iterations))
    return {"value": n / wall, "unit": "LM iterations/s", "cores": threads, "kind": "port",
            "sample": "oracle/ba_oracle.c (C restatement of the reference's cost functors and of Ceres 2.0.0's trust-region loop; "
                      "linear solver = the reference's SPARSE_SCHUR setting: explicit S in envelope storage + sparse Cholesky, exact "
                      "step), OpenMP %d threads, %d LM iterations of the SAME problem actually run in %.2f s wall (nothing "
                      "extrapolated); Ceres itself cannot be built in this image" % (threads, n, wall),
            "lm_iterations": n, "seconds": wall, "seconds_linearize": s.seconds_linearize, "seconds_linear_solve": s.seconds_linear_solve,
            "final_cost": s.final_cost, "rc": rc,
            "jacobian_obs_per_s": problem.n_obs * (n + 1) / max(s.seconds_linearize, 1e-12)}


def bench_config(args, wl, full, world, K):
    """The workload description both arms print (identical for --impl b200 and --impl reference)."""
    flush = full.n_obs * 36 < 512e6
    return {"workload": args.workload + ": " + wl["desc"], "n_cam": int(full.n_cam), "n_pt": int(full.n_pt), "n_obs": int(full.n_obs),
            "scale": args.scale,
            "cost_model": {(0, 0): "NS: reprojection residuals, fixed intrinsics", (1, 1): "REF: reprojection + depth prior + free "
                           "intrinsics with prior (the reference's cost)"}.get(tuple(wl["mode"]), str(wl["mode"])),
            "step": "one Levenberg-Marquardt iteration of a fixed-iteration-count solve (tolerances disabled)", "lm_iterations": K,
            "linear_solver_requested": args.solver if wl["mode"] == (0, 0) else "auto",
            "parallelism": "single GPU" if world == 1 else "points and their observations sharded over %d GPUs, cameras replicated" % world,
            "l2": ("streaming inputs larger than L2 (factored store %.0f MB per pass); L2-resident structures (block-sparse S, fronts "
                   "of the sparse Cholesky) are timed as they run inside the solve" % (full.n_obs * 36 / 1e6)) if not flush
                  else "L2 flushed (512 MiB write) between timed launches of the kernel hooks"}


def kernel_rooflines(ba_b200, s, problem, wl, solver_used, flush, peak):
    """Times the hot kernels of the uploaded problem (ba_gpu_time_kernel: CUDA events on the solver
    stream) and prices them with the algorithmic bytes of the store in force."""
    cap = ba_b200.capi
    n_o, n_p, n_c = problem.n_obs, problem.n_pt, problem.n_cam
    store = STORE_NAME.get(s.jacobian_store_used(), "planes")
    bt = BYTES[store]

    def nbytes(t):
        return t[0] * n_o + t[1] * n_p + t[2] * n_c

    roof = {}
    ms_lin = s.time_kernel(cap.BA_KERNEL_LINEARIZE, 3, 20, flush)
    dom = "linearize (%s store)" % store
    roof[dom] = (nbytes(bt["linearize"]), ms_lin)
    if solver_used in (3, 4):
        # block-CSR product = phase I of the persistent PCG kernel: every stored (upper) block is read twice
        # (as itself and transposed): 288 B block + 8 B entry + 48 B gathered vector per row entry
        n_ent, n_blk = s.sparse_stats()
        ms_mv = s.time_kernel(cap.BA_KERNEL_SCHUR_MATVEC, 3, 20, False)
        dom = "block-CSR product (k_bsr_spmv = phase I of the persistent PCG kernel)"
        roof[dom] = (n_ent * (288 + 8 + 48) + n_c * 96, ms_mv)
    elif wl["mode"] == (0, 0):
        two = "factored" if store == "tiled" else store
        if store == "tiled":
            ms_f = s.time_kernel(cap.BA_KERNEL_SCHUR_MATVEC, 3, 20, flush)
            dom = "kt_schur_fused (tile-fused product)"
            roof[dom] = (nbytes(bt["fused"]), ms_f)
        bt2 = BYTES[two]
        ms_p1 = s.time_kernel(cap.BA_KERNEL_SCHUR_PASS1, 3, 20, flush)
        ms_p2 = s.time_kernel(cap.BA_KERNEL_SCHUR_PASS2, 3, 20, flush)
        roof["schur_pass1 (two-pass, %s)" % two] = (nbytes(bt2["pass1"]), ms_p1)
        roof["schur_pass2 (two-pass, %s)" % two] = (nbytes(bt2["pass2"]), ms_p2)
        if store != "tiled":
            dom = max((k for k in roof if k.startswith("schur_pass")), key=lambda k: roof[k][1])
    kernels = {k: {"bytes": b, "ms": ms, "achieved_gbs": b / ms / 1e6, "frac": b / ms / 1e6 / peak} for k, (b, ms) in roof.items()}
    if n_o == 8000000:  # the ncu captures are of cfg5 on one GPU
        for k in kernels:
            kernels[k]["ncu_dram_bytes"] = ncu_traffic("cfg5", k)[0]
    return kernels, dom, store, ms_lin


FP64_NOMINAL_TFLOPS = 40.0  # B200 vector fp64, nominal (MEASURED_PEAKS.json holds no fp64 figure)
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures of this round
# (profiles/r02_ncu_full_cfg5.csv), config 5 on one GPU
_NCU_SRC = "ncu --set full, profiles/r02_ncu_full_cfg5.csv / r02_ncu_cfg5_summary.txt (one GPU, cold cache, per launch)"
NCU_TRAFFIC_R02_CFG5 = {
    # k_sp_schur 646.4 MB read + 45.0 MB written (the gathers of the 3.0 GB of requested operands hit L1 83 % / L2 52 %)
    "schur_complement": (691.4e6, _NCU_SRC),
    # k_spchol_tree 143.6 MB read + 168.7 MB written (fronts and update matrices mostly stay in L2)
    "linear_solve": (312.3e6, _NCU_SRC),
    # kf_linearize<0> 567.7 + kf_pt_blocks 617.4 + kf_linearize<1> 569.6 + kf_cam_blocks 394.0 MB
    "accept_relinearize": (2148.7e6, _NCU_SRC),
    # kf_schur_pass1<1,0> 582.6 + kf_model_cost 518.2 + k_cost 245.3 MB
    "back_substitution_model_cost": (1346.1e6, _NCU_SRC),
    "point_inverse": (445.2e6, _NCU_SRC),
    "reduced_rhs": (369.0e6, _NCU_SRC),
}


def executed_roofline(workload, phase_ms, n_iter, solver_used, full, n_pairs, n_ent, spchol, pcg_total, peak, peak_src):
    """The roofline entry of the phase that took the largest share of the timed solve AS EXECUTED (CUDA events recorded on
    the solver stream at the phase boundaries while the solve ran, ba_gpu_phase_times), with the algorithmic bytes (or
    flops) of the kernels of that phase."""
    if not phase_ms or n_iter <= 0:
        return None, {}
    per = {k: v / n_iter for k, v in phase_ms.items()}
    n_o, n_p, n_c = full.n_obs, full.n_pt, full.n_cam
    total = sum(per.values())
    table = {}

    def hbm(name, kernels, nbytes, ms, limiter, note=None):
        # `bound` is the contract's enum (every phase of this path moves bytes: "hbm", against the measured copy bandwidth);
        # `limiter` says what actually holds the phase back when that is not bandwidth
        table[name] = {"kernels": kernels, "bound": "hbm", "limiter": limiter, "bytes": nbytes, "ms": ms,
                       "share_of_step": ms / total if total else None,
                       "achieved": nbytes / ms / 1e6 if ms > 0 else None, "peak": peak, "unit": "GB/s",
                       "frac": nbytes / ms / 1e6 / peak if ms > 0 else None, "note": note}

    if solver_used in (3, 4):
        hbm("schur_complement", "k_sp_schur (+ k_sp_add_diag)", 124.0 * n_pairs, per.get("schur_complement", 0.0),
            "latency of dependent gathers (pair -> two observation records + Vs) at 8 warps per SM; operands mostly hit L1 / L2",
            "124 B per same-point observation pair: pair 8 + point id 4 + two factored records 64 + Vs 48")
    if solver_used == 4 and spchol:
        # (one persistent launch does factorisation and both substitutions; with BA_SPCHOL_LEVELS=1 the backward
        # substitution shows up as its own phase -- added here either way)
        ms = per.get("linear_solve_factor_or_pcg", 0.0) + per.get("linear_solve_substitution", 0.0)
        # algorithmic bytes of one factorisation + both substitutions, 288 B per 6x6 block: stored blocks of S read, panels
        # written, their border rows read again by the update items, update matrices written and read (extend-add), panels
        # read by the backward substitution
        n_sblk = spchol.get("s_blocks", 0)
        blocks = n_sblk + 3 * spchol.get("panel_blocks", 0) + 2 * spchol.get("update_blocks", 0)
        flops = spchol.get("flops", 0)
        hbm("linear_solve", "k_spchol_rhs, k_spchol_tree (factor / update / substitution items of the supernodal tree, one persistent launch)",
            288.0 * blocks, ms, "latency: dependent chain of %d tree levels on single SMs (fp64); the data stays in L2" % spchol.get("levels", 0),
            "288 B x (stored blocks of S + 3 x panel blocks + 2 x update-matrix blocks); %d nodes in %d levels, critical path %d block "
            "operations of %d total; fp64: %.2f GFLOP -> %.2f TFLOP/s of nominal %.0f"
            % (spchol.get("nodes", 0), spchol.get("levels", 0), spchol.get("critical_path_block_ops", 0), flops // 432, flops / 1e9,
               flops / ms / 1e9 if ms > 0 else 0.0, FP64_NOMINAL_TFLOPS))
        table["linear_solve"]["flops"] = flops
    elif solver_used == 3 and pcg_total > 0:
        ms = per.get("linear_solve_substitution", 0.0) + per.get("linear_solve_factor_or_pcg", 0.0)
        hbm("pcg", "k_pcg_sparse_persistent (all PCG iterations of a step)", (n_ent * 344.0 + n_c * 96.0) * pcg_total / n_iter, ms,
            "L2 bandwidth / latency (S is L2-resident)", "per PCG iteration: 288 B block + 8 B entry + 48 B gathered vector per row entry")
    # factored store: kf_linearize x2 (96 B/obs each), kf_pt_blocks (48 B/obs + 96 B/pt), kf_cam_blocks (48 B/obs), state copies
    hbm("accept_relinearize", "k_accept, kf_linearize<0>, kf_pt_blocks, kf_linearize<1>, kf_cam_blocks, k_cam_blocks_fin, k_state_norms",
        (96.0 + 96.0 + 48.0 + 48.0) * n_o + (96.0 + 2 * 48.0) * n_p + (288.0 + 2 * 112.0) * n_c, per.get("accept_relinearize", 0.0), "bandwidth + L1 request rate of the point-major gathers")
    hbm("back_substitution_model_cost", "k_pack_camx, kf_schur_pass1<1,0>, kf_model_cost, k_candidate, k_cost",
        (48.0 + 48.0 + 44.0) * n_o + (48.0 + 32.0 + 24.0 + 48.0) * n_p, per.get("back_substitution_model_cost", 0.0) + per.get("candidate_cost", 0.0),
        "bandwidth + L1 request rate of the point-major gathers")
    hbm("point_inverse", "kf_point_inverse", (48.0 + 24.0 + 24.0 + 24.0 + 48.0 + 48.0 + 32.0) * n_p, per.get("point_inverse", 0.0), "bandwidth")
    hbm("reduced_rhs", "kf_schur_pass2", 68.0 * n_o + 96.0 * n_c, per.get("reduced_rhs", 0.0), "bandwidth")
    live = {k: v for k, v in table.items() if v["ms"] and v["ms"] > 0}
    if not live:
        return None, table
    if workload == "cfg5":
        for k, v in table.items():
            if k in NCU_TRAFFIC_R02_CFG5:
                v["traffic"] = NCU_TRAFFIC_R02_CFG5[k][0]
    dom = max(live, key=lambda k: live[k]["ms"])
    d = live[dom]
    traffic = NCU_TRAFFIC_R02_CFG5.get(dom) if workload == "cfg5" else None
    roof = {"kernel": "%s: %s" % (dom, d["kernels"]), "bound": d["bound"], "limiter": d.get("limiter"), "achieved": d["achieved"],
            "peak": d["peak"], "unit": d["unit"],
            "frac": d["frac"], "traffic": traffic[0] if traffic else None, "traffic_source": traffic[1] if traffic else None,
            "peak_source": peak_src, "note": d.get("note"), "share_of_step": d["share_of_step"],
            "ms_per_step": d["ms"],
            "timing": "CUDA events recorded on the solver stream at the phase boundaries of every LM iteration of the timed solve "
                      "(ba_gpu_phase_times): the phase as executed, not a stand-alone launch",
            "bytes" if d["unit"] == "GB/s" else "flops": d.get("bytes", d.get("flops"))}
    return roof, table


def parity_vs_n1(workload, scale, solver_used, trace):
    """Final cost / accept sequence of this run against the committed single-GPU trace of the same workload
    (tests/golden/bench_trace.json, written by --write-golden on one GPU)."""
    path = os.path.join(ROOT, "tests", "golden", "bench_trace.json")
    if not os.path.exists(path) or scale != 1.0:
        return None
    g = json.load(open(path)).get("%s/solver%d" % (workload, solver_used))
    if not g:
        return None
    n = min(len(trace), len(g["cost"]))
    rel = max(abs(trace[i]["cost"] - g["cost"][i]) / abs(g["cost"][i]) for i in range(n))
    same = [t["step_is_successful"] for t in trace[:n]] == g["successful"][:n]
    return {"iterations_compared": n - 1, "max_rel_cost_diff": rel, "accept_sequence_equal": same, "ok": bool(same and rel <= 1e-8),
            "tolerance": 1e-8, "golden": "tests/golden/bench_trace.json (%s, 1 GPU)" % g.get("when", "?")}


def pinned_copy(a):
    """numpy view of pinned host memory holding a copy of `a` (H2D at full PCIe speed)."""
    import torch
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy()


def n_blk_all(s):
    return s.sparse_stats()[1]


DUMP_BYTES = 64e6


def write_outputs(path, arrays):
    """Writes every array as path/<name>.npy in float64.  When they would pass DUMP_BYTES together, the largest is cut
    to a fixed, seeded sample of its rows (in row order) so that the files stay comparable between runs."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        big = max(arrays, key=lambda k: arrays[k].nbytes)
        a = arrays[big]
        keep = int((DUMP_BYTES - (total - a.nbytes)) // (a.nbytes // a.shape[0]))
        arrays[big] = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; reported in config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--solver", default="auto", choices=sorted(SOLVERS),
                    help="large NS-mode workloads: auto = the library's choice (block-sparse explicit S on one GPU, "
                         "sharded implicit on several), implicit = matrix-free two/one-pass product, sparse = block-sparse S")
    ap.add_argument("--with-implicit-path", action="store_true",
                    help="single GPU: also time the matrix-free implicit-Schur PCG solver on the same problem (adds its W + K LM iterations)")
    ap.add_argument("--write-golden", action="store_true", help="single GPU: store this run's LM trace as the reference of parity_vs_n1")
    ap.add_argument("--store", type=int, default=0, help="BA_JAC_* for the implicit solver (0 auto, 1 planes, 2 factored, 3 tiled)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single GPU: write the poses, points, intrinsics and per-iteration cost of the timed solve to DIR/<name>.npy "
                         "(float64, at most 64 MB in all: a seeded sample of the points beyond that)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs needs --impl b200 on one GPU")
    wl = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 0)

    import ba_b200
    syn = ba_b200.synthetic

    def build_problem():
        if args.workload == "cfg3ref":
            c3 = syn.CONFIGS[3]
            n_kf = max(4, int(round(c3["n_kf"] * args.scale)))
            seq = syn.make_tum_sequence(n_kf, max(8, int(round(c3["n_lm"] * args.scale))), max(24, int(round(c3["n_obs"] * args.scale))),
                                        syn.SEED_BASE + 3)
            return syn.window_problem(seq, 0, n_kf - 1).problem
        pr = syn.make_config(wl["cfg"], scale=args.scale)
        if wl["cfg"] == 2:
            pr = syn.window_problem(pr, 0, 19).problem
        return pr

    if args.impl == "reference":
        # the reference's CPU implementation of the path: the oracle port with the reference's own linear solver setting
        # (SPARSE_SCHUR), RUN for W + K LM iterations on the same problem, all host threads (Ceres itself cannot be built
        # here: no Ceres / Eigen in the image).  Rank 0 only.
        if rank != 0:
            return 0
        problem = build_problem()
        threads = os.cpu_count() or 1
        base = cpu_reference_run(problem, wl["mode"], K, threads, warmup=W)
        n_it = base["lm_iterations"]
        line = {"metric": "LM iterations/s", "value": base["value"], "unit": "LM iterations/s", "n_gpus": args.gpus, "steps": K,
                "warmup": W, "ms_per_step": 1e3 * base["seconds"] / max(n_it, 1), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": bench_config(args, wl, problem, args.gpus, K),
                "final_cost": base["final_cost"],
                "note": "CPU restatement of the reference path (oracle/, not Ceres), linear solver = the reference's SPARSE_SCHUR "
                        "setting; every reported iteration was executed inside this run",
                "cpu_baseline": base, "e2e": {"value": base["value"], "unit": "LM iterations/s", "h2d_bytes_per_step": 0,
                                              "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    t_gen = time.time()
    full = build_problem()
    t_gen = time.time() - t_gen
    if world > 1 and wl["mode"] != (0, 0):
        raise SystemExit("windowed (explicit) workloads are single-GPU; use --workload cfg4/cfg5 with --gpus > 1")
    problem, _ = syn.shard_points(full, rank, world)
    opts = dict(use_depth_prior=wl["mode"][0], optimize_intrinsics=wl["mode"][1], function_tolerance=0.0,
                parameter_tolerance=0.0, gradient_tolerance=0.0, device=local_rank, n_obs_total=full.n_obs,
                jacobian_store=args.store)
    if wl["mode"] == (0, 0):
        opts["solver"] = SOLVERS[args.solver]
    s = ba_b200.GpuSolver(max_num_iterations=max(W, 1), **opts)
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idbuf.copy_(torch.frombuffer(bytearray(ba_b200.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idbuf, 0)
        s.comm_init(bytes(idbuf.cpu().numpy().tobytes()), rank, world)

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def maxr(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # pinned host copies for the end-to-end leg
    hp = problem.copy()
    for f in ("pose7", "pt3", "cam_idx", "pt_idx", "uv2", "depth"):
        setattr(hp, f, pinned_copy(getattr(hp, f)))

    # ---- warm-up: W LM iterations (plus kernel warm-up of the timing hooks)
    s.upload(hp)
    if W > 0:
        s.solve()
    # ---- timed: K LM iterations, inputs resident in HBM (upload outside the region)
    s.set_options(max_num_iterations=K)
    s.upload(hp)
    # (the sampler is started BEFORE the barrier: spawning nvidia-smi takes ~20 ms on rank 0, and a rank that enters the
    # solve late makes the others wait inside their first collective -- counted in their solve time)
    clocks = ClockSampler(local_rank) if rank == 0 else None
    sync_all()
    t0 = time.time()
    summ = s.solve()
    sync_all()
    wall_solve = time.time() - t0
    solve_ms = maxr(summ.solve_ms)
    trace = s.trace()
    phase_ms = s.phase_times()
    spchol = s.spchol_info()
    n_iter = summ.num_iterations
    pcg_counts = [t["linear_iters"] for t in trace[1:]]
    if args.dump_outputs:
        pose_k, pt_k, intr_k = s.download()
        outputs = {"pose7": pose_k, "points": pt_k, "intrinsics": intr_k, "cost_per_iteration": [t["cost"] for t in trace]}
    # ---- end to end through the C-ABI with host buffers (pinned, inputs and outputs): upload + solve + download
    out_bufs = (pinned_copy(np.zeros((problem.n_cam, 7))), pinned_copy(np.zeros((problem.n_pt, 3))), pinned_copy(np.zeros(4)))
    sync_all()
    t0 = time.time()
    s.upload(hp)
    summ2 = s.solve()
    pose, pt, intr = s.download(out=out_bufs)
    sync_all()
    e2e_s = maxr(time.time() - t0)
    clk = clocks.stop() if clocks else None
    h2d = sum(int(a.nbytes) for a in (hp.pose7, hp.pt3, hp.cam_idx, hp.pt_idx, hp.uv2, hp.intr, hp.intr_prior) if a is not None)
    if hp.depth is not None and wl["mode"][0]:
        h2d += int(hp.depth.nbytes)
    d2h = int(pose.nbytes + pt.nbytes + intr.nbytes)

    # ---- kernel timings for the roofline (CUDA events on the solver's stream, inputs >> L2 at cfg4/5;
    #      L2 flushed between launches otherwise)
    peak, peak_src = peaks()
    flush = full.n_obs * 36 < 512e6
    solver_used = int(summ.solver_used)
    kernels, dom, store, ms_lin = kernel_rooflines(ba_b200, s, problem, wl, solver_used, flush, peak)
    jac_obs_s = full.n_obs / (maxr(ms_lin) * 1e-3)
    # the matrix-free (north-star) path beside it when AUTO chose the block-sparse solver
    implicit_path = None
    if solver_used in (3, 4) and world == 1 and args.with_implicit_path:
        s2 = ba_b200.GpuSolver(max_num_iterations=max(W, 1), **dict(opts, solver=2))
        s2.upload(hp)
        if W > 0:
            s2.solve()
        s2.set_options(max_num_iterations=K)
        s2.upload(hp)
        sm2 = s2.solve()
        k2, d2, st2, _ = kernel_rooflines(ba_b200, s2, problem, wl, 2, flush, peak)
        implicit_path = {"value": sm2.num_iterations / (sm2.solve_ms * 1e-3), "unit": "LM iterations/s",
                         "ms_per_step": sm2.solve_ms / max(sm2.num_iterations, 1), "jacobian_store": st2,
                         "pcg_iterations_total": int(sm2.total_linear_iters), "final_cost": sm2.final_cost,
                         "gpu_launches": int(sm2.kernel_launches), "dominant_kernel": d2, "roofline_kernels": k2}
        s2.close()

    # the MATERIALISED Jacobian evaluation (r + Jc 2x6 + Jp 2x3 written per observation: SURVEY 8d's "Jacobian-eval"
    # kernel) and the planes-store Schur passes beside the factored / tiled / block-sparse kernels
    planes_kernels = None
    if wl["mode"] == (0, 0) and world == 1:
        s3 = ba_b200.GpuSolver(max_num_iterations=1, **dict(opts, solver=2, jacobian_store=1))
        s3.upload(hp)
        planes_kernels, _, _, ms_lin_planes = kernel_rooflines(ba_b200, s3, problem, wl, 2, flush, peak)
        s3.close()
        jac_obs_s_factored, jac_obs_s = jac_obs_s, full.n_obs / (ms_lin_planes * 1e-3)
    else:
        jac_obs_s_factored = None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    n_ent, n_blk = s.sparse_stats()
    n_pairs = s.sparse_pairs()
    if spchol:
        spchol["s_blocks"] = n_blk
    roof, phase_table = executed_roofline(args.workload, phase_ms, n_iter, solver_used, full, n_pairs, n_ent, spchol,
                                          int(summ.total_linear_iters), peak, peak_src)
    if roof is None:  # windowed explicit solver (graph replay: no phase events): the stand-alone kernel hook
        roof = {"kernel": dom, "bound": "launch latency (problem fits L2 many times over)", "achieved": kernels[dom]["achieved_gbs"],
                "peak": peak, "unit": "GB/s", "frac": kernels[dom]["frac"], "traffic": None, "peak_source": peak_src,
                "timing": "stand-alone launches of the kernel hook, CUDA events, mean of 20 after 3 warm-ups, L2 flushed",
                "bytes": kernels[dom]["bytes"]}
    line = {
        "metric": "LM iterations/s", "value": n_iter / (solve_ms * 1e-3), "unit": "LM iterations/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": solve_ms / max(n_iter, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args, wl, full, world, K),
        "detail": {"solver": SOLVER_NAME.get(solver_used, str(solver_used)), "jacobian_store": store, "lm_iterations": n_iter,
                   "pcg_iterations_total": int(summ.total_linear_iters), "pcg_iterations_per_lm": pcg_counts,
                   "exchange": None if world == 1 else
                   ("per LM iteration: NCCL all-reduce of camera blocks / reduced rhs / scalars; "
                    + ("distributed factorisation: every rank factorises its own subtrees of the supernodal tree, sums only the blocks of S "
                       "another rank needs (%d bytes instead of %d), the update matrices of the subtree roots (%d bytes) and the step; the top "
                       "part of the tree (%d cameras) runs on every rank" % (288 * spchol.get("s_exchange_blocks", 0), 288 * n_blk_all(s),
                                                                             spchol.get("exchange_bytes", 0), spchol.get("top_cameras", 0))
                       if spchol.get("distributed") else "all-reduce of the block-sparse S values; the factorisation runs replicated on every rank")
                    if solver_used == 4 else
                    "per LM iteration: NCCL all-reduce of the block-sparse S; persistent PCG row-sharded, exchange through tagged "
                    "slots in NVLink peer memory inside the kernel" if solver_used == 3 else
                    "NCCL all-reduce of camera-sized vectors (one per PCG iteration)"),
                   "generate_s": round(t_gen, 2), "sparse_blocks": n_blk, "sparse_pairs": n_pairs},
        "jacobian_eval_obs_per_s": jac_obs_s,
        "jacobian_eval_note": ("materialised r + Jc (2x6) + Jp (2x3), 208 B/obs (k_linearize, planes store; SURVEY 8d's definition)"
                               if planes_kernels is not None else "kernel of the store in force (see roofline_kernels)"),
        "jacobian_eval_factored_obs_per_s": jac_obs_s_factored,
        "final_cost": summ.final_cost, "initial_cost": summ.initial_cost,
        "solve_wall_ms": wall_solve * 1e3,
        "e2e": {"value": summ2.num_iterations / e2e_s, "unit": "LM iterations/s", "h2d_bytes_per_step": h2d // max(K, 1),
                "d2h_bytes_per_step": d2h // max(K, 1), "seconds": e2e_s,
                "note": "upload (pinned host -> HBM, index + structure build, symbolic factorisation) + solve + download through "
                        "ba_gpu_* with host buffers"},
        "gpu_launches": int(summ.kernel_launches),
        "roofline": roof,
        "phase_rooflines": phase_table,
        "roofline_kernels": kernels,
        "roofline_kernels_note": "stand-alone launches of single kernels (ba_gpu_time_kernel hook), CUDA events, 20 launches after 3 warm-ups",
        "phase_ms_per_step": {k: v / max(n_iter, 1) for k, v in phase_ms.items()},
        "sparse_cholesky": spchol,
        "parity_vs_n1": parity_vs_n1(args.workload, args.scale, solver_used, trace),
        "clocks": clk,
    }
    if args.write_golden and world == 1:
        path = os.path.join(ROOT, "tests", "golden", "bench_trace.json")
        g = json.load(open(path)) if os.path.exists(path) else {}
        g["%s/solver%d" % (args.workload, solver_used)] = {
            "cost": [t["cost"] for t in trace], "successful": [t["step_is_successful"] for t in trace],
            "when": time.strftime("%Y-%m-%d"), "solver": SOLVER_NAME.get(solver_used)}
        json.dump(g, open(path, "w"), indent=1)
    if args.workload == "cfg2" and world == 1:
        # the reference's own loop (src/main.cpp:161-166): windowOptimize over the last 20 keyframes every frame_frequency = 10
        # keyframes, warm-started, through the reference-facing entry point (host extraction + upload + solve + download per call)
        gp = ba_b200.CeresGlobalProblem(max_num_iterations=K, window_size=20)
        sw = ba_b200.GpuSolver(gp.gpu_options(function_tolerance=0.0, parameter_tolerance=0.0, gradient_tolerance=0.0, device=local_rank))
        for rep in range(2):  # pass 0 warms the context up (first-use allocations, module loading); pass 1 is reported
            seq2 = syn.make_config(2, scale=args.scale)
            intr0, intr1 = seq2.K.copy(), seq2.K.copy()
            n_win = n_it = 0
            phases = {}
            t0 = time.time()
            for n_kf in range(20, seq2.pose.shape[0] + 1, gp.frame_frequency):
                ok, sm = ba_b200.window_optimize(gp, n_kf - 20, n_kf - 1, seq2, intr0, intr1, solver=sw, return_summary=True,
                                                 timing=phases)
                n_win += 1
                n_it += sm.num_iterations
            torch.cuda.synchronize()
            dt = time.time() - t0
        sw.close()
        cabi = phases.get("upload", 0.0) + phases.get("solve", 0.0) + phases.get("download", 0.0)
        line["sliding_sequence"] = {"windows": n_win, "lm_iterations": n_it, "seconds": dt, "lm_iterations_per_s": n_it / dt,
                                    "windows_per_s": n_win / dt,
                                    "ms_per_window": {k: 1e3 * v / max(n_win, 1) for k, v in phases.items()},
                                    "c_abi_windows_per_s": n_win / cabi if cabi > 0 else None,
                                    "c_abi_note": "upload + solve + download only (the C-ABI calls); 'extract' / 'write_back' are the "
                                                  "Python stand-ins for the C++ wrapper's container walk",
                                    "note": "second pass over 79 warm-started 20-keyframe windows of the 800-keyframe sequence through window_optimize "
                                            "(Python mirror of windowOptimize: container walk, upload, K LM iterations, download, write-back)"}
        # the same schedule through the COMPILED drop-in (host/OptimizationUtils_gpu.cpp: windowOptimize with the reference's
        # signature over std::vector<KeyFrame> / Map3D, hash-map walk included) -- what main.cpp would call
        for rep in range(2):
            seq3 = syn.make_config(2, scale=args.scale)
            cpp = ba_b200.hostlib.sliding_sequence(seq3, 20, gp.frame_frequency, max_num_iterations=K, fixed_iterations=True)
        line["sliding_sequence"]["cpp_dropin"] = {
            "windows": cpp["windows"], "lm_iterations": cpp["lm_iterations"],
            "windows_per_s": 1e3 * cpp["windows"] / cpp["ms"]["total"], "lm_iterations_per_s": 1e3 * cpp["lm_iterations"] / cpp["ms"]["total"],
            "ms_per_window": {k: v / max(cpp["windows"], 1) for k, v in cpp["ms"].items()},
            "note": "windowOptimize of the compiled C++ drop-in over the reference's containers (second pass; host wall clock)"}
    if implicit_path is not None:
        line["implicit_path"] = implicit_path
    if planes_kernels is not None:
        line["planes_store_kernels"] = planes_kernels
    if not args.no_cpu_baseline and world == 1:
        # bounded sample of the same workload on the host cores: a few LM iterations actually run (about 10-30 s at config 5)
        sample_iters = min(K, 3 if full.n_obs > 100000 else K)
        line["cpu_baseline"] = cpu_reference_run(full, wl["mode"], sample_iters, os.cpu_count() or 1)
    print(json.dumps(line))
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
