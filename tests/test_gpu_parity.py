"""Parity of the CUDA path (through the C-ABI) against the CPU oracle and the
mpmath golden vectors.  Tolerances are the north star's: indices bit-exact;
residuals / Jacobians 1e-12 relative; final cost 1e-8 relative; poses
1e-6 m / 1e-6 rad after a fixed LM iteration count."""
import json
import os

import numpy as np
import pytest

from helpers import ba_b200, mode_opts, ora, pose_err, rel_err, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "residual_jacobian_golden.json")))


def _problem(name):
    if name == "cfg1":
        return syn.make_config(1)
    if name == "cfg1_small":
        return syn.make_config(1, scale=0.1)
    if name == "cfg3_small":
        return syn.make_config(3, scale=0.02)
    if name == "cfg4_small":
        return syn.make_config(4, scale=0.02)
    if name == "cfg4_tenth":
        return syn.make_config(4, scale=0.1)
    if name == "cfg3_tenth":
        return syn.make_config(3, scale=0.1)
    if name == "window20":
        seq = syn.make_tum_sequence(40, 4000, 24000, seed=5)
        return syn.window_problem(seq, 10, 29).problem
    raise KeyError(name)


@pytest.fixture(scope="module")
def solver_cache():
    cache = {}
    yield cache
    for s in cache.values():
        s.close()


def _solver(cache, **kw):
    key = tuple(sorted(kw.items()))
    if key not in cache:
        cache[key] = ba_b200.GpuSolver(**kw)
    return cache[key]


# ---------------------------------------------------------------- indices
@pytest.mark.parametrize("name", ["cfg1", "cfg3_small", "cfg4_small", "window20"])
def test_indices_bit_exact(name, solver_cache):
    p = _problem(name)
    g, _ = mode_opts("NS")
    s = _solver(solver_cache, **g)
    s.upload(p)
    perm, pt_rowptr, cam_rowptr = s.indices()
    operm, opt, ocam = ora.build_indices(to_oracle(p))
    assert np.array_equal(perm, operm)
    assert np.array_equal(pt_rowptr, opt)
    assert np.array_equal(cam_rowptr, ocam)
    # stable counting sort property, independently of the oracle
    assert np.array_equal(perm, np.argsort(p.pt_idx, kind="stable").astype(np.int32))


def test_upload_rejects_unsorted(solver_cache):
    p = _problem("cfg1_small")
    p.cam_idx = p.cam_idx[::-1].copy()
    s = _solver(solver_cache, **mode_opts("NS")[0])
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(p)
    assert e.value.code == ba_b200.capi.BA_ERR_INVALID


@pytest.mark.parametrize("bad", ["pt_negative", "pt_large", "cam_negative", "cam_large"])
def test_upload_rejects_out_of_range_indices(bad, solver_cache):
    """Out-of-range indices must come back as BA_ERR_INVALID with the context still usable (the index build guards every
    kernel that runs before the host reads the error flag: no out-of-bounds write, no poisoned context)."""
    p = _problem("cfg1_small")
    q = p.copy()
    k = q.n_obs // 2
    if bad == "pt_negative":
        q.pt_idx[k] = -1
    elif bad == "pt_large":
        q.pt_idx[k] = q.n_pt + 1000
    elif bad == "cam_negative":
        q.cam_idx[0] = -1
    else:
        q.cam_idx[-1] = q.n_cam + 1000
    s = _solver(solver_cache, **mode_opts("NS")[0])
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(q)
    assert e.value.code == ba_b200.capi.BA_ERR_INVALID
    s.upload(p)   # the same context still works
    assert s.solve().final_cost > 0.0


# ---------------------------------------------------------------- residuals / Jacobians
@pytest.mark.parametrize("mode", ["REF", "NS", "DEPTH", "INTR"])
@pytest.mark.parametrize("name", ["cfg1", "cfg4_small"])
def test_eval_vs_oracle(name, mode, solver_cache):
    p = _problem(name)
    if p.depth is None and mode in ("REF", "DEPTH"):
        pytest.skip("no depth in this config")
    g, o = mode_opts(mode)
    s = _solver(solver_cache, **g)
    s.upload(p)
    out = s.eval()
    ref = ora.evaluate(to_oracle(p), ora.default_options(**o))
    assert ref["rc"] == 0
    sw = np.sqrt(1.0 / p.n_obs)
    # residuals: differences of O(640 px) quantities -> scale by the pixel magnitude
    assert rel_err(out["r"][:, :2], ref["r"][:, :2], scale=sw * 640.0) < 1e-12
    if g["use_depth_prior"]:
        assert rel_err(out["r"][:, 2], ref["r"][:, 2], scale=np.sqrt(10.0 / p.n_obs) * 4.0) < 1e-12
    # the constant pose block is not part of the program (:299): its Jacobian
    # columns are never formed -- the device stores zeros there
    free = p.cam_idx != p.fixed_cam
    assert np.all(out["Jc"][~free] == 0.0)
    assert rel_err(out["Jc"][free], ref["Jc"][free]) < 1e-12
    assert rel_err(out["Jp"], ref["Jp"]) < 1e-12
    if g["optimize_intrinsics"]:
        assert rel_err(out["Jk"], ref["Jk"]) < 1e-12
    assert abs(out["cost"] - ref["cost"]) <= 1e-12 * abs(ref["cost"])
    assert rel_err(out["g_c"], ref["g_c"]) < 1e-11
    assert rel_err(out["g_p"], ref["g_p"]) < 1e-11
    if g["optimize_intrinsics"]:
        assert rel_err(out["g_k"], ref["g_k"]) < 1e-11


def test_eval_vs_mpmath_golden(solver_cache):
    """One-observation problems built from the 60-digit golden vectors."""
    s = _solver(solver_cache, **mode_opts("REF", HUB_P_REPR=1e30, HUB_P_UNPR=1e30)[0])
    for g in GOLD["residual_jacobian"]:
        n = int(round(1.0 / g["w_repr"]))
        assert abs(1.0 / n - g["w_repr"]) < 1e-18 and abs(10.0 / n - g["w_unpr"]) < 1e-15
        p = ba_b200.BAProblem(np.array([g["pose"]]), np.array([g["pt"]]), [0], [0], np.array([g["uv"]]),
                              np.array([g["depth"]]), np.array(g["intr"]), None, -1)
        s.set_options(n_obs_total=n)
        s.upload(p)
        out = s.eval()
        sw = np.sqrt(g["w_repr"])
        assert rel_err(out["r"][0, :2], g["r"][:2], scale=sw * 640.0) < 1e-12
        assert rel_err(out["r"][0, 2:], g["r"][2:], scale=np.sqrt(g["w_unpr"]) * max(1.0, g["depth"])) < 1e-12
        for row in range(3):
            assert rel_err(out["Jc"][0, row], g["Jpose"][row]) < 1e-12
        assert rel_err(out["Jp"][0], g["Jpt"]) < 1e-12
        assert rel_err(out["Jk"][0], np.array(g["Jintr"])[:2]) < 1e-12


def test_huber_region_active(solver_cache):
    """Most residuals sit in Huber's linear region (SURVEY Appendix A): make sure
    both branches are exercised by the parity problems."""
    p = _problem("cfg1")
    ref = ora.evaluate(to_oracle(p), ora.default_options())
    s2 = np.sum(ref["r"][:, :2] ** 2, axis=1)
    assert np.count_nonzero(s2 > 0.9e-6) > 100


def test_se3_plus_vs_oracle(solver_cache):
    s = _solver(solver_cache, **mode_opts("NS")[0])
    rng = np.random.default_rng(7)
    n = 200
    pose = ba_b200.se3.exp(rng.normal(size=(n, 6)))
    delta = rng.normal(size=(n, 6)) * (10.0 ** rng.uniform(-13, 0, size=(n, 1)))
    delta[0] = 0.0
    out = s.se3_plus(pose, delta)
    for i in range(n):
        ref = ora.se3_mul(pose[i], ora.se3_exp(delta[i]))
        assert np.max(np.abs(out[i] - ref)) < 4e-15, i


# ---------------------------------------------------------------- implicit Schur product
@pytest.mark.parametrize("store", [1, 2, 3], ids=["planes", "factored", "tiled"])
@pytest.mark.parametrize("name", ["cfg1", "cfg4_small", "cfg3_small"])
def test_schur_matvec_vs_oracle(name, store, solver_cache):
    p = _problem(name)
    g, o = mode_opts("NS", solver=2, jacobian_store=store)
    s = _solver(solver_cache, **g)
    s.upload(p)
    rng = np.random.default_rng(1)
    for radius in (1e4, 3.7):
        x = rng.normal(size=6 * p.n_cam)
        y = s.schur_matvec(radius, x)
        yref = ora.schur_matvec(to_oracle(p), ora.default_options(**o), radius, x)
        assert rel_err(y, yref) < 1e-10
    # linearity and symmetry of S (size-independent properties)
    x1, x2 = rng.normal(size=6 * p.n_cam), rng.normal(size=6 * p.n_cam)
    y1, y2 = s.schur_matvec(1e4, x1), s.schur_matvec(1e4, x2)
    y12 = s.schur_matvec(1e4, 2.0 * x1 - 3.0 * x2)
    assert rel_err(y12, 2.0 * y1 - 3.0 * y2) < 1e-11
    assert abs(x1 @ y2 - x2 @ y1) <= 1e-10 * (abs(x1 @ y2) + np.linalg.norm(y1) * np.linalg.norm(x2))


# ---------------------------------------------------------------- full LM solves
def _compare_solve(p, mode, solver, iters, cache, lockstep=True, cost_tol=1e-8, pose_tol=1e-6, pt_tol=1e-5, trace_tol=1e-8,
                   **extra):
    g, o = mode_opts(mode, solver=solver, max_num_iterations=iters, **extra)
    s = _solver(cache, **g)
    s.upload(p)
    summ = s.solve()
    pose, pt, intr = s.download()
    tr = s.trace()
    op = to_oracle(p)
    rc, osum, otr = ora.solve(op, ora.default_options(**o))
    assert rc == 0
    assert summ.termination == osum.termination
    assert summ.num_iterations == osum.num_iterations
    assert summ.num_successful == osum.num_successful and summ.num_unsuccessful == osum.num_unsuccessful
    assert abs(summ.initial_cost - osum.initial_cost) <= 1e-12 * osum.initial_cost
    assert abs(summ.final_cost - osum.final_cost) <= cost_tol * osum.final_cost
    dt, dr = pose_err(pose, op.pose7)
    assert dt < pose_tol and dr < 1e-6, (dt, dr)
    assert np.max(np.abs(pt - op.pt3)) < pt_tol
    if mode in ("REF", "INTR"):
        assert np.max(np.abs(intr - op.intr)) < 1e-5
    if lockstep:
        assert len(tr) == len(otr)
        for a, b in zip(tr, otr):
            assert a["iteration"] == b["iteration"]
            assert a["step_is_valid"] == b["step_is_valid"] and a["step_is_successful"] == b["step_is_successful"]
            assert abs(a["cost"] - b["cost"]) <= trace_tol * abs(b["cost"]), (a, b)
            assert abs(a["radius"] - b["radius"]) <= 1e-6 * abs(b["radius"]), (a, b)
    return summ, osum


@pytest.mark.parametrize("mode", ["REF", "NS", "DEPTH", "INTR"])
def test_solve_explicit_cfg1(mode, solver_cache):
    summ, _ = _compare_solve(_problem("cfg1"), mode, 1, 10, solver_cache)
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_EXPLICIT_CHOLESKY
    assert summ.final_cost < 0.5 * summ.initial_cost


def test_solve_explicit_window20_ref(solver_cache):
    summ, _ = _compare_solve(_problem("window20"), "REF", 0, 10, solver_cache)
    assert summ.reduced_dim == 6 * 19 + 4 and summ.solver_used == ba_b200.capi.BA_SOLVER_EXPLICIT_CHOLESKY


@pytest.mark.parametrize("n_kf", [27, 28, 33, 43, 60, 200])
def test_solve_explicit_blocked_cholesky_ref(n_kf, solver_cache):
    """The reference's global optimisation (windowOptimize over ALL keyframes, REF cost with free intrinsics,
    src/main.cpp:179-182) beyond the register-resident L D L^T (n > 159): reduced dimension 6 (n_kf - 1) + 4 = 160 -> the
    shared-memory L D L^T (k_ldlt_solve, which runs at this size only); 166 (three tiles, the shortest look-ahead schedule),
    196 (last tile of 4 rows), 256 (full tiles only), 358 / 1198 (ragged last tile) -> the blocked dense Cholesky
    (ba_kernels_chol.cuh: fused diagonal kernel, three-stream look-ahead, flag-in-data substitution).  Exact step: lock step
    with the oracle's dense Schur at the north-star tolerance 1e-8 (measured worst per-iteration difference over the blocked
    sizes: 4.6e-12 relative, profiles/r02_chol_tolerance.txt)."""
    seq = syn.make_tum_sequence(n_kf, 30 * n_kf, 180 * n_kf, seed=21)
    p = syn.window_problem(seq, 0, n_kf - 1).problem
    summ, _ = _compare_solve(p, "REF", 0, 6, solver_cache)
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_EXPLICIT_CHOLESKY and summ.reduced_dim == 6 * (n_kf - 1) + 4
    assert summ.final_cost < 0.5 * summ.initial_cost


def test_blocked_cholesky_schedules_are_bit_identical(monkeypatch, solver_cache):
    """The three-stream look-ahead schedule (fused diagonal kernel, side buffer for the panel tile below the diagonal,
    flag-in-data substitution) performs the same operations per matrix entry in the same order as the plain right-looking
    sequence on one stream (BA_NO_LOOKAHEAD=1): every LM iteration's cost and the final state agree bit for bit."""
    n_kf = 50
    seq = syn.make_tum_sequence(n_kf, 30 * n_kf, 180 * n_kf, seed=5)
    p = syn.window_problem(seq, 0, n_kf - 1).problem   # n = 298: five tiles, ragged last one
    g, _ = mode_opts("REF", solver=0, max_num_iterations=5)

    def run():
        s = ba_b200.GpuSolver(**g)   # the schedule switches are read when the context is created / at every solve
        s.upload(p)
        summ = s.solve()
        pose, pt, intr = s.download()
        costs = [t["cost"] for t in s.trace()]
        s.close()
        return summ, pose, pt, intr, costs

    a = run()
    monkeypatch.setenv("BA_NO_LOOKAHEAD", "1")
    b = run()
    assert a[0].reduced_dim == 6 * (n_kf - 1) + 4 and a[0].num_iterations == b[0].num_iterations >= 3
    assert a[4] == b[4] and a[0].final_cost == b[0].final_cost
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])


def test_solve_to_convergence_ref(solver_cache):
    """Reference settings (75 iterations, tolerances on): same termination."""
    _compare_solve(_problem("cfg1"), "REF", 1, 75, solver_cache)


@pytest.mark.parametrize("store", [1, 2, 3], ids=["planes", "factored", "tiled"])
@pytest.mark.parametrize("name", ["cfg1", "cfg3_small"])
def test_solve_implicit_pcg(name, store, solver_cache):
    """Implicit Schur + block-Jacobi PCG against the oracle's own PCG, in lock
    step: same PCG iteration counts, cost 1e-8, poses 1e-6 (well-conditioned
    TUM-shaped problems)."""
    summ, osum = _compare_solve(_problem(name), "NS", 2, 8, solver_cache, jacobian_store=store)
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_IMPLICIT_PCG
    assert summ.total_linear_iters == osum.total_linear_iters


@pytest.mark.parametrize("store", [1, 2, 3], ids=["planes", "factored", "tiled"])
def test_solve_implicit_pcg_ill_conditioned(store, solver_cache):
    """BAL-shaped loop: the reduced system is so ill-conditioned that PCG stops on
    its iteration cap / eta = 1e-6 far from the exact step, and summation-order
    round-off (1e-16) is amplified by cond(S) into 1e-6 relative cost differences
    between ANY two implementations (oracle vs oracle with another thread count
    included).  Parity here: same accept/reject sequence, cost to 1e-5, poses to
    1e-4 of the 30 m scene."""
    p = _problem("cfg4_small")
    g, o = mode_opts("NS", solver=2, max_num_iterations=8, jacobian_store=store)
    s = _solver(solver_cache, **g)
    s.upload(p)
    summ = s.solve()
    pose, pt, _ = s.download()
    op = to_oracle(p)
    rc, osum, otr = ora.solve(op, ora.default_options(**o))
    assert rc == 0 and summ.num_iterations == osum.num_iterations
    assert [t["step_is_successful"] for t in s.trace()] == [t["step_is_successful"] for t in otr]
    assert abs(summ.final_cost - osum.final_cost) <= 1e-5 * osum.final_cost
    dt, dr = pose_err(pose, op.pose7)
    assert dt < 3e-3 and dr < 1e-4, (dt, dr)
    assert abs(summ.total_linear_iters - osum.total_linear_iters) <= 0.05 * osum.total_linear_iters


# ---------------------------------------------------------------- explicit block-sparse Schur complement + PCG
@pytest.mark.parametrize("name", ["cfg1", "cfg4_small", "cfg3_small"])
def test_sparse_schur_product_vs_oracle(name, solver_cache):
    """The block-sparse S times x equals the oracle's implicit product (and is symmetric)."""
    p = _problem(name)
    g, o = mode_opts("NS", solver=3)
    s = _solver(solver_cache, **g)
    s.upload(p)
    rng = np.random.default_rng(2)
    for radius in (1e4, 3.7):
        x = rng.normal(size=6 * p.n_cam)
        y = s.schur_matvec(radius, x)
        yref = ora.schur_matvec(to_oracle(p), ora.default_options(**o), radius, x)
        assert rel_err(y, yref) < 1e-10
    x1, x2 = rng.normal(size=6 * p.n_cam), rng.normal(size=6 * p.n_cam)
    y1, y2 = s.schur_matvec(1e4, x1), s.schur_matvec(1e4, x2)
    assert abs(x1 @ y2 - x2 @ y1) <= 1e-10 * (abs(x1 @ y2) + np.linalg.norm(y1) * np.linalg.norm(x2))


@pytest.mark.parametrize("persistent", [0, 1], ids=["launch-per-step", "persistent"])
@pytest.mark.parametrize("name", ["cfg1", "cfg3_small"])
def test_solve_sparse_schur_pcg(name, persistent, solver_cache):
    """Explicit block-sparse S + PCG against the oracle's PCG, in lock step on the
    well-conditioned TUM-shaped problems; the PCG loop as one persistent
    cooperative kernel or as one launch per step."""
    summ, osum = _compare_solve(_problem(name), "NS", 3, 8, solver_cache, persistent_pcg=persistent)
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_SPARSE_SCHUR_PCG
    assert abs(summ.total_linear_iters - osum.total_linear_iters) <= max(2, 0.02 * osum.total_linear_iters)


def test_sparse_schur_duplicate_camera_observations(solver_cache):
    """A camera that observes the same landmark twice: the diagonal block needs both
    orders of the pair."""
    p = _problem("cfg1")
    # duplicate the first 40 observations of camera 3 (same landmark, shifted pixel), keep camera-major order
    idx = np.flatnonzero(p.cam_idx == 3)[:40]
    ins = idx[-1] + 1
    p.cam_idx = np.insert(p.cam_idx, ins, p.cam_idx[idx])
    p.pt_idx = np.insert(p.pt_idx, ins, p.pt_idx[idx])
    p.uv2 = np.insert(p.uv2, ins, p.uv2[idx] + 0.25, axis=0)
    if p.depth is not None:
        p.depth = np.insert(p.depth, ins, p.depth[idx])
    g, o = mode_opts("NS", solver=3)
    s = _solver(solver_cache, **g)
    s.upload(p)
    x = np.random.default_rng(5).normal(size=6 * p.n_cam)
    y = s.schur_matvec(1e4, x)
    yref = ora.schur_matvec(to_oracle(p), ora.default_options(**o), 1e4, x)
    assert rel_err(y, yref) < 1e-10


def test_sparse_schur_rejected_outside_ns(solver_cache):
    p = _problem("cfg1_small")
    s = _solver(solver_cache, use_depth_prior=1, optimize_intrinsics=0, solver=3)
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(p)
    assert e.value.code == ba_b200.capi.BA_ERR_UNSUPPORTED


# ---------------------------------------------------------------- exact sparse Cholesky of the block-sparse S
@pytest.mark.parametrize("name", ["cfg1", "cfg3_small", "cfg4_small", "cfg4_tenth", "cfg3_tenth"])
def test_spchol_solve_inverts_the_product(name, solver_cache):
    """(S + D^2)^-1 through the supernodal multifrontal Cholesky, checked against the block-CSR product of the same
    matrix (itself checked against the oracle above) and against a dense solve assembled from products with unit vectors."""
    p = _problem(name)
    g, _ = mode_opts("NS", solver=4)
    s = _solver(solver_cache, **g)
    s.upload(p)
    info = s.spchol_info()
    assert info["nodes"] >= 1 and info["n_cam"] == p.n_cam
    rng = np.random.default_rng(11)
    for radius in (1e4, 3.7):
        b = rng.normal(size=6 * p.n_cam)
        y = s.schur_solve(radius, b)
        back = s.schur_matvec(radius, y)
        assert rel_err(back, b) < 1e-9, (name, radius)
    if p.n_cam <= 40:
        n = 6 * p.n_cam
        A = np.stack([s.schur_matvec(1e4, np.eye(n)[k]) for k in range(n)], axis=1)
        b = rng.normal(size=n)
        y = s.schur_solve(1e4, b)
        yref = np.linalg.solve(A, b)
        assert rel_err(y, yref) < 1e-9


@pytest.mark.parametrize("name,iters", [("cfg1", 8), ("cfg3_small", 8), ("cfg4_small", 8), ("cfg4_tenth", 6), ("cfg3_tenth", 6)])
def test_solve_spchol_lockstep(name, iters, solver_cache):
    """Exact step by the sparse Cholesky against the oracle's SPARSE_SCHUR-equivalent (envelope Cholesky): lock step,
    cost 1e-8, poses 1e-6 -- also on the BAL-shaped loop where the inexact PCG step only reaches 1e-5."""
    summ, osum = _compare_solve(_problem(name), "NS", 4, iters, solver_cache)
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY
    assert summ.total_linear_iters == 0
    assert summ.final_cost < 0.5 * summ.initial_cost


def test_spchol_fixed_camera_anywhere(solver_cache):
    p = _problem("cfg3_small")
    for fixed in (5, -1, p.n_cam - 1):
        q = p.copy()
        q.fixed_cam = fixed
        _compare_solve(q, "NS", 4, 4, solver_cache)


def test_auto_picks_sparse_cholesky_on_sequential_data(solver_cache):
    p = _problem("cfg4_tenth")
    g, _ = mode_opts("NS", solver=0, max_num_iterations=3)
    s = _solver(solver_cache, **g)
    s.upload(p)
    summ = s.solve()
    assert summ.solver_used == ba_b200.capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY and s.spchol_info()["levels"] >= 3


def test_spchol_small_leaves_same_result(monkeypatch, solver_cache):
    """Another dissection (leaves of 6 cameras: deeper tree, more extend-add) solves the same system."""
    p = _problem("cfg4_tenth")
    g, _ = mode_opts("NS", solver=4, max_num_iterations=4)
    out = []
    for leaf in (None, "6"):
        if leaf:
            monkeypatch.setenv("BA_SPCHOL_LEAF", leaf)
        s = ba_b200.GpuSolver(**g)
        s.upload(p)
        summ = s.solve()
        out.append((summ.final_cost, s.download()[0], s.spchol_info()["nodes"]))
        s.close()
    assert out[1][2] != out[0][2]   # really another tree
    assert abs(out[0][0] - out[1][0]) <= 1e-10 * out[0][0]
    assert pose_err(out[0][1], out[1][1])[0] < 1e-8


@pytest.mark.parametrize("name,parts", [("cfg4_tenth", 2), ("cfg4_tenth", 8), ("cfg3_tenth", 4), ("cfg4_tenth", 3)])
def test_spchol_partitioned_tree_same_bits(name, parts, monkeypatch):
    """The subtree-to-rank partition of the multi-GPU factorisation, all parts on this GPU one after the other (phase A per part,
    then top part + backward substitution): the same arithmetic in the same order per node, so the same bits as one queue."""
    p = _problem(name)
    g, _ = mode_opts("NS", solver=4, max_num_iterations=4)
    out = []
    monkeypatch.setenv("BA_SPCHOL_LEAF", "6")   # (deep tree on the reduced test sizes)
    for n in (None, str(parts)):
        if n:
            monkeypatch.setenv("BA_SPCHOL_PARTS", n)
        s = ba_b200.GpuSolver(**g)
        s.upload(p)
        summ = s.solve()
        out.append((summ.final_cost, s.download()[0].copy(), s.spchol_info()))
        s.close()
    assert out[0][2]["parts"] == 1
    if out[1][2]["parts"] == 1:
        pytest.skip("tree too small for %d parts" % parts)
    assert out[1][2]["parts"] == parts and out[1][2]["top_cameras"] > 0
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])


def test_spchol_repeated_solves_are_deterministic(solver_cache):
    p = _problem("cfg4_tenth")
    g, _ = mode_opts("NS", solver=4, max_num_iterations=4)
    s = _solver(solver_cache, **g)
    out = []
    for _ in range(2):
        s.upload(p)
        summ = s.solve()
        out.append((summ.final_cost, s.download()[0].copy()))
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])


def test_explicit_and_implicit_agree(solver_cache):
    """A converged PCG step equals the Cholesky step: same optimum."""
    p = _problem("cfg3_small")
    res = []
    for solver in (1, 2):
        g, _ = mode_opts("NS", solver=solver, max_num_iterations=60, explicit_max_dim=1024, function_tolerance=1e-13,
                         parameter_tolerance=1e-13)
        s = _solver(solver_cache, **g)
        s.upload(p)
        summ = s.solve()
        res.append((summ.final_cost, s.download()[0]))
    # LM with inexact steps creeps towards the optimum the Cholesky path reaches
    assert abs(res[0][0] - res[1][0]) <= 2e-5 * res[0][0]
    dt, dr = pose_err(res[0][1], res[1][1])
    assert dt < 2e-3 and dr < 2e-3


def test_noise_free_problem_reaches_zero_cost(solver_cache):
    """Known-answer: exact observations, perturbed start -> cost ~ 0, poses -> truth."""
    seq = syn.make_tum_sequence(7, 300, 1800, seed=21, noise=False)
    truth = syn.window_problem(seq, 0, 6, use_depth=False).problem
    rng = np.random.default_rng(2)
    p = truth.copy()
    d = np.concatenate([0.01 * rng.normal(size=(7, 3)), 0.005 * rng.normal(size=(7, 3))], axis=1)
    d[0] = 0
    p.pose7 = ba_b200.se3.mul(truth.pose7, ba_b200.se3.exp(d))
    p.pt3 = truth.pt3 + 0.01 * rng.normal(size=truth.pt3.shape)
    # float-rounded pixels keep the optimum ~1e-5 px away from the truth
    g, _ = mode_opts("NS", solver=1, max_num_iterations=50, function_tolerance=1e-14, HUB_P_REPR=1.0)
    s = _solver(solver_cache, **g)
    s.upload(p)
    summ = s.solve()
    assert summ.final_cost < 1e-9 * summ.initial_cost


def test_repeated_solves_are_deterministic(solver_cache):
    p = _problem("cfg3_small")
    g, _ = mode_opts("NS", solver=2, max_num_iterations=5)
    s = _solver(solver_cache, **g)
    out = []
    for _ in range(2):
        s.upload(p)
        summ = s.solve()
        out.append((summ.final_cost, s.download()[0].copy()))
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])


def test_window_optimize_mirror(solver_cache):
    """windowOptimize drop-in semantics: in-place mutation + frame change."""
    seq = syn.make_tum_sequence(30, 3000, 18000, seed=9)
    seq_o = syn.make_tum_sequence(30, 3000, 18000, seed=9)
    gp = ba_b200.CeresGlobalProblem(max_num_iterations=10)
    intr = seq.K.copy()
    ok, summ = ba_b200.window_optimize(gp, 10, 29, seq, seq.K.copy(), intr, return_summary=True)
    assert ok and summ.final_cost < summ.initial_cost
    # oracle on the same window
    win = syn.window_problem(seq_o, 10, 29)
    op = to_oracle(win.problem)
    rc, osum, _ = ora.solve(op, ora.default_options(max_num_iterations=10))
    syn.write_back(seq_o, win, op.pose7, op.pt3)
    assert abs(summ.final_cost - osum.final_cost) <= 1e-8 * osum.final_cost
    dt, dr = pose_err(seq.pose, seq_o.pose)
    assert dt < 1e-6 and dr < 1e-6
    assert np.max(np.abs(intr - op.intr)) < 1e-5
    # poses outside the window untouched
    assert np.array_equal(seq.pose[:10], seq_o.pose[:10])


def test_factored_store_rejected_outside_ns_implicit(solver_cache):
    p = _problem("cfg1_small")
    s = _solver(solver_cache, use_depth_prior=1, optimize_intrinsics=1, jacobian_store=2)
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(p)
    assert e.value.code == ba_b200.capi.BA_ERR_UNSUPPORTED


def test_tiled_store_needs_index_locality(solver_cache):
    """Point ids relabelled at random: a 128-point tile then spans every camera.
    The tiled store refuses (explicit request) / AUTO falls back to the two-pass
    factored product, which still matches the oracle."""
    p = syn.make_config(4, scale=0.1)
    assert p.n_cam > 64
    rng = np.random.default_rng(3)
    relabel = rng.permutation(p.n_pt).astype(np.int32)
    p.pt_idx = relabel[p.pt_idx]
    inv = np.empty_like(relabel)
    inv[relabel] = np.arange(p.n_pt, dtype=np.int32)
    p.pt3 = p.pt3[inv].copy()
    g, o = mode_opts("NS", solver=2, jacobian_store=3)
    s = _solver(solver_cache, **g)
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(p)
    assert e.value.code == ba_b200.capi.BA_ERR_UNSUPPORTED
    g, o = mode_opts("NS", solver=2, jacobian_store=0)
    s = _solver(solver_cache, **g)
    s.upload(p)
    assert s.jacobian_store_used() == ba_b200.capi.BA_JAC_FACTORED
    x = rng.normal(size=6 * p.n_cam)
    y = s.schur_matvec(1e4, x)
    yref = ora.schur_matvec(to_oracle(p), ora.default_options(**o), 1e4, x)
    assert rel_err(y, yref) < 1e-10


def test_auto_store_is_tiled_on_sequential_data(solver_cache):
    p = _problem("cfg3_small")
    g, _ = mode_opts("NS", solver=2)
    s = _solver(solver_cache, **g)
    s.upload(p)
    assert s.jacobian_store_used() == ba_b200.capi.BA_JAC_TILED


def test_eval_hook_with_factored_store(solver_cache):
    """The un-scaled evaluation hook materialises planes on demand."""
    p = _problem("cfg3_small")
    g, o = mode_opts("NS", solver=2, jacobian_store=2)
    s = _solver(solver_cache, **g)
    s.upload(p)
    out = s.eval()
    ref = ora.evaluate(to_oracle(p), ora.default_options(**o))
    free = p.cam_idx != p.fixed_cam
    assert rel_err(out["Jc"][free], ref["Jc"][free]) < 1e-12 and rel_err(out["Jp"], ref["Jp"]) < 1e-12
    summ = s.solve()
    assert summ.final_cost < summ.initial_cost


# ---------------------------------------------------------------- windowed explicit path: variants of the same solve
def _explicit_run(p, env=None, iters=8, **kw):
    """One REF-mode explicit solve in a fresh context under temporary environment switches (A/B aids of the library)."""
    env = env or {}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        g, _ = mode_opts("REF", solver=1, max_num_iterations=iters, **kw)
        s = ba_b200.GpuSolver(**g)
        try:
            s.upload(p)
            summ = s.solve()
            pose, pt, intr = s.download()
            tr = s.trace()
        finally:
            s.close()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return summ, pose, pt, intr, tr


@pytest.mark.parametrize("name", ["cfg1", "window20"])
def test_window_graph_and_device_pairs_are_bit_identical(name):
    """The CUDA-graph replay of the LM iteration and the two-stream fork change HOW the work is enqueued, not the
    arithmetic: results must equal the direct-enqueue / single-stream run bit for bit."""
    p = _problem(name)
    base = _explicit_run(p)
    for env in ({"BA_NO_LM_GRAPH": "1"}, {"BA_NO_FORK": "1"}):
        other = _explicit_run(p, env)
        assert other[0].num_iterations == base[0].num_iterations
        assert other[0].final_cost == base[0].final_cost, env
        assert np.array_equal(other[1], base[1]) and np.array_equal(other[2], base[2]) and np.array_equal(other[3], base[3]), env
        assert [t["cost"] for t in other[4]] == [t["cost"] for t in base[4]], env


def test_window_reupload_updates_graph():
    """Sliding windows through ONE context: every upload re-captures the LM iteration and updates the graph executable
    in place; each window must equal its solve in a fresh context."""
    seq = syn.make_tum_sequence(60, 6000, 36000, seed=9)
    g, _ = mode_opts("REF", solver=1, max_num_iterations=6)
    s = ba_b200.GpuSolver(**g)
    try:
        for a in (0, 10, 25, 40, 3):  # different sizes, last one smaller again
            p = syn.window_problem(seq, a, min(a + 19, 59) if a != 3 else 9).problem
            s.upload(p)
            summ = s.solve()
            pose, pt, intr = s.download()
            ref = _explicit_run(p, iters=6)
            assert summ.final_cost == ref[0].final_cost
            assert np.array_equal(pose, ref[1]) and np.array_equal(pt, ref[2])
    finally:
        s.close()


def test_explicit_duplicate_camera_observations(solver_cache):
    """A camera that observes the same landmark twice, through the dense explicit path (device-built pair list):
    lock step with the oracle."""
    p = _problem("cfg1")
    idx = np.flatnonzero(p.cam_idx == 3)[:40]
    ins = idx[-1] + 1
    p.cam_idx = np.insert(p.cam_idx, ins, p.cam_idx[idx])
    p.pt_idx = np.insert(p.pt_idx, ins, p.pt_idx[idx])
    p.uv2 = np.insert(p.uv2, ins, p.uv2[idx] + 0.25, axis=0)
    if p.depth is not None:
        p.depth = np.insert(p.depth, ins, p.depth[idx])
    _compare_solve(p, "REF", 1, 6, solver_cache)
