"""The sparse Cholesky of the reduced camera system with depth prior and / or free intrinsics (REF / DEPTH / INTR cost):
block-sparse S from the planes store, the four intrinsics columns as a border solved by a 4 x 4 Schur complement between the
forward and the backward substitution.  Exact LM steps: lock step with the oracle's SPARSE_SCHUR-equivalent solve and with the
dense explicit path on the GPU; beyond the dense path's 16,384 unknowns AUTO takes this path."""
import numpy as np
import pytest

from helpers import ba_b200, mode_opts, ora, pose_err, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic
capi = ba_b200.capi


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


def _tum_ref(scale, seed=None):
    """A TUM-shaped REF sequence built like bench.py's cfg3ref at the given scale (all keyframes in one problem)."""
    c3 = syn.CONFIGS[3]
    n_kf = max(4, int(round(c3["n_kf"] * scale)))
    seq = syn.make_tum_sequence(n_kf, max(8, int(round(c3["n_lm"] * scale))), max(24, int(round(c3["n_obs"] * scale))),
                                syn.SEED_BASE + 3 if seed is None else seed)
    return syn.window_problem(seq, 0, n_kf - 1).problem


def _problem(name):
    if name == "cfg1":
        return syn.make_config(1)
    if name == "window20":
        seq = syn.make_tum_sequence(40, 4000, 24000, seed=5)
        return syn.window_problem(seq, 10, 29).problem
    if name == "tum0.02":
        return _tum_ref(0.02)
    if name == "tum0.1":
        return _tum_ref(0.1)
    if name == "tum_narrow":  # short co-visibility: the leaf size changes the tree
        seq = syn.make_tum_sequence(200, 12000, 36000, seed=17)
        return syn.window_problem(seq, 0, 199).problem
    raise KeyError(name)


def _lockstep_oracle(p, mode, iters, cache, cost_tol=1e-8, pose_tol=1e-6, intr_tol=1e-5, **extra):
    g, o = mode_opts(mode, solver=4, max_num_iterations=iters, **extra)
    s = _solver(cache, **g)
    s.upload(p)
    summ = s.solve()
    pose, pt, intr = s.download()
    tr = s.trace()
    op = to_oracle(p)
    rc, osum, otr = ora.solve(op, ora.default_options(**o))
    assert rc == 0
    assert summ.solver_used == capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY and summ.total_linear_iters == 0
    assert s.spchol_info()["nodes"] >= 1
    assert summ.termination == osum.termination and summ.num_iterations == osum.num_iterations
    assert summ.num_successful == osum.num_successful and summ.num_unsuccessful == osum.num_unsuccessful
    assert abs(summ.final_cost - osum.final_cost) <= cost_tol * osum.final_cost
    assert len(tr) == len(otr)
    for a, b in zip(tr, otr):
        assert a["step_is_valid"] == b["step_is_valid"] and a["step_is_successful"] == b["step_is_successful"]
        assert abs(a["cost"] - b["cost"]) <= cost_tol * abs(b["cost"]), (a, b)
    dt, dr = pose_err(pose, op.pose7)
    assert dt < pose_tol and dr < pose_tol, (dt, dr)
    if mode in ("REF", "INTR"):
        assert np.max(np.abs(intr - op.intr)) < intr_tol
    return s, summ


# ---------------------------------------------------------------- 1. lock step with the oracle
@pytest.mark.parametrize("mode", ["REF", "DEPTH", "INTR"])
@pytest.mark.parametrize("name", ["cfg1", "window20"])
def test_lockstep_oracle_modes(name, mode, solver_cache):
    s, summ = _lockstep_oracle(_problem(name), mode, 10, solver_cache)
    assert summ.final_cost < summ.initial_cost
    ph = s.phase_times()
    assert ph["linear_solve_factor_or_pcg"] > 0.0 and ph["schur_complement"] > 0.0


@pytest.mark.parametrize("name", ["tum0.02", "tum0.1"])
def test_lockstep_oracle_tum_ref(name, solver_cache):
    _, summ = _lockstep_oracle(_problem(name), "REF", 6, solver_cache)
    assert summ.final_cost < 0.5 * summ.initial_cost


# ---------------------------------------------------------------- 2. against the dense explicit path on the GPU
def test_sparse_vs_dense_explicit_ref():
    p = _problem("tum0.1")
    out = []
    for solver in (4, 1):
        g, _ = mode_opts("REF", solver=solver, max_num_iterations=8)
        s = ba_b200.GpuSolver(**g)
        s.upload(p)
        summ = s.solve()
        out.append((summ, s.trace(), s.download()[0].copy()))
        s.close()
    (ss, ts, ps), (sd, td, pd) = out
    assert ss.solver_used == capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY and sd.solver_used == capi.BA_SOLVER_EXPLICIT_CHOLESKY
    assert len(ts) == len(td)
    for a, b in zip(ts, td):
        assert a["step_is_valid"] == b["step_is_valid"] and a["step_is_successful"] == b["step_is_successful"]
        assert abs(a["cost"] - b["cost"]) <= 1e-10 * abs(b["cost"]), (a, b)
    dt, dr = pose_err(ps, pd)
    assert dt < 1e-8 and dr < 1e-8, (dt, dr)


# ---------------------------------------------------------------- 3. fixed camera
@pytest.mark.parametrize("fixed", [5, -1, "last"])
def test_fixed_camera_ref(fixed, solver_cache):
    p = _problem("window20")
    p.fixed_cam = p.n_cam - 1 if fixed == "last" else fixed
    _lockstep_oracle(p, "REF", 8, solver_cache)


# ---------------------------------------------------------------- 4. determinism and execution modes
def _run(p):
    g, _ = mode_opts("REF", solver=4, max_num_iterations=6)
    s = ba_b200.GpuSolver(**g)
    s.upload(p)
    summ = s.solve()
    r = (summ.final_cost, s.download()[0].copy(), [t["cost"] for t in s.trace()], s.spchol_info()["nodes"])
    s.close()
    return r


def test_repeated_solves_bit_identical(solver_cache):
    p = _problem("tum0.1")
    g, _ = mode_opts("REF", solver=4, max_num_iterations=6)
    s = _solver(solver_cache, **g)
    res = []
    for _ in range(2):
        s.upload(p)
        summ = s.solve()
        res.append((summ.final_cost, s.download()[0].copy(), [t["cost"] for t in s.trace()]))
    assert res[0][0] == res[1][0] and np.array_equal(res[0][1], res[1][1]) and res[0][2] == res[1][2]


def test_other_tree_agrees(monkeypatch):
    p = _problem("tum_narrow")
    base = _run(p)
    monkeypatch.setenv("BA_SPCHOL_LEAF", "6")
    leaf = _run(p)
    assert leaf[3] != base[3]  # really another tree
    assert abs(leaf[0] - base[0]) <= 1e-10 * base[0]
    assert pose_err(leaf[1], base[1])[0] < 1e-8


# ---------------------------------------------------------------- 5. beyond the dense explicit limit
N_KF_BIG = 2800


def _big_sequence():
    return syn.make_tum_sequence(N_KF_BIG, 40000, 280000, seed=33)


def test_auto_beyond_dense_limit():
    seq = _big_sequence()
    p = syn.window_problem(seq, 0, N_KF_BIG - 1).problem
    assert 6 * (p.n_cam - 1) + 4 > 16384
    g, o = mode_opts("REF", max_num_iterations=2)   # AUTO
    s = ba_b200.GpuSolver(**g)
    s.upload(p)
    summ = s.solve()
    pose, _, intr = s.download()
    tr = s.trace()
    s.close()
    assert summ.solver_used == capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY and summ.reduced_dim == 6 * (p.n_cam - 1) + 4
    op = to_oracle(p)
    rc, osum, otr = ora.solve(op, ora.default_options(solver=2, **o))
    assert rc == 0
    assert len(tr) == len(otr)
    for a, b in zip(tr, otr):
        assert a["step_is_valid"] == b["step_is_valid"] and a["step_is_successful"] == b["step_is_successful"]
        assert abs(a["cost"] - b["cost"]) <= 1e-8 * abs(b["cost"]), (a, b)
    assert abs(summ.final_cost - osum.final_cost) <= 1e-8 * osum.final_cost
    dt, dr = pose_err(pose, op.pose7)
    assert dt < 1e-6 and dr < 1e-6
    assert np.max(np.abs(intr - op.intr)) < 1e-5


def test_window_optimize_beyond_dense_limit():
    seq = _big_sequence()
    pose0 = seq.pose.copy()
    gp = ba_b200.CeresGlobalProblem(max_num_iterations=2)
    intr = seq.K.copy()
    ok, summ = ba_b200.window_optimize(gp, 0, N_KF_BIG - 1, seq, seq.K.copy(), intr, return_summary=True)
    assert ok and summ.solver_used == capi.BA_SOLVER_SPARSE_SCHUR_CHOLESKY
    assert summ.final_cost < summ.initial_cost and not np.array_equal(seq.pose, pose0)


# ---------------------------------------------------------------- 6. rejections
def test_rejected_when_fronts_cannot_fit(solver_cache):
    """Observations assigned to random points: the co-visibility is dense over 800 cameras, no front fits shared memory."""
    p = _tum_ref(1.0)
    rng = np.random.default_rng(7)
    p.pt_idx = rng.integers(0, p.n_pt, size=p.n_obs).astype(np.int32)
    g, _ = mode_opts("REF", solver=4)
    s = _solver(solver_cache, **g)
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(p)
    assert e.value.code == capi.BA_ERR_UNSUPPORTED
    assert "does not fit shared memory" in str(e.value)


def test_rejected_with_factored_store(solver_cache):
    g, _ = mode_opts("REF", solver=4, jacobian_store=2)
    s = _solver(solver_cache, **g)
    with pytest.raises(ba_b200.BAError) as e:
        s.upload(_problem("cfg1"))
    assert e.value.code == capi.BA_ERR_UNSUPPORTED


def test_schur_hooks_stay_ns_only(solver_cache):
    g, _ = mode_opts("DEPTH", solver=4)
    s = _solver(solver_cache, **g)
    p = _problem("window20")
    s.upload(p)
    with pytest.raises(ba_b200.BAError) as e:
        s.schur_solve(1e4, np.zeros(6 * p.n_cam))
    assert e.value.code == capi.BA_ERR_UNSUPPORTED


def test_sparse_stats_report_the_block_structure(solver_cache):
    """The block-sparse S of this path is the one the NS path builds for the same co-visibility."""
    p = _problem("window20")
    got = []
    for mode in ("REF", "NS"):
        s = _solver(solver_cache, **mode_opts(mode, solver=4)[0])
        s.upload(p)
        got.append((s.sparse_stats(), s.sparse_pairs()))
    assert got[0][0][1] > 0 and got[0][1] > 0
    assert got[0] == got[1]


# ---------------------------------------------------------------- 7. one context, cost mode changed between uploads
def _solve_state(s, p, rhs):
    s.upload(p)
    summ = s.solve()
    pose, pt, intr = s.download()
    y = s.schur_solve(1e4, rhs) if rhs is not None else None
    return summ.final_cost, pose.copy(), pt.copy(), intr.copy(), [t["cost"] for t in s.trace()], y


def _same(a, b):
    assert a[0] == b[0] and a[4] == b[4]
    for x, y in zip(a[1:4], b[1:4]):
        assert np.array_equal(x, y)
    if a[5] is not None:
        assert np.array_equal(a[5], b[5])


def test_context_reused_between_ref_and_ns():
    """REF through the bordered tree, then (set_options) NS through the one-row tree on a problem with more cameras, then REF
    again, all on one context: every solve is bit-identical to the same solve on a fresh context (the NS step carries no
    border of the earlier problem)."""
    ref_p, ns_p = _problem("window20"), syn.make_config(4, scale=0.1)
    assert ns_p.n_cam > ref_p.n_cam
    rhs = np.random.default_rng(2).normal(size=6 * ns_p.n_cam)
    g_ref, _ = mode_opts("REF", solver=4, max_num_iterations=6)
    g_ns, _ = mode_opts("NS", solver=4, max_num_iterations=6)
    fresh = {}
    for name, g, p, r in (("REF", g_ref, ref_p, None), ("NS", g_ns, ns_p, rhs)):
        f = ba_b200.GpuSolver(**g)
        fresh[name] = _solve_state(f, p, r)
        f.close()
    s = ba_b200.GpuSolver(**g_ref)
    _same(_solve_state(s, ref_p, None), fresh["REF"])
    s.set_options(use_depth_prior=0, optimize_intrinsics=0)
    ns = _solve_state(s, ns_p, rhs)
    assert s.spchol_info()["n_cam"] == ns_p.n_cam
    _same(ns, fresh["NS"])
    s.set_options(use_depth_prior=1, optimize_intrinsics=1)
    _same(_solve_state(s, ref_p, None), fresh["REF"])
    s.close()
