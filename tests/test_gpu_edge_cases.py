"""Edge cases of the C-ABI on the GPU: empty and ragged inputs, unobserved cameras / points,
observations of the fixed camera only, the AUTO policy, full-size properties (cfg 5)."""
import numpy as np
import pytest

from helpers import ba_b200, mode_opts, ora, pose_err, rel_err, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic
cap = ba_b200.capi


def _tiny(n_cam=4, n_pt=30, seed=0):
    p = syn.make_config(1, scale=0.2)
    return p


def _solver(**kw):
    return ba_b200.GpuSolver(**kw)


@pytest.mark.parametrize("solver", [1, 2, 3, 4])
def test_no_observations(solver):
    """An upload without observations: zero cost, nothing moves, no crash (any solver)."""
    p = _tiny()
    q = p.copy()
    q.cam_idx = q.cam_idx[:0].copy()
    q.pt_idx = q.pt_idx[:0].copy()
    q.uv2 = q.uv2[:0].copy()
    if q.depth is not None:
        q.depth = q.depth[:0].copy()
    g, _ = mode_opts("NS", solver=solver, max_num_iterations=5)
    s = _solver(**g)
    try:
        s.upload(q)
        summ = s.solve()
        pose, pt, _ = s.download()
        assert summ.initial_cost == 0.0 and summ.final_cost == 0.0
        assert np.array_equal(pose, q.pose7) and np.array_equal(pt, q.pt3)
    finally:
        s.close()


@pytest.mark.parametrize("solver", [1, 2, 3, 4])
def test_ragged_problem_matches_oracle(solver):
    """Cameras without observations, points seen once, points never seen, a camera seen only through the
    fixed pose's points: the solve still tracks the oracle."""
    p = syn.make_config(3, scale=0.02)
    keep = np.ones(p.n_obs, dtype=bool)
    keep[p.cam_idx == 5] = False                       # camera 5 loses all its observations
    rng = np.random.default_rng(1)
    drop_pts = rng.choice(p.n_pt, size=p.n_pt // 10, replace=False)
    keep[np.isin(p.pt_idx, drop_pts)] = False          # 10 % of the points are never observed
    once = rng.choice(np.setdiff1d(np.arange(p.n_pt), drop_pts), size=p.n_pt // 10, replace=False)
    for q in once:                                     # another 10 % keep a single observation
        idx = np.flatnonzero((p.pt_idx == q) & keep)
        keep[idx[1:]] = False
    p.cam_idx, p.pt_idx, p.uv2 = p.cam_idx[keep].copy(), p.pt_idx[keep].copy(), p.uv2[keep].copy()
    if p.depth is not None:
        p.depth = p.depth[keep].copy()
    g, o = mode_opts("NS", solver=solver, max_num_iterations=6, explicit_max_dim=1024)
    s = _solver(**g)
    try:
        s.upload(p)
        summ = s.solve()
        pose, pt, _ = s.download()
        op = to_oracle(p)
        rc, osum, _ = ora.solve(op, ora.default_options(**o))
        assert rc == 0 and summ.num_iterations == osum.num_iterations
        assert abs(summ.final_cost - osum.final_cost) <= 1e-7 * osum.final_cost
        dt, dr = pose_err(pose, op.pose7)
        assert dt < 1e-5 and dr < 1e-5
        assert np.array_equal(pose[5], p.pose7[5])      # the unobserved camera does not move
        assert np.array_equal(pt[drop_pts], p.pt3[drop_pts])
    finally:
        s.close()


def test_single_camera_window():
    """One keyframe, fixed: nothing to optimise on the camera side; the (perturbed) points are pulled
    back onto their single observation (REF cost, intrinsics free with a prior)."""
    p = syn.make_config(1)
    keep = p.cam_idx == 0
    q = p.copy()
    q.pose7 = p.pose7[:1].copy()
    q.cam_idx, q.pt_idx, q.uv2, q.depth = p.cam_idx[keep].copy(), p.pt_idx[keep].copy(), p.uv2[keep].copy(), p.depth[keep].copy()
    seen = np.unique(q.pt_idx)
    q.pt3 = q.pt3.copy()
    q.pt3[seen] += np.random.default_rng(0).normal(size=(seen.size, 3)) * 0.01
    s = _solver(max_num_iterations=8)
    try:
        s.upload(q)
        summ = s.solve()
        pose, pt, intr = s.download()
        assert np.array_equal(pose, q.pose7)
        assert summ.initial_cost > 1e-8 and summ.final_cost < 1e-3 * summ.initial_cost
        op = to_oracle(q)
        rc, osum, _ = ora.solve(op, ora.default_options(max_num_iterations=8))
        assert rc == 0 and summ.num_iterations == osum.num_iterations
        assert abs(summ.final_cost - osum.final_cost) <= 1e-8 * summ.initial_cost
        assert np.max(np.abs(pt - op.pt3)) < 1e-6 and np.max(np.abs(intr - op.intr)) < 1e-5
    finally:
        s.close()


def test_auto_policy():
    """AUTO: dense explicit for windows, block-sparse S factorised exactly for large sequential NS problems, implicit
    when the co-visibility is dense (pairs per observation above the threshold).  Then the whole table of cost mode x solver x
    Jacobian store on three problems: the upload's return code, the solver and store in force, and whether the block-sparse S
    and the supernodal tree exist."""
    s = _solver()
    try:
        s.upload(syn.make_config(1))
        assert s.solve().solver_used == cap.BA_SOLVER_EXPLICIT_CHOLESKY
    finally:
        s.close()
    p = syn.make_config(3, scale=0.05)
    g, _ = mode_opts("NS", max_num_iterations=2, explicit_max_dim=36)
    s = _solver(**g)
    try:
        s.upload(p)
        assert s.solve().solver_used == cap.BA_SOLVER_SPARSE_SCHUR_CHOLESKY
        n_ent, n_blk = s.sparse_stats()
        assert n_blk > 0 and n_ent == 2 * n_blk - p.n_cam + (1 if p.fixed_cam >= 0 else 0)
    finally:
        s.close()
    s = _solver(sparse_max_pairs_per_obs=0, **g)
    try:
        s.upload(p)
        assert s.solve().solver_used == cap.BA_SOLVER_IMPLICIT_PCG
    finally:
        s.close()
    # every cost mode x solver x Jacobian store on a window, on the sequence above and on wide co-visibility
    seq = p.copy()
    seq.depth = syn.camera_point(seq.pose7[seq.cam_idx], seq.pt3[seq.pt_idx])[:, 2].copy()  # (for the depth-prior modes)
    problems = [("cfg1", syn.make_config(1), {}, True), ("seq", seq, dict(explicit_max_dim=36), True),
                ("wide", _wide_covisibility(), {}, False)]
    wrong = []
    for name, prob, kw, fronts_fit in problems:
        tiles_ok = _tiles_fit(prob)
        for mode in ("NS", "DEPTH", "INTR", "REF"):
            for solver in range(5):
                for store in range(4):
                    n_red = 6 * (prob.n_cam - 1) + (4 if mode in ("INTR", "REF") else 0)
                    want = _expected_plan(mode, solver, store, n_red, kw.get("explicit_max_dim", 160), fronts_fit, tiles_ok)
                    wrong += _check_plan(prob, mode, solver, store, kw, want, (name, mode, solver, store))
    assert not wrong, "\n".join(wrong)


def _wide_covisibility(n_cam=800, n_pt=4000, seed=5):
    """Every point is seen by three random cameras of 800: few observation pairs per observation, so AUTO builds the block-sparse
    S on an NS problem, but the co-visibility is so wide that no front of its Cholesky fits shared memory.  The cameras sit on
    a plane and look along +z at points 20 to 40 m away."""
    rng = np.random.default_rng(seed)
    K = syn.K_TUM.copy()
    truth = np.zeros((n_cam, 7))
    truth[:, 3] = 1.0
    truth[:, 4:6] = rng.uniform(-2.0, 2.0, (n_cam, 2))
    truth_pt = np.stack([rng.uniform(-3, 3, n_pt), rng.uniform(-2, 2, n_pt), rng.uniform(20, 40, n_pt)], axis=1)
    cam = np.concatenate([rng.choice(n_cam, 3, replace=False) for _ in range(n_pt)])
    lm = np.repeat(np.arange(n_pt), 3)
    order = np.lexsort((lm, cam))
    cam, lm = cam[order], lm[order]
    uv, z = syn.project(truth[cam], truth_pt[lm], K)
    uv = uv + 0.5 * rng.standard_normal(uv.shape)
    pose = truth.copy()
    pose[1:, 4:] += 0.01 * rng.standard_normal((n_cam - 1, 3))
    pt = truth_pt + 0.05 * rng.standard_normal(truth_pt.shape)
    return ba_b200.BAProblem(pose, pt, cam.astype(np.int32), lm.astype(np.int32), uv, z + 0.01 * rng.standard_normal(z.shape),
                             K, None, 0)


def _tiles_fit(p, tile_pts=128, max_span=64, max_obs=2048):
    """The tiled store's bounds (BA_JAC_TILED): every tile of 128 consecutive points spans <= 64 cameras and holds <= 2048
    observations."""
    tile = p.pt_idx // tile_pts
    for t in np.unique(tile):
        c = p.cam_idx[tile == t]
        if c.max() - c.min() + 1 > max_span or c.size > max_obs:
            return False
    return True


def _expected_plan(mode, solver, store, n_red, explicit_max_dim, fronts_fit, tiles_ok):
    """(upload return code, solver_used, jacobian_store_used) by the rules of include/ba_gpu.h for one GPU below the dense
    limit (BA_SOLVER_* and BA_JAC_* comments; AUTO's pair threshold holds on these problems)."""
    U = cap.BA_ERR_UNSUPPORTED
    depth, intr = mode in ("DEPTH", "REF"), mode in ("INTR", "REF")
    if solver == 4 and (depth or intr):        # the bordered sparse Cholesky: planes store only
        if store in (cap.BA_JAC_FACTORED, cap.BA_JAC_TILED) or not fronts_fit:
            return U, None, None
        return 0, 4, cap.BA_JAC_PLANES
    s = solver
    if s == 0:
        s = 1 if (n_red <= explicit_max_dim or intr) else 2
    if s in (2, 3, 4) and intr:                 # points-only solvers
        return U, None, None
    if s in (3, 4) and depth:                   # the block-sparse solvers need NS mode
        return U, None, None
    if s == 1:                                  # dense: planes store (FACTORED needs NS + PCG, TILED falls back)
        return (U, None, None) if store == cap.BA_JAC_FACTORED else (0, 1, cap.BA_JAC_PLANES)
    if s == 2 and depth:                        # matrix-free with depth prior: planes store
        return (U, None, None) if store == cap.BA_JAC_FACTORED else (0, 2, cap.BA_JAC_PLANES)
    if store == cap.BA_JAC_PLANES:              # NS: the block-sparse solvers rebuild S from the factored store
        return (U, None, None) if s in (3, 4) else (0, 2, cap.BA_JAC_PLANES)
    if s == 2 and solver == 0:                  # AUTO on a large NS problem with sparse co-visibility: block-sparse S,
        return 0, 4 if fronts_fit else 3, cap.BA_JAC_FACTORED   # factorised when the fronts fit, else PCG
    if s == 2:                                  # matrix-free: tiled where the tile bounds hold
        if tiles_ok and store != cap.BA_JAC_FACTORED:
            return 0, 2, cap.BA_JAC_TILED
        return (U, None, None) if store == cap.BA_JAC_TILED else (0, 2, cap.BA_JAC_FACTORED)
    if s == 4 and not fronts_fit:
        return U, None, None
    return 0, s, cap.BA_JAC_FACTORED


def _check_plan(prob, mode, solver, store, kw, want, case):
    g, _ = mode_opts(mode, solver=solver, jacobian_store=store, max_num_iterations=1, **kw)
    s = _solver(**g)
    try:
        try:
            s.upload(prob)
        except ba_b200.BAError as e:
            return [] if e.code == want[0] else [f"{case}: upload rc {e.code} ({e}), expected {want}"]
        if want[0] != 0:
            return [f"{case}: upload succeeded, expected rc {want[0]}"]
        used, store_used = s.solve().solver_used, s.jacobian_store_used()
        sparse_s, tree = s.sparse_stats()[1] > 0, bool(s.spchol_info())
        got = (used, store_used, sparse_s, tree)
        exp = (want[1], want[2], want[1] in (3, 4), want[1] == 4)
        return [] if got == exp else [f"{case}: (solver_used, store, sparse S, tree) {got}, expected {exp}"]
    finally:
        s.close()


def test_full_size_properties_cfg5():
    """BASELINE's full size (10k cameras, 2M points, 8M observations): size-independent properties --
    indices are the stable sort, the block-sparse product is symmetric and linear and agrees with the
    matrix-free products, one LM iteration decreases the cost."""
    p = syn.make_config(5)
    rng = np.random.default_rng(0)
    x1, x2 = rng.normal(size=6 * p.n_cam), rng.normal(size=6 * p.n_cam)
    ys = {}
    for name, kw in (("sparse", dict(solver=3)), ("tiled", dict(solver=2, jacobian_store=3)), ("factored", dict(solver=2, jacobian_store=2))):
        g, _ = mode_opts("NS", max_num_iterations=1, **kw)
        s = _solver(**g)
        try:
            s.upload(p)
            if name == "sparse":
                perm, pt_rowptr, cam_rowptr = s.indices()
                assert np.array_equal(perm, np.argsort(p.pt_idx, kind="stable").astype(np.int32))
                assert pt_rowptr[-1] == p.n_obs and cam_rowptr[-1] == p.n_obs
            y1, y2 = s.schur_matvec(1e4, x1), s.schur_matvec(1e4, x2)
            y12 = s.schur_matvec(1e4, 2.0 * x1 - 3.0 * x2)
            assert rel_err(y12, 2.0 * y1 - 3.0 * y2) < 1e-11
            assert abs(x1 @ y2 - x2 @ y1) <= 1e-10 * (abs(x1 @ y2) + np.linalg.norm(y1) * np.linalg.norm(x2))
            ys[name] = y1
            if name == "sparse":
                summ = s.solve()
                assert summ.final_cost < summ.initial_cost and np.isfinite(summ.final_cost)
        finally:
            s.close()
    assert rel_err(ys["tiled"], ys["sparse"]) < 1e-10
    assert rel_err(ys["factored"], ys["sparse"]) < 1e-10
