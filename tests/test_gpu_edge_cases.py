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
    when the co-visibility is dense (pairs per observation above the threshold)."""
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
