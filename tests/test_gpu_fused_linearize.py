"""The factored store's point-major linearisation (V, g_p reduced straight from the projection) and the back-substitution
that projects every observation again: the shared-memory camera run and its fallback for point tiles that span more
cameras than the stage holds, the point-major records kept for the implicit solver only (AUTO decides after the pair
count), and the kernel-timing hook on a block-sparse context, which has no point-major records."""
import math

import numpy as np
import pytest

import irregular_problems as ip
from helpers import ba_b200, mode_opts, ora, pose_err, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic
cap = ba_b200.capi

TILE_PTS = 128     # BA_TILE_PTS
STAGE_CAMS = 96    # BA_STAGE_CAMS


def _max_tile_span(p):
    tile = p.pt_idx // TILE_PTS
    n_t = int(tile.max()) + 1
    lo = np.full(n_t, np.iinfo(np.int64).max)
    hi = np.full(n_t, -1)
    np.minimum.at(lo, tile, p.cam_idx)
    np.maximum.at(hi, tile, p.cam_idx)
    return int(np.max(hi - lo + 1))


def _solve_vs_oracle(p, cost_tol, pose_tol, **kw):
    g, o = mode_opts("NS", max_num_iterations=6, **kw)
    s = ba_b200.GpuSolver(**g)
    try:
        s.upload(p)
        summ = s.solve()
        pose, _, _ = s.download()
    finally:
        s.close()
    op = to_oracle(p)
    rc, osum, _ = ora.solve(op, ora.default_options(**o))
    assert rc == 0 and summ.num_iterations == osum.num_iterations
    assert summ.num_successful == osum.num_successful
    assert abs(summ.final_cost - osum.final_cost) <= cost_tol * osum.final_cost
    assert summ.final_cost < 0.5 * summ.initial_cost
    dt, dr = pose_err(pose, op.pose7)
    assert dt < pose_tol and dr < pose_tol, (dt, dr)
    return summ


@pytest.mark.parametrize("solver", [2, 4])
def test_wide_tile_lockstep_oracle(solver):
    """A loop closure over 120 keyframes: the first point tile is seen by the first and the last cameras, more than the
    shared-memory stage holds, so the point-major linearisation and the back-substitution gather the camera records from
    global memory.  NS through the implicit solver (factored store, which also keeps the point-major records for its
    product) and through the sparse Cholesky, against the oracle."""
    p = ip.closure_problem("a")
    assert _max_tile_span(p) > STAGE_CAMS
    if solver == 2:
        # (an inexact Krylov step amplifies summation-order round-off by cond(S), DESIGN section 6: the tolerances of
        # test_gpu_fullsize's PCG lock step)
        summ = _solve_vs_oracle(p, 1e-5, 3e-3, solver=2, jacobian_store=2)
        assert summ.solver_used == cap.BA_SOLVER_IMPLICIT_PCG
    else:
        summ = _solve_vs_oracle(p, 1e-8, 1e-6, solver=4)
        assert summ.solver_used == cap.BA_SOLVER_SPARSE_SCHUR_CHOLESKY


@pytest.mark.parametrize("end", ["sparse", "implicit"])
def test_auto_solves_on_either_side(end):
    """AUTO allocates the point-major records only when the pair count sends it to the implicit solver; both outcomes
    solve the problem as the oracle does."""
    p = syn.make_config(3, scale=0.05)
    assert _max_tile_span(p) <= STAGE_CAMS
    if end == "sparse":
        summ = _solve_vs_oracle(p, 1e-8, 1e-6, explicit_max_dim=36)
        assert summ.solver_used == cap.BA_SOLVER_SPARSE_SCHUR_CHOLESKY
    else:
        # (the oracle's side: its implicit PCG, what mode_opts maps solver = 2 to)
        g, o = mode_opts("NS", max_num_iterations=6, solver=2)
        g.pop("solver")
        s = ba_b200.GpuSolver(explicit_max_dim=36, sparse_max_pairs_per_obs=0, **g)
        try:
            s.upload(p)
            summ = s.solve()
            pose, _, _ = s.download()
        finally:
            s.close()
        assert summ.solver_used == cap.BA_SOLVER_IMPLICIT_PCG
        op = to_oracle(p)
        rc, osum, _ = ora.solve(op, ora.default_options(**o))
        assert rc == 0 and summ.num_iterations == osum.num_iterations
        assert abs(summ.final_cost - osum.final_cost) <= 1e-7 * osum.final_cost
        dt, dr = pose_err(pose, op.pose7)
        assert dt < 1e-5 and dr < 1e-5, (dt, dr)


def test_time_kernel_on_sparse_context():
    """The timing hook on a solver-4 context: the linearisation and the block-CSR product time finitely without the
    point-major records; the two-pass product, which reads them, is refused."""
    p = syn.make_config(3, scale=0.05)
    g, _ = mode_opts("NS", solver=4, max_num_iterations=2)
    s = ba_b200.GpuSolver(**g)
    try:
        s.upload(p)
        for which in (cap.BA_KERNEL_LINEARIZE, cap.BA_KERNEL_SCHUR_MATVEC):
            ms = s.time_kernel(which, 1, 3)
            assert math.isfinite(ms) and ms > 0.0
        with pytest.raises(Exception):
            s.time_kernel(cap.BA_KERNEL_SCHUR_PASS1, 1, 3)
        assert s.solve().solver_used == cap.BA_SOLVER_SPARSE_SCHUR_CHOLESKY
    finally:
        s.close()
