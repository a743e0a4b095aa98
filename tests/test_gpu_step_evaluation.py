"""The factored store's step evaluation: the candidate cameras (k_candidate), then one point-major pass per point tile that
does the back-substitution, the model cost change, the candidate point and the candidate cost (kf_step_eval).
Both variants of the pass, the camera run staged in shared memory and the gather fallback for tiles that span more
cameras than the stage holds, under the implicit PCG (2), the block-sparse PCG (3) and the sparse Cholesky (4):
  - the model cost change and the cost change of the first iteration in the trace against the oracle's;
  - the candidate points, through that (accepted) step, against the oracle's;
  - over six iterations, the oracle's accept / reject sequence, and the same bits from two solves.
Printed with -s: the largest relative differences."""
import numpy as np
import pytest

import irregular_problems as ip
from helpers import ba_b200, mode_opts, ora, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic

TILE_PTS = 128     # BA_TILE_PTS
STAGE_CAMS = 96    # BA_STAGE_CAMS

PROBLEMS = {
    "cfg3_small": lambda: syn.make_config(3, scale=0.02),
    "cfg4_small": lambda: syn.make_config(4, scale=0.02),
    "wide_tile": lambda: ip.closure_problem("a"),   # first tile seen by the first and the last cameras: gather fallback
}
# relative tolerances (model cost change, cost change, points) after the first iteration.  The differences to the oracle are
# those of the step: the exact solver's differs by the linear solve's round-off (up to 6e-13, 3e-13, 3e-11 here), the
# Krylov solvers' by their stopping tolerance (implicit PCG up to 4e-11, 2e-9, 3e-7; block-sparse PCG up to 1e-8, 6e-7,
# 1e-4 on cfg4_small and the closure problem).  The four-launch step evaluation this pass replaced had the same differences
# to three digits on every case.
TOL = {4: (1e-11, 1e-11, 1e-9), 2: (1e-9, 1e-7, 1e-5), 3: (1e-6, 1e-5, 1e-3)}


def _max_tile_span(p):
    tile = p.pt_idx // TILE_PTS
    n_t = int(tile.max()) + 1
    lo = np.full(n_t, np.iinfo(np.int64).max)
    hi = np.full(n_t, -1)
    np.minimum.at(lo, tile, p.cam_idx)
    np.maximum.at(hi, tile, p.cam_idx)
    return int(np.max(hi - lo + 1))


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


def _solve(p, g):
    s = ba_b200.GpuSolver(**g)
    try:
        s.upload(p)
        summ = s.solve()
        pose, pt, _ = s.download()
        return summ, s.trace(), pose.copy(), pt.copy()
    finally:
        s.close()


@pytest.mark.parametrize("solver", [2, 3, 4])
@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_step_evaluation_vs_oracle(name, solver):
    p = PROBLEMS[name]()
    assert (_max_tile_span(p) > STAGE_CAMS) == (name == "wide_tile")
    extra = dict(jacobian_store=2) if solver == 2 else {}
    # one iteration: the step, its model cost change, the candidate and its cost, against the oracle's
    g1, o1 = mode_opts("NS", solver=solver, max_num_iterations=1, **extra)
    summ, tr, _, pt = _solve(p, g1)
    assert summ.solver_used == solver
    op = to_oracle(p)
    rc, _, otr = ora.solve(op, ora.default_options(**o1))
    assert rc == 0 and len(tr) == len(otr) == 2
    a, b = tr[1], otr[1]
    assert a["step_is_valid"] == b["step_is_valid"] == 1 and a["step_is_successful"] == b["step_is_successful"] == 1
    e_mcc, e_cc = _rel(a["model_cost_change"], b["model_cost_change"]), _rel(a["cost_change"], b["cost_change"])
    e_pt = float(np.max(np.abs(pt - op.pt3)) / np.max(np.abs(op.pt3)))
    print(f"\n{name} solver {solver}: model cost change {e_mcc:.2e}, cost change {e_cc:.2e}, points {e_pt:.2e}")
    t_mcc, t_cc, t_pt = TOL[solver]
    assert e_mcc <= t_mcc and e_cc <= t_cc and e_pt <= t_pt, (e_mcc, e_cc, e_pt)
    # several iterations: the same accept / reject sequence as the oracle's; then the same bits on a second solve
    g, o = mode_opts("NS", solver=solver, max_num_iterations=6, **extra)
    first = _solve(p, g)
    rc, _, otr = ora.solve(to_oracle(p), ora.default_options(**o))
    assert rc == 0 and len(first[1]) == len(otr)
    for a, b in zip(first[1], otr):
        assert a["step_is_valid"] == b["step_is_valid"] and a["step_is_successful"] == b["step_is_successful"]
    second = _solve(p, g)
    assert first[1] == second[1]
    assert np.array_equal(first[2], second[2]) and np.array_equal(first[3], second[3])
