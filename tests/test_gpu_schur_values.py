"""Values of the block-sparse Schur complement (k_sp_schur, fp64 DMMA): blocks whose pair lists end anywhere in a trip of
32 pairs and in a DMMA step of two, against the oracle's product and a dense float64 numpy S; bit identity from run to run."""
import numpy as np
import pytest

from helpers import ba_b200, mode_opts, ora, rel_err, to_oracle

pytestmark = pytest.mark.gpu
syn = ba_b200.synthetic
K = np.array([525.0, 525.0, 319.5, 239.5])

# (camera i, camera j, points seen by exactly these two): every remainder of a trip of 32 and of a step of 2;
# camera 0 is the fixed camera
PAIRS = [(0, 1, 1), (1, 2, 2), (2, 3, 3), (3, 4, 31), (4, 5, 32), (5, 6, 33), (6, 7, 64), (7, 8, 65), (0, 8, 5)]


def pair_problem(seed, diag_only=False):
    """Cameras on a line looking down +z; the points of a pair are seen by its two cameras only.  With diag_only, one
    more camera sees 33 points nobody else sees: its only block is its diagonal block."""
    rng = np.random.default_rng(seed)
    n_cam = 10 if diag_only else 9
    pose = np.zeros((n_cam, 7))
    pose[:, 3] = 1.0
    pose[:, 4] = 0.15 * np.arange(n_cam) + 0.01 * rng.standard_normal(n_cam)
    pose[:, 5:] = 0.01 * rng.standard_normal((n_cam, 2))
    groups = [(i, j, n) for i, j, n in PAIRS] + ([(9, 9, 33)] if diag_only else [])
    pts, obs = [], []
    for i, j, n in groups:
        for _ in range(n):
            p = len(pts)
            pts.append([rng.uniform(-1.0, 2.0), rng.uniform(-0.8, 0.8), rng.uniform(2.0, 4.0)])
            obs += [(i, p)] if i == j else [(i, p), (j, p)]
    pts = np.array(pts)
    obs = np.array(sorted(obs))
    cam, pt = obs[:, 0], obs[:, 1]
    uv, z = syn.project(pose[cam], pts[pt], K)
    uv = uv + 0.5 * rng.standard_normal(uv.shape)
    pts = pts + 0.02 * rng.standard_normal(pts.shape)
    return ba_b200.BAProblem(pose, pts, cam.astype(np.int32), pt.astype(np.int32), uv, z, K.copy(), fixed_cam=0)


def dense_schur(p, out):
    """S = Hcc - Hcp Hpp^-1 Hpc in float64 numpy from the device's own Jacobians (unscaled, undamped)."""
    n_cam, n_pt = p.n_cam, p.n_pt
    Jc, Jp = out["Jc"][:, :2, :], out["Jp"][:, :2, :]
    Hcc = np.zeros((6 * n_cam, 6 * n_cam))
    W = np.zeros((n_pt, 6 * n_cam, 3))
    V = np.zeros((n_pt, 3, 3))
    for o in range(p.n_obs):
        c, q = p.cam_idx[o], p.pt_idx[o]
        Hcc[6 * c:6 * c + 6, 6 * c:6 * c + 6] += Jc[o].T @ Jc[o]
        W[q, 6 * c:6 * c + 6] += Jc[o].T @ Jp[o]
        V[q] += Jp[o].T @ Jp[o]
    return Hcc - np.einsum("pij,pjk->ik", W, np.linalg.solve(V, W.transpose(0, 2, 1)))


def probe(s, n, radius):
    return np.stack([s.schur_matvec(radius, np.eye(n)[k]) for k in range(n)], axis=1)


@pytest.mark.parametrize("diag_only", [False, True], ids=["pairs", "diag-only-camera"])
def test_pair_counts_vs_oracle(diag_only):
    p = pair_problem(3, diag_only)
    g, o = mode_opts("NS", solver=3)
    s = ba_b200.GpuSolver(**g)
    try:
        s.upload(p)
        rng = np.random.default_rng(7)
        for radius in (1e4, 3.7):
            x = rng.normal(size=6 * p.n_cam)
            y = s.schur_matvec(radius, x)
            yref = ora.schur_matvec(to_oracle(p), ora.default_options(**o), radius, x)
            assert rel_err(y, yref) < 1e-10, radius
    finally:
        s.close()


def test_every_block_vs_dense_numpy():
    """Unit-vector probes of every block (9 cameras) against S in float64 numpy.  The damping changes S by ~1e-2 / radius
    here (two-view points with short baselines amplify the damping of V): radius 1e16 puts it below 1e-13."""
    p = pair_problem(5)
    g, _ = mode_opts("NS", solver=3)
    s = ba_b200.GpuSolver(**g)
    try:
        s.upload(p)
        A = probe(s, 6 * p.n_cam, 1e16)
        Sref = dense_schur(p, s.eval())
    finally:
        s.close()
    assert rel_err(A, Sref) < 1e-10
    co = {(min(i, j), max(i, j)) for i, j, _ in PAIRS} | {(i, i) for i in range(p.n_cam)}
    for i in range(p.n_cam):
        for j in range(p.n_cam):
            blk = A[6 * i:6 * i + 6, 6 * j:6 * j + 6]
            if (min(i, j), max(i, j)) not in co:
                assert np.all(blk == 0.0), (i, j)
            elif i != 0 and j != 0:
                ref = Sref[6 * i:6 * i + 6, 6 * j:6 * j + 6]
                assert rel_err(blk, ref) < 1e-8, (i, j)


def test_same_bits_on_repeat():
    p = syn.make_config(3, scale=0.05)
    runs = []
    for _ in range(2):
        g, _ = mode_opts("NS", solver=4, max_num_iterations=6)
        s = ba_b200.GpuSolver(**g)
        try:
            s.upload(p)
            x = np.random.default_rng(1).normal(size=6 * p.n_cam)
            y = s.schur_matvec(1e4, x)
            summ = s.solve()
            runs.append((y, summ.final_cost, [(t["cost"], t["step_is_successful"]) for t in s.trace()], s.download()[0]))
        finally:
            s.close()
    (y1, c1, t1, p1), (y2, c2, t2, p2) = runs
    assert np.array_equal(y1, y2)
    assert c1 == c2 and t1 == t2
    assert np.array_equal(p1, p2)
