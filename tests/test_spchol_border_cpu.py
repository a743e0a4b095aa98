"""The sparse Cholesky with the intrinsics border (REF cost: free intrinsics as a dense 4-column border of the reduced camera
system) on the CPU: the multifrontal solve with five right-hand-side rows, the 4 x 4 border system and the backward
substitution with z - Z y_k (numpy emulation over the symbolic structures of libba_gpu.so) must equal a dense solve of the
whole bordered system."""
import numpy as np
import pytest

from helpers import ba_b200
from spchol_border_emulation import bordered_solve
from spchol_emulation import Symbolic, covisibility_blocks

syn = ba_b200.synthetic


def _bordered_system(n_cam, bi, bj, fixed, rng):
    """Random SPD bordered system with the given block pattern of A; the fixed camera's border rows are zero."""
    A = np.zeros((6 * n_cam, 6 * n_cam))
    blocks = np.zeros((len(bi), 6, 6))
    for k, (i, j) in enumerate(zip(bi, bj)):
        Bk = rng.normal(size=(6, 6))
        if i == j:
            Bk = Bk + Bk.T
        blocks[k] = Bk
        A[6 * i:6 * i + 6, 6 * j:6 * j + 6] = Bk
        A[6 * j:6 * j + 6, 6 * i:6 * i + 6] = Bk.T
    shift = np.abs(A).sum(axis=1).max() + 1.0
    dsq = np.full((n_cam, 6), shift)
    A = A + shift * np.eye(6 * n_cam)
    B = rng.normal(size=(n_cam, 6, 4))
    if fixed >= 0:
        B[fixed] = 0.0
    Bf = B.reshape(6 * n_cam, 4)
    G = rng.normal(size=(4, 4))
    C = Bf.T @ np.linalg.solve(A, Bf) + G @ G.T + np.eye(4)  # Schur complement of A stays SPD
    b = rng.normal(size=(n_cam, 6))
    bk = rng.normal(size=4)
    full = np.block([[A, Bf], [Bf.T, C]])
    ref = np.linalg.solve(full, np.concatenate([b.reshape(-1), bk]))
    return blocks, dsq, b, B, C, bk, ref


def _check(n_cam, bi, bj, fixed, seed, **kw):
    rng = np.random.default_rng(seed)
    sym = Symbolic(n_cam, bi, bj, **kw)
    blocks, dsq, b, B, C, bk, ref = _bordered_system(n_cam, bi, bj, fixed, rng)
    yc, yk = bordered_solve(sym, blocks, dsq, b, B, C, bk)
    got = np.concatenate([yc.reshape(-1), yk])
    assert np.max(np.abs(got - ref)) <= 1e-10 * np.max(np.abs(ref))
    return sym


def test_banded_sequence():
    p = syn.make_config(3, scale=0.05)
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    sym = _check(p.n_cam, bi, bj, p.fixed_cam, 3, leaf=8, cap=300)
    assert sym.n_levels >= 3


def test_small_leaves_deep_tree():
    seq = syn.make_tum_sequence(160, 8000, 24000, seed=17)
    w = syn.window_problem(seq, 0, 159).problem
    bi, bj = covisibility_blocks(w.cam_idx, w.pt_idx, w.n_cam, w.fixed_cam)
    deep = _check(w.n_cam, bi, bj, w.fixed_cam, 4, leaf=6, cap=760)
    wide = Symbolic(w.n_cam, bi, bj, leaf=32, cap=760)
    assert deep.n_nodes > wide.n_nodes and deep.n_levels > wide.n_levels


@pytest.mark.parametrize("fixed", [-1, 5])
def test_covisibility_in_several_trees(fixed):
    """Two unconnected halves, a loop closure inside each, and an isolated camera (damping only): a forest."""
    n = 60
    pairs = set((i, i) for i in range(n) if i != 17)
    for i in range(n):
        for d in (1, 2, 3):
            if i + d < n and i != 17 and i + d != 17 and not (i < 30 <= i + d):
                pairs.add((i, i + d))
    pairs.add((0, 29)); pairs.add((1, 28)); pairs.add((31, 59))
    pairs = sorted(pairs)
    bi = np.array([a for a, _ in pairs], dtype=np.int32)
    bj = np.array([b for _, b in pairs], dtype=np.int32)
    sym = _check(n, bi, bj, fixed, 6, leaf=6, cap=760)
    roots = int(np.sum(sym.node[:, 4] < 0))
    assert roots >= 2
