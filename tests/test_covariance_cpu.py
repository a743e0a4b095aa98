"""Covariance by selected inversion over the supernodal tree, on the CPU: the numpy emulation of ba_gpu_covariance's
recurrence (selinv_emulation, driven by the symbolic structures of libba_gpu.so) must equal the dense inverse of the whole
bordered system -- camera diagonal blocks, every stored block of S, the camera-intrinsics and intrinsics blocks -- on a banded
sequence, a deep tree and a forest with loop closures and an isolated camera."""
import numpy as np
import pytest

from helpers import ba_b200
from selinv_emulation import Covariance
from spchol_emulation import Symbolic, covisibility_blocks
from test_spchol_border_cpu import _bordered_system

syn = ba_b200.synthetic
TOL = 1e-10


def _check(n_cam, bi, bj, fixed, seed, **kw):
    rng = np.random.default_rng(seed)
    sym = Symbolic(n_cam, bi, bj, **kw)
    blocks, dsq, _, B, C, _, _ = _bordered_system(n_cam, bi, bj, fixed, rng)
    A = np.zeros((6 * n_cam, 6 * n_cam))
    for k, (i, j) in enumerate(zip(bi, bj)):
        A[6 * i:6 * i + 6, 6 * j:6 * j + 6] = blocks[k]
        A[6 * j:6 * j + 6, 6 * i:6 * i + 6] = blocks[k].T
    A += np.diag(dsq.reshape(-1))
    Bf = B.reshape(6 * n_cam, 4)
    inv = np.linalg.inv(np.block([[A, Bf], [Bf.T, C]]))
    cov = Covariance(sym, blocks, dsq, B, C)
    free = [c for c in range(n_cam) if c != fixed]

    def close(got, ref):
        got, ref = np.asarray(got), np.asarray(ref)
        assert np.max(np.abs(got - ref)) <= TOL * np.max(np.abs(ref))

    cam = lambda i, j: inv[6 * i:6 * i + 6, 6 * j:6 * j + 6]
    close([cov.cc(c, c) for c in free], [cam(c, c) for c in free])
    close([cov.cc(i, j) for i, j in zip(bi, bj)], [cam(i, j) for i, j in zip(bi, bj)])
    close([cov.cc(j, i) for i, j in zip(bi, bj)], [cam(j, i) for i, j in zip(bi, bj)])
    close([cov.ck(c) for c in free], [inv[6 * c:6 * c + 6, 6 * n_cam:] for c in free])
    close(cov.kk(), inv[6 * n_cam:, 6 * n_cam:])
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
    sym = _check(w.n_cam, bi, bj, w.fixed_cam, 4, leaf=6, cap=760)
    assert sym.n_levels >= 4


@pytest.mark.parametrize("fixed", [-1, 5])
def test_forest_with_loop_closures(fixed):
    """Two unconnected halves, a loop closure inside each, and an isolated camera (its diagonal only): a forest."""
    n = 60
    pairs = set((i, i) for i in range(n) if i != 17)
    for i in range(n):
        for d in (1, 2, 3):
            if i + d < n and i != 17 and i + d != 17 and not (i < 30 <= i + d):
                pairs.add((i, i + d))
    pairs.add((0, 29)); pairs.add((1, 28)); pairs.add((31, 59))
    if fixed >= 0:
        pairs = set((a, b) for a, b in pairs if a != fixed and b != fixed)
    pairs = sorted(pairs)
    bi = np.array([a for a, _ in pairs], dtype=np.int32)
    bj = np.array([b for _, b in pairs], dtype=np.int32)
    sym = _check(n, bi, bj, fixed, 6, leaf=6, cap=760)
    assert int(np.sum(sym.node[:, 4] < 0)) >= 2
