"""Covariance of any two cameras by sparse forward solves on the supernodal Cholesky, on the CPU: the numpy emulation of
ba_gpu_covariance_blocks' path products (covblocks_emulation, driven by the symbolic structures of libba_gpu.so) must equal the
dense inverse of the whole bordered system for EVERY camera pair -- also the pairs that share no block of S, and pairs across
the trees of a forest -- and L^-1 E_c must vanish outside the own rows of c's root path.  The cases are those of
test_covariance_cpu.py."""
import numpy as np
import pytest

from covblocks_emulation import PathCovariance
from helpers import ba_b200
from spchol_emulation import K0, M, Symbolic, covisibility_blocks
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
    full = np.block([[A, Bf], [Bf.T, C]])
    inv = np.linalg.inv(full)
    ainv = np.linalg.inv(A)
    cov = PathCovariance(sym, blocks, dsq, B, C)
    free = [c for c in range(n_cam) if c != fixed]
    scale = np.max(np.abs(inv))
    err_a = err_cc = 0.0
    for a in free:
        for b in free:
            err_cc = max(err_cc, np.max(np.abs(cov.cc(a, b) - inv[6 * a:6 * a + 6, 6 * b:6 * b + 6])))
            err_a = max(err_a, np.max(np.abs(cov.a_inv(a, b) - ainv[6 * a:6 * a + 6, 6 * b:6 * b + 6])))
    assert err_cc <= TOL * scale and err_a <= TOL * np.max(np.abs(ainv)), (err_cc, err_a)
    # L^-1 E_c is zero outside the own rows of the nodes on c's root path
    for c in free:
        rows = np.zeros(6 * n_cam, dtype=bool)
        for id_ in cov.path(c):
            N = sym.node[id_]
            rows[6 * N[K0]:6 * (N[K0] + N[M])] = True
        col = cov.full_column(c)
        assert not col[~rows].any()
        # and it is L^-1 E_c: L (L^-1 E_c) = E_c in elimination order
        Ap = A[np.ix_((6 * sym.perm[:, None] + np.arange(6)).reshape(-1), (6 * sym.perm[:, None] + np.arange(6)).reshape(-1))]
        L = np.linalg.cholesky(Ap)
        E = np.zeros((6 * n_cam, 6))
        E[6 * sym.pos[c] + np.arange(6), np.arange(6)] = 1.0
        assert np.max(np.abs(L @ col - E)) <= 1e-12 * max(1.0, np.max(np.abs(L)))
        break  # (one dense Cholesky is enough: the emulation is the same code for every camera)
    return sym, cov


def _far_pairs(cov, free, bi, bj):
    """Free camera pairs that share no block of S (the ones ba_gpu_covariance rejects)."""
    blocks = set(zip(bi.tolist(), bj.tolist()))
    return [(a, b) for a in free for b in free if a < b and (a, b) not in blocks]


def test_banded_sequence():
    p = syn.make_config(3, scale=0.05)
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    sym, _ = _check(p.n_cam, bi, bj, p.fixed_cam, 3, leaf=8, cap=300)
    assert sym.n_levels >= 3


def test_small_leaves_deep_tree():
    seq = syn.make_tum_sequence(160, 8000, 24000, seed=17)
    w = syn.window_problem(seq, 0, 159).problem
    bi, bj = covisibility_blocks(w.cam_idx, w.pt_idx, w.n_cam, w.fixed_cam)
    sym, cov = _check(w.n_cam, bi, bj, w.fixed_cam, 4, leaf=6, cap=760)
    assert sym.n_levels >= 4
    assert _far_pairs(cov, [c for c in range(w.n_cam) if c != w.fixed_cam], bi, bj)  # (the check covered pairs outside S)


@pytest.mark.parametrize("fixed", [-1, 5])
def test_forest_with_loop_closures(fixed):
    """Two unconnected halves, a loop closure inside each, and an isolated camera: pairs across the trees are zero in A^-1
    (only the border term remains)."""
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
    sym, cov = _check(n, bi, bj, fixed, 6, leaf=6, cap=760)
    assert int(np.sum(sym.node[:, 4] < 0)) >= 2
    # across the two halves the paths meet no common node: A^-1 vanishes there
    a, b = 3, 40
    assert cov.path(a)[-1] != cov.path(b)[-1]
    assert not cov.a_inv(a, b).any()


def test_cov_block_layout_matches_header(tmp_path):
    """The ctypes mirror of ba_cov_block and the BA_COV_* kinds against the C compiler's view of include/ba_gpu.h."""
    import ctypes as C
    import os
    import subprocess
    capi = ba_b200.capi
    src = tmp_path / "cb.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ba_gpu.h"\nint main(){printf("%zu %zu %zu %d %d %d\\n",'
                   'sizeof(ba_cov_block),offsetof(ba_cov_block,kind),offsetof(ba_cov_block,index),'
                   'BA_COV_CAMERA,BA_COV_POINT,BA_COV_INTRINSICS);return 0;}\n')
    exe = tmp_path / "cb"
    subprocess.check_call(["gcc", "-I", os.path.dirname(capi.HEADER_PATH), str(src), "-o", str(exe)])
    size, o_kind, o_index, cam, pt, intr = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert C.sizeof(capi.CovBlock) == size
    assert capi.CovBlock.kind.offset == o_kind and capi.CovBlock.index.offset == o_index
    assert (capi.BA_COV_CAMERA, capi.BA_COV_POINT, capi.BA_COV_INTRINSICS) == (cam, pt, intr)
