"""numpy emulation of the sparse Cholesky WITH the intrinsics border (csrc/ba_kernels_spchol.cuh, NR = 5 right-hand-side rows),
driven by the symbolic structures the kernels consume (csrc/ba_sparse_symbolic.h through the C-ABI, spchol_emulation.Symbolic).

    [ A   B ] [y_c]   [b_c]      A: block-sparse 6x6 blocks (the tree), B: 6 x 4 per camera, C: 4 x 4
    [ B^T C ] [y_k] = [b_k]

Forward substitution fused into the factorisation with five rows (z = L^-1 b_c, Z = L^-1 B), the border system
T y_k = t with T = C - Z^T Z and t = b_k - Z^T z, backward substitution L^T y_c = z - Z y_k.  TEST INFRASTRUCTURE: the
kernels mirror these loops."""
import numpy as np

from spchol_emulation import AENT, BORD, CHILD, INV, K0, M, NAENT, NB, NCHILD, REL

NR = 5


def _front_blocks(sym, N, blocks, dsq, F):
    for e in sym.aent[N[AENT]:N[AENT] + N[NAENT]]:
        code, lr, lc, cam = int(e[0]) & 0xffffffff, e[1], e[2], e[3]
        blk = code & 0x3fffffff
        if code & 0x40000000:
            Bd = np.zeros((6, 6))
            if blk != 0x3fffffff:
                up = np.triu(blocks[blk])
                Bd = up + np.triu(up, 1).T
            Bd = Bd + np.diag(dsq[cam])
        elif code & 0x80000000:
            Bd = blocks[blk].T
        else:
            Bd = blocks[blk]
        F[lr, lc] = Bd


def bordered_solve(sym, blocks, dsq, b, B, C, bk):
    """blocks [n_blk,6,6] stored upper blocks of A (without damping), dsq [n_cam,6], b [n_cam,6], B [n_cam,6,4], C [4,4],
    bk [4] -> (y_c [n_cam,6], y_k [4]) of the bordered system (A + diag(dsq) in the camera block)."""
    n = sym.n_cam
    rhs = np.concatenate([b[:, :, None], B], axis=2)  # (camera, component, row): row 0 = b_c, rows 1..4 = B
    panels, Us, rus = [None] * sym.n_nodes, [None] * sym.n_nodes, [None] * sym.n_nodes
    zpos = np.zeros((n, 6, NR))
    order = [i for lvl in range(sym.n_levels) for i in sym.level_nodes[sym.level_ptr[lvl]:sym.level_ptr[lvl + 1]]]
    for id_ in order:
        N = sym.node[id_]
        k0, m, nb = N[K0], N[M], N[NB]
        F = np.zeros((m + nb, m, 6, 6))
        zf = rhs[sym.perm[k0:k0 + m]].copy()
        _front_blocks(sym, N, blocks, dsq, F)
        for ch in sym.children[N[CHILD]:N[CHILD] + N[NCHILD]]:
            Cn = sym.node[ch]
            rel = sym.rel[Cn[REL]:Cn[REL] + Cn[NB]]
            for i in range(Cn[NB]):
                if rel[i] < m:
                    zf[rel[i]] -= rus[ch][i]
                for j in range(i + 1):
                    if rel[j] < m:
                        F[rel[i], rel[j]] -= Us[ch][i, j]
        for k in range(m):
            Lk = np.linalg.cholesky(F[k, k])
            T = np.linalg.inv(Lk)
            F[k, k] = Lk
            zf[k] = T @ zf[k]
            for r in range(k + 1, m + nb):
                F[r, k] = F[r, k] @ T.T
            for j in range(k + 1, m):
                zf[j] -= F[j, k] @ zf[k]
                for r in range(j, m + nb):
                    F[r, j] -= F[r, k] @ F[j, k].T
        zpos[k0:k0 + m] = zf
        U = np.zeros((nb, nb, 6, 6))
        ru = np.zeros((nb, 6, NR))
        for i in range(nb):
            for k in range(m):
                ru[i] += F[m + i, k] @ zf[k]
            for j in range(i + 1):
                for k in range(m):
                    U[i, j] += F[m + i, k] @ F[m + j, k].T
        for ch in sym.children[N[CHILD]:N[CHILD] + N[NCHILD]]:
            Cn = sym.node[ch]
            inv = sym.inv[Cn[INV]:Cn[INV] + nb]
            for i in range(nb):
                if inv[i] < 0:
                    continue
                ru[i] += rus[ch][inv[i]]
                for j in range(i + 1):
                    if inv[j] >= 0:
                        U[i, j] += Us[ch][inv[i], inv[j]]
        panels[id_], Us[id_], rus[id_] = F, U, ru
    # border system: sums over elimination positions in position order
    z, Z = zpos[:, :, 0], zpos[:, :, 1:]
    T = C - np.einsum("pra,prb->ab", Z, Z)
    t = bk - np.einsum("pra,pr->a", Z, z)
    L4 = np.linalg.cholesky(T)
    yk = np.linalg.solve(L4.T, np.linalg.solve(L4, t))
    # backward substitution with the right-hand side z - Z y_k
    w_all = z - Z @ yk
    ypos = np.zeros((n, 6))
    for id_ in order[::-1]:
        N = sym.node[id_]
        k0, m, nb = N[K0], N[M], N[NB]
        F = panels[id_]
        bord = sym.bord[N[BORD]:N[BORD] + nb]
        w = w_all[k0:k0 + m].copy()
        for k in range(m):
            for i in range(nb):
                w[k] -= F[m + i, k].T @ ypos[bord[i]]
        for k in range(m - 1, -1, -1):
            for r in range(k + 1, m):
                w[k] -= F[r, k].T @ ypos[k0 + r]
            ypos[k0 + k] = np.linalg.solve(F[k, k].T, w[k])
    yc = np.zeros((n, 6))
    yc[sym.perm] = ypos
    return yc, yk
