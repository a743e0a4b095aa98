"""numpy emulation of the covariance of ba_gpu_covariance (csrc/ba_kernels_selinv.cuh), driven by the symbolic structures the
kernels consume (csrc/ba_sparse_symbolic.h through the C-ABI, spchol_emulation.Symbolic).

    [ A   B ]^-1        A: block-sparse 6x6 blocks (the tree, A = L L^T), B: 6 x 4 per camera, C: 4 x 4
    [ B^T C ]

Selected inversion of A on the pattern of L, nodes top-down (Takahashi recurrence): with Y = L_BO L_OO^-1,
S_BO = -S_BB Y and S_OO = L_OO^-T L_OO^-1 - Y^T S_BO, S_BB gathered from the parent's front through `rel`.  Border:
X = A^-1 B (backward substitution per column), T = C - B^T X, Sigma_kk = T^-1, Sigma_ck = -X T^-1,
Sigma_cc(a, b) = (A^-1)_ab + X_a T^-1 X_b^T.  TEST INFRASTRUCTURE: the kernels mirror these loops."""
import numpy as np

from spchol_emulation import BORD, K0, M, NB, PARENT, REL, Multifrontal


def _dense(F, rows, cols, lower=False):
    out = np.zeros((6 * len(rows), 6 * len(cols)))
    for a, r in enumerate(rows):
        for b, c in enumerate(cols):
            if not lower or a >= b:
                out[6 * a:6 * a + 6, 6 * b:6 * b + 6] = F[r, c]
    return out


def selected_inverse(sym, panels):
    """panels[id] = F [m + nb, m, 6, 6] holding L after the factorisation -> fronts[id]: dense Sigma over the node's
    (own + border) cameras, i.e. the entries of A^-1 on the pattern of L."""
    fronts = [None] * sym.n_nodes
    order = [i for lvl in range(sym.n_levels - 1, -1, -1) for i in sym.level_nodes[sym.level_ptr[lvl]:sym.level_ptr[lvl + 1]]]
    for id_ in order:
        N = sym.node[id_]
        m, nb = N[M], N[NB]
        F = panels[id_]
        Loo = _dense(F, range(m), range(m), lower=True)
        Linv = np.linalg.inv(Loo)
        G = Linv.T @ Linv
        if nb == 0:
            fronts[id_] = G
            continue
        rel = sym.rel[N[REL]:N[REL] + nb]
        idx = (6 * rel[:, None] + np.arange(6)).reshape(-1)
        Sbb = fronts[N[PARENT]][np.ix_(idx, idx)]
        Y = _dense(F, range(m, m + nb), range(m)) @ Linv
        Sbo = -Sbb @ Y
        Soo = G - Y.T @ Sbo
        fronts[id_] = np.block([[Soo, Sbo.T], [Sbo, Sbb]])
    return fronts


class Covariance:
    """Sigma of the bordered system (A + diag(dsq) in the camera block) through the tree."""

    def __init__(self, sym, blocks, dsq, B, C):
        self.sym = sym
        n = sym.n_cam
        order = [i for lvl in range(sym.n_levels) for i in sym.level_nodes[sym.level_ptr[lvl]:sym.level_ptr[lvl + 1]]]
        self.X = np.zeros((n, 6, 4))
        panels = None
        for q in range(4):  # X = L^-T (L^-1 B), one column at a time
            mf = Multifrontal(sym, blocks, dsq, B[:, :, q])
            mf.factor(order)
            mf.solve(order[::-1])
            self.X[:, :, q] = mf.y()
            panels = mf.panels
        T = C - np.einsum("cra,crb->ab", B, self.X)
        self.Tinv = np.linalg.inv(T)
        self.fronts = selected_inverse(sym, panels)
        self.node_of = np.zeros(n, dtype=np.int64)
        for id_, N in enumerate(sym.node):
            self.node_of[N[K0]:N[K0] + N[M]] = id_

    def a_inv(self, i, j):
        """(A^-1)(cam i, cam j), for cameras whose positions share a front (a block of the pattern of L)."""
        sym = self.sym
        pi, pj = sym.pos[i], sym.pos[j]
        c, r = min(pi, pj), max(pi, pj)
        N = sym.node[self.node_of[c]]
        k0, m, nb = N[K0], N[M], N[NB]
        if r < k0 + m:
            lr = r - k0
        else:
            bord = list(sym.bord[N[BORD]:N[BORD] + nb])
            lr = m + bord.index(r)
        lc = c - k0
        blk = self.fronts[self.node_of[c]][6 * lr:6 * lr + 6, 6 * lc:6 * lc + 6]
        return blk if pi == r else blk.T

    def cc(self, i, j):
        return self.a_inv(i, j) + self.X[i] @ self.Tinv @ self.X[j].T

    def ck(self, i):
        return -self.X[i] @ self.Tinv

    def kk(self):
        return self.Tinv
