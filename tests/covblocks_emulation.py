"""numpy emulation of ba_gpu_covariance_blocks (csrc/ba_kernels_covblocks.cuh), driven by the symbolic structures the kernels
consume (spchol_emulation.Symbolic) and the panels of spchol_emulation.Multifrontal.

    [ A   B ]^-1        A = L L^T block-sparse (the tree), B: 6 x 4 per camera, C: 4 x 4
    [ B^T C ]

F_c = L^-1 E_c by the forward substitution along c's root path: at c's node the right-hand side is E_c on c's own rows, at
every later node it is the border part the child on the path carried up (through the child's rel / inv maps); the node solves
its own rows with L_OO and carries r_B - L_BO z_O to its parent.  Then (A^-1)_ab = sum over the nodes common to both paths of
F_a[n]^T F_b[n], and Sigma_cc(a, b) = (A^-1)_ab + X_a T^-1 X_b^T with X = A^-1 B, T = C - B^T X.  TEST INFRASTRUCTURE: the
kernels mirror these loops."""
import numpy as np

from spchol_emulation import INV, K0, M, NB, PARENT, REL, Multifrontal


class PathCovariance:
    def __init__(self, sym, blocks, dsq, B, C):
        self.sym = sym
        n = sym.n_cam
        order = [i for lvl in range(sym.n_levels) for i in sym.level_nodes[sym.level_ptr[lvl]:sym.level_ptr[lvl + 1]]]
        self.X = np.zeros((n, 6, 4))
        for q in range(4):  # X = L^-T (L^-1 B), one column at a time
            mf = Multifrontal(sym, blocks, dsq, B[:, :, q])
            mf.factor(order)
            mf.solve(order[::-1])
            self.X[:, :, q] = mf.y()
        self.panels = mf.panels
        self.Tinv = np.linalg.inv(C - np.einsum("cra,crb->ab", B, self.X))
        self.node_of = np.zeros(n, dtype=np.int64)
        for id_, N in enumerate(sym.node):
            self.node_of[N[K0]:N[K0] + N[M]] = id_
        self._F = {}

    def path(self, c):
        """Nodes from camera c's node to its root."""
        out, id_ = [], int(self.node_of[self.sym.pos[c]])
        while id_ >= 0:
            out.append(id_)
            id_ = int(self.sym.node[id_][PARENT])
        return out

    def forward(self, c):
        """{node: F_c on the node's own rows [6 m, 6]} for the nodes of c's path (F_c is zero elsewhere)."""
        if c in self._F:
            return self._F[c]
        sym, out = self.sym, {}
        carry, prev = None, None
        for id_ in self.path(c):
            N = sym.node[id_]
            k0, m, nb = N[K0], N[M], N[NB]
            P = self.panels[id_]
            r = np.zeros((6 * m, 6))
            rb = np.zeros((6 * nb, 6))
            if prev is None:
                q = sym.pos[c] - k0
                r[6 * q:6 * q + 6] = np.eye(6)
            else:
                Cn = sym.node[prev]
                rel = sym.rel[Cn[REL]:Cn[REL] + Cn[NB]]
                for i, ri in enumerate(rel):
                    if ri < m:
                        r[6 * ri:6 * ri + 6] = carry[6 * i:6 * i + 6]
                inv = sym.inv[Cn[INV]:Cn[INV] + nb]
                for i, ii in enumerate(inv):
                    if ii >= 0:
                        rb[6 * i:6 * i + 6] = carry[6 * ii:6 * ii + 6]
            z = np.zeros((6 * m, 6))
            for k in range(m):  # left-looking, with the inverse pivot block
                v = r[6 * k:6 * k + 6].copy()
                for j in range(k):
                    v -= P[k, j] @ z[6 * j:6 * j + 6]
                z[6 * k:6 * k + 6] = np.linalg.inv(P[k, k]) @ v
            for i in range(nb):
                for k in range(m):
                    rb[6 * i:6 * i + 6] -= P[m + i, k] @ z[6 * k:6 * k + 6]
            out[id_] = z
            carry, prev = rb, id_
        self._F[c] = out
        return out

    def a_inv(self, a, b):
        """(A^-1)(cam a, cam b): F_a^T F_b over the common part of the two root paths, root to lca."""
        Fa, Fb = self.forward(a), self.forward(b)
        pa, pb = self.path(a)[::-1], self.path(b)[::-1]
        s = np.zeros((6, 6))
        for na, nb_ in zip(pa, pb):
            if na != nb_:
                break
            s += Fa[na].T @ Fb[na]
        return s

    def cc(self, a, b):
        return self.a_inv(a, b) + self.X[a] @ self.Tinv @ self.X[b].T

    def full_column(self, c):
        """L^-1 E_c as a dense [6 n_cam, 6] array by elimination position."""
        out = np.zeros((6 * self.sym.n_cam, 6))
        for id_, z in self.forward(c).items():
            k0 = self.sym.node[id_][K0]
            out[6 * k0:6 * k0 + z.shape[0]] = z
        return out
