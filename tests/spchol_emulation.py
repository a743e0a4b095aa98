"""numpy emulation of the numeric phase of the sparse Cholesky (csrc/ba_kernels_spchol.cuh), driven by the SAME symbolic
structures the kernels consume (csrc/ba_sparse_symbolic.h through the C-ABI).  TEST INFRASTRUCTURE: validates ordering,
supernodes, extend-add maps and entry lists on the CPU; the kernels mirror these loops."""
import ctypes as C

import numpy as np

from helpers import ba_b200

NI = 16
K0, M, NB, BORD, PARENT, LEVEL, CHILD, NCHILD, AENT, NAENT, REL, INV, PLO, PHI, ULO, UHI = range(16)


class Symbolic:
    def __init__(self, n_cam, bi, bj, leaf=32, cap=760, max_own=64):
        lib = ba_b200.capi.load()
        bi = np.ascontiguousarray(bi, dtype=np.int32)
        bj = np.ascontiguousarray(bj, dtype=np.int32)
        h = C.c_void_p()
        rc = lib.ba_sparse_symbolic_create(n_cam, len(bi), ba_b200.capi.ip(bi), ba_b200.capi.ip(bj), leaf, cap, max_own, C.byref(h))
        if rc:
            raise RuntimeError("ba_sparse_symbolic_create rc=%d" % rc)
        info = (C.c_int64 * 24)()
        lib.ba_sparse_symbolic_info(h, info)
        self.info = list(info)
        names = ["perm", "pos", "node", "bord", "children", "rel", "inv", "aent", "level_ptr", "level_nodes"]
        for w, name in enumerate(names):
            a = np.zeros(max(1, self.info[12 + w]), dtype=np.int32)
            lib.ba_sparse_symbolic_get(h, w, ba_b200.capi.ip(a))
            setattr(self, name, a[:self.info[12 + w]])
        self.n_cam, self.n_nodes, self.n_levels = self.info[0], self.info[1], self.info[2]
        self.partitions = {}
        for parts in (2, 3, 4, 8):  # subtree-to-rank partitions of the multi-GPU factorisation
            part = np.zeros(max(1, self.n_nodes), dtype=np.int32)
            work = np.zeros(3)
            got = lib.ba_sparse_symbolic_partition(h, parts, ba_b200.capi.ip(part), ba_b200.capi.dp(work))
            self.partitions[parts] = (got, part[:self.n_nodes].copy(), work.copy())
        self.queues = {}
        for n_sm in (148, 5):  # (a B200, and few SMs: more tiles per node on the upper levels)
            self.queues[("selinv", n_sm)] = _queue(lib, h, self.n_nodes, 1, 1, -1, n_sm)
            for parts in (1, 2, 3, 4, 8):  # work queues of k_spchol_tree: one GPU running every part, then each rank's own
                for rank in range(-1, parts if parts > 1 else 0):
                    self.queues[("chol", parts, rank, n_sm)] = _queue(lib, h, self.n_nodes, 0, parts, rank, n_sm)
        lib.ba_sparse_symbolic_destroy(h)
        self.node = self.node.reshape(-1, NI)
        self.aent = self.aent.reshape(-1, 4)
        self.bi, self.bj = bi, bj

    def stats(self):
        m, nb = self.node[:, M], self.node[:, NB]
        lev = np.diff(self.level_ptr)
        return dict(nodes=self.n_nodes, levels=self.n_levels, max_m=int(m.max()), max_nb=int(nb.max()), mean_m=float(m.mean()),
                    mean_nb=float(nb.mean()), max_front=self.info[5], panel_MB=self.info[3] * 288 / 1e6, u_MB=self.info[4] * 288 / 1e6,
                    gflop=self.info[9] / 1e9, crit_blocks=self.info[10], level_sizes=lev.tolist())


def _queue(lib, h, nn, which, parts, rank, n_sm):
    """One work queue through the C-ABI (ba_sparse_symbolic_queue): dict of items (n x 2: node, kind), tiles, and for the sparse
    Cholesky the parts in force, qA, qB, qB_n, cnt_init, topcams."""
    ip = ba_b200.capi.ip
    info = np.zeros(4, dtype=np.int32)
    got = lib.ba_sparse_symbolic_queue(h, which, parts, rank, n_sm, ip(info), None, None, None, None, None)
    if got < 1:
        raise RuntimeError("ba_sparse_symbolic_queue rc=%d" % got)
    q = np.zeros(2 * max(1, info[0]), dtype=np.int32)
    tiles = np.zeros(max(1, nn), dtype=np.int32)
    qA = np.zeros(got + 1, dtype=np.int32)
    cnt = np.zeros(3 * nn + 16, dtype=np.int32)
    top = np.zeros(max(1, info[3]), dtype=np.int32)
    lib.ba_sparse_symbolic_queue(h, which, parts, rank, n_sm, ip(info), ip(q), ip(tiles), ip(qA), ip(cnt), ip(top))
    out = dict(items=q[:2 * info[0]].reshape(-1, 2), tiles=tiles[:nn])
    if which == 0:
        out.update(parts=got, qA=qA, qB=int(info[1]), qB_n=int(info[2]), cnt_init=cnt, topcams=top[:info[3]])
    return out


def covisibility_blocks(cam_idx, pt_idx, n_cam, fixed_cam):
    """Upper blocks (i <= j) of S: camera pairs that share a point (free cameras only), sorted by (i, j)."""
    order = np.argsort(pt_idx, kind="stable")
    c, p = cam_idx[order].astype(np.int64), pt_idx[order]
    keep = c != fixed_cam
    c, p = c[keep], p[keep]
    keys = [c * n_cam + c]
    d = 1
    while True:
        same = p[d:] == p[:-d]
        if not same.any():
            break
        a, b = c[:-d][same], c[d:][same]
        keys.append(np.minimum(a, b) * n_cam + np.maximum(a, b))
        d += 1
    k = np.unique(np.concatenate(keys))
    return (k // n_cam).astype(np.int32), (k % n_cam).astype(np.int32)


class Multifrontal:
    """Numeric phase, node by node, with the state the kernels keep in global memory (panels, update matrices, rhs updates, z, y by
    position) -- so that the nodes can be processed in the groups of the distributed factorisation (own subtrees, exchange of the
    subtree roots' update matrices, top part, backward substitution top-down)."""

    def __init__(self, sym, blocks, dsq, b):
        self.sym, self.blocks, self.dsq, self.b = sym, blocks, dsq, b
        nn = sym.n_nodes
        self.panels, self.Us, self.rus = [None] * nn, [None] * nn, [None] * nn
        self.z = np.zeros((sym.n_cam, 6))      # by position
        self.ypos = np.zeros((sym.n_cam, 6))   # by position

    def nodes_bottom_up(self, keep):
        sym = self.sym
        return [id_ for lvl in range(sym.n_levels) for id_ in sym.level_nodes[sym.level_ptr[lvl]:sym.level_ptr[lvl + 1]] if keep(id_)]

    def factor(self, ids):
        sym, blocks, dsq, b = self.sym, self.blocks, self.dsq, self.b
        panels, Us, rus, z = self.panels, self.Us, self.rus, self.z
        for id_ in ids:
            N = sym.node[id_]
            k0, m, nb = N[K0], N[M], N[NB]
            F = np.zeros((m + nb, m, 6, 6))
            zf = np.zeros((m, 6))
            for q in range(m):
                zf[q] = b[sym.perm[k0 + q]]
            for e in sym.aent[N[AENT]:N[AENT] + N[NAENT]]:
                code, lr, lc, cam = int(e[0]) & 0xffffffff, e[1], e[2], e[3]
                blk = code & 0x3fffffff
                if code & 0x40000000:
                    B = np.zeros((6, 6))
                    if blk != 0x3fffffff:
                        up = np.triu(blocks[blk])
                        B = up + np.triu(up, 1).T
                    B = B + np.diag(dsq[cam])
                elif code & 0x80000000:
                    B = blocks[blk].T
                else:
                    B = blocks[blk]
                assert np.all(F[lr, lc] == 0.0)
                F[lr, lc] = B
            U = np.zeros((nb, nb, 6, 6))
            ru = np.zeros((nb, 6))
            for ch in sym.children[N[CHILD]:N[CHILD] + N[NCHILD]]:
                Cn = sym.node[ch]
                rel = sym.rel[Cn[REL]:Cn[REL] + Cn[NB]]
                for i in range(Cn[NB]):
                    if rel[i] < m:
                        zf[rel[i]] -= rus[ch][i]
                    for j in range(i + 1):
                        if rel[j] < m:
                            assert rel[i] >= rel[j]
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
            z[k0:k0 + m] = zf
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

    def solve(self, ids_top_down):
        sym, panels, z, ypos = self.sym, self.panels, self.z, self.ypos
        for id_ in ids_top_down:
            N = sym.node[id_]
            k0, m, nb = N[K0], N[M], N[NB]
            F = panels[id_]
            bord = sym.bord[N[BORD]:N[BORD] + nb]
            w = z[k0:k0 + m].copy()
            for k in range(m):
                for i in range(nb):
                    w[k] -= F[m + i, k].T @ ypos[bord[i]]
            for k in range(m - 1, -1, -1):
                for r in range(k + 1, m):
                    w[k] -= F[r, k].T @ ypos[k0 + r]
                ypos[k0 + k] = np.linalg.solve(F[k, k].T, w[k])

    def y(self):
        out = np.zeros((self.sym.n_cam, 6))
        out[self.sym.perm] = self.ypos
        return out


def factor_solve(sym, blocks, dsq, b):
    """blocks [n_blk,6,6] stored upper blocks of S, dsq [n_cam,6] damping, b [n_cam,6] -> y [n_cam,6]
    solving (S + diag(dsq)) y = b through the supernodal multifrontal scheme."""
    mf = Multifrontal(sym, blocks, dsq, b)
    order = mf.nodes_bottom_up(lambda id_: True)
    mf.factor(order)
    mf.solve(order[::-1])
    return mf.y()


def block_owner(sym, part):
    """Part that assembles every stored block of S (-1: top part): the part of the node that owns the earlier-eliminated of the
    block's two cameras -- the rule of build_spchol() (csrc/ba_gpu.cu) for the sparse exchange of S."""
    node_of = np.zeros(sym.n_cam, dtype=np.int64)
    for id_, N in enumerate(sym.node):
        node_of[N[K0]:N[K0] + N[M]] = id_
    return part[node_of[np.minimum(sym.pos[sym.bi], sym.pos[sym.bj])]]


def distributed_solve_inprocess(sym, part, world, blocks, dsq, b, touch):
    """The protocol of the distributed factorisation (DESIGN.md section 5) with the ranks simulated one after the other in this
    process: touch[r, blk] = rank r's points contribute to the block (contributions sum to `blocks`).  Returns (y, exchanged
    blocks of S).  Blocks a rank neither assembles itself nor shares in the top part are NaN for it."""
    owner = block_owner(sym, part)
    share = touch.sum(axis=0)
    assert (share > 0).all()
    local = [np.where(touch[r][:, None, None], blocks / share[:, None, None], 0.0) for r in range(world)]
    mask = np.zeros(len(blocks), dtype=bool)
    for r in range(world):
        mask |= touch[r] & (owner != r)
    summed = sum(l[mask] for l in local)
    mfs = []
    for r in range(world):
        S = local[r].copy()
        S[mask] = summed
        S[~((owner == r) | (owner == -1))] = np.nan
        mf = Multifrontal(sym, S, dsq, b)
        mf.factor(mf.nodes_bottom_up(lambda id_: part[id_] == r))
        mfs.append(mf)
    for id_, N in enumerate(sym.node):  # exchange of the subtree roots
        if part[id_] >= 0 and N[PARENT] >= 0 and part[N[PARENT]] == -1:
            src = mfs[part[id_]]
            for r in range(world):
                mfs[r].Us[id_], mfs[r].rus[id_] = src.Us[id_], src.rus[id_]
    ypos = np.zeros((sym.n_cam, 6))
    for r in range(world):
        mf = mfs[r]
        top = mf.nodes_bottom_up(lambda id_: part[id_] == -1)
        mf.factor(top)
        mf.solve(top[::-1])
        mf.solve(mf.nodes_bottom_up(lambda id_: part[id_] == r)[::-1])
        for id_, N in enumerate(sym.node):
            if part[id_] == r or (part[id_] == -1 and r == 0):
                ypos[N[K0]:N[K0] + N[M]] += mf.ypos[N[K0]:N[K0] + N[M]]
    y = np.zeros((sym.n_cam, 6))
    y[sym.perm] = ypos
    return y, int(mask.sum())
