"""Order of the work queues of the persistent tree kernels (csrc/ba_sparse_symbolic.h, spq_cholesky / spq_selinv, through the
C-ABI).  k_spchol_tree and k_selinv_tree hand their items out by a ticket counter and spin on completion counters: they
cannot deadlock only if every item an item waits for is earlier in the same launch or was done by an earlier launch over the
same counters.  This test restates each kernel's waits and checks that property, plus that every item is there exactly once
and that the tiles match tiles[].  CPU only."""
import numpy as np
import pytest

import irregular_problems as ip
from spchol_emulation import CHILD, K0, M, NB, NCHILD, PARENT, Symbolic, covisibility_blocks

syn = ip.syn
FACTOR, SOLVE, FINISH = -1, -2, -3   # (prepare is kind -1 of the selected inversion's queue)
PRESET = 1 << 20                     # cnt_init: "all update tiles done" for a subtree root another rank factorises


def _waits_cholesky(sym, tiles, it):
    """What k_spchol_tree waits for before item `it`: (counter, node, count) triples."""
    n, kind = it
    if kind == FACTOR:
        # every tile of every child.  (The kernel waits for udone >= tiles[child]; a child has a border, so at least one tile:
        # a child without tiles here is one this queue never factorises, and its update matrix must come from the exchange.)
        lo, cnt = sym.node[n][CHILD], sym.node[n][NCHILD]
        return [("udone", c, max(1, tiles[c])) for c in sym.children[lo:lo + cnt]]
    if kind == SOLVE:
        par = sym.node[n][PARENT]
        return [("sdone", par, 1)] if par >= 0 else [("fdone", n, 1)]
    return [("fdone", n, 1)]                                   # update tile


def _waits_selinv(sym, tiles, it):
    n, kind = it
    if kind == FACTOR:                                         # prepare: the parent's Sigma front
        par = sym.node[n][PARENT]
        return [("sdone", par, 1)] if par >= 0 else []
    if kind == FINISH:
        return [("pdone", n, 1), ("tdone", n, tiles[n])]
    return [("pdone", n, 1)]                                   # product tile


def _publishes(it, selinv):
    n, kind = it
    if kind >= 0:
        return ("tdone" if selinv else "udone"), n
    return {FACTOR: "pdone" if selinv else "fdone", SOLVE: "sdone", FINISH: "sdone"}[kind], n


def _run(sym, items, tiles, launches, selinv=False, counters=None, between=None):
    """Runs the launches in queue order (one valid schedule of the persistent grid) on the completion counters and asserts
    that every wait is met by then.  between(k, counters) runs after launch k (the exchange, a counter reset)."""
    cnt = counters if counters is not None else {}
    waits = _waits_selinv if selinv else _waits_cholesky
    for k, (first, n) in enumerate(launches):
        for i in range(first, first + n):
            it = (int(items[i][0]), int(items[i][1]))
            for name, node, want in waits(sym, tiles, it):
                assert cnt.get((name, node), 0) >= want, "item %d %s waits for %s of node %d" % (i, it, name, node)
            c = _publishes(it, selinv)
            cnt[c] = cnt.get(c, 0) + 1
        if between:
            between(k, cnt)
    return cnt


def _expected(sym, tiles, nodes, kinds):
    want = []
    for n in nodes:
        for kind in kinds:
            want += [(n, t) for t in range(tiles[n])] if kind == 0 else [(n, kind)]
    return sorted(want)


def _check_tiles(sym, tiles, nodes):
    for n in range(sym.n_nodes):
        if n in nodes:
            assert (tiles[n] > 0) == (sym.node[n][NB] > 0) and tiles[n] <= 8, (n, tiles[n])
        else:
            assert tiles[n] == 0, n


def _check_cholesky(sym, parts, rank, n_sm):
    Q = sym.queues[("chol", parts, rank, n_sm)]
    items, tiles, P = Q["items"], Q["tiles"], Q["parts"]
    part = sym.partitions[parts][1] if P > 1 else np.zeros(sym.n_nodes, dtype=np.int32)
    qA, qB, qB_n = Q["qA"], Q["qB"], Q["qB_n"]
    assert qA[0] == 0 and np.all(np.diff(qA) >= 0) and qA[P] == qB and qB + qB_n == len(items)
    me = rank if (rank >= 0 and P == parts) else -1
    mine = [n for n in range(sym.n_nodes) if part[n] < 0 or me < 0 or part[n] == me]
    # every item of the nodes this GPU runs, exactly once; tiles as announced
    got = sorted((int(a), int(b)) for a, b in items)
    assert got == _expected(sym, tiles, mine, (FACTOR, 0, SOLVE))
    _check_tiles(sym, tiles, set(mine))
    # phase A holds factor and update items only, the top part's are in phase B
    assert all(items[i][1] != SOLVE and part[items[i][0]] >= 0 for i in range(qB))
    # counters before a solve: presets exactly for the other ranks' nodes; the cameras of the top part
    cnt0 = Q["cnt_init"]
    others = [n for n in range(sym.n_nodes) if me >= 0 and part[n] >= 0 and part[n] != me]
    assert np.all(cnt0[:16 + sym.n_nodes] == 0) and np.all(cnt0[16 + 2 * sym.n_nodes:] == 0)
    assert sorted(np.flatnonzero(cnt0[16 + sym.n_nodes:16 + 2 * sym.n_nodes]).tolist()) == others
    assert np.all(cnt0[16 + sym.n_nodes + np.array(others, dtype=np.int64)] == PRESET)
    top = [int(sym.perm[k]) for n in range(sym.n_nodes) if part[n] < 0 for k in range(sym.node[n][K0], sym.node[n][K0] + sym.node[n][M])]
    assert Q["topcams"].tolist() == (top if P > 1 else [])
    preset = {("udone", n): PRESET for n in others}
    if P == 1:
        # one launch; or the factor prefix, then the backward substitution (intrinsics border of the LM step)
        _run(sym, items, tiles, [(0, len(items))])
        _run(sym, items, tiles, [(0, qB), (qB, qB_n)])
        # the covariance's border columns: one factor launch, then the solve suffix once per column with only sdone reset
        def reset_sdone(k, cnt):
            for key in [key for key in cnt if key[0] == "sdone"]:
                del cnt[key]
        _run(sym, items, tiles, [(0, qB)] + [(qB, qB_n)] * 4, between=reset_sdone)
    else:
        # phase A part by part (on this GPU's counters), the exchange, phase B
        launches = [(qA[p], qA[p + 1] - qA[p]) for p in range(P)] + [(qB, qB_n)]
        _run(sym, items, tiles, launches, counters=dict(preset))


def _check_selinv(sym, n_sm):
    Q = sym.queues[("selinv", n_sm)]
    items, tiles = Q["items"], Q["tiles"]
    got = sorted((int(a), int(b)) for a, b in items)
    assert got == _expected(sym, tiles, range(sym.n_nodes), (FACTOR, 0, FINISH))
    _check_tiles(sym, tiles, set(range(sym.n_nodes)))
    _run(sym, items, tiles, [(0, len(items))], selinv=True)


def _check_all(sym):
    for n_sm in (148, 5):
        _check_selinv(sym, n_sm)
        _check_cholesky(sym, 1, -1, n_sm)
        for parts in (2, 3, 4, 8):
            for rank in range(-1, parts):
                _check_cholesky(sym, parts, rank, n_sm)


# small trees with small fronts (as test_sparse_symbolic.py), and the full-size configs with the device's parameters
@pytest.mark.parametrize("cfg,scale,leaf,cap,max_own", [(3, 0.05, 8, 300, 64), (4, 0.05, 8, 300, 64), (4, 0.1, 16, 300, 64),
                                                       (3, 1.0, ip.GPU_LEAF, ip.GPU_CAP, ip.GPU_MAX_OWN),
                                                       (4, 1.0, ip.GPU_LEAF, ip.GPU_CAP, ip.GPU_MAX_OWN)])
def test_banded_configs(cfg, scale, leaf, cap, max_own):
    p = syn.make_config(cfg, scale=scale)
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    sym = Symbolic(p.n_cam, bi, bj, leaf=leaf, cap=cap, max_own=max_own)
    assert sym.n_levels >= 3 and any(sym.partitions[k][0] == k for k in (2, 3, 4, 8))
    _check_all(sym)


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_loop_closures(case):
    p = ip.closure_problem(case)
    _check_all(ip.gpu_symbolic(p))
    _check_all(ip.gpu_symbolic(p, leaf=6))


def test_closed_street():
    _check_all(ip.gpu_symbolic(ip.closed_street()))


def test_forest():
    _check_all(ip.gpu_symbolic(ip.two_maps(ip.tum_window(12, 5), ip.tum_window(10, 6)), leaf=4))


def test_ragged():
    q = ip.ragged(ip.tum_window(12, 5), empty_cam=3, one_obs_cam=7, once=20, unobserved=5, duplicates=10)
    _check_all(ip.gpu_symbolic(q, leaf=4))
