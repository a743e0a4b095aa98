"""Seeded problems whose co-visibility is not a band: loop closures, a street loop whose tracks wrap around, two unconnected maps,
and ragged inputs (a camera without observations, a camera with one, points seen once or never, duplicate observations).

The generators of synthetic.py make landmark tracks that are runs of consecutive cameras, so the reduced camera system S is
block-banded and the nested dissection of ba_sparse_symbolic.h always finds a narrow cut.  These problems reach the other
shapes of the symbolic phase: a range with no cut (eliminated as one chain), separators and borders with far cameras
(non-contiguous extend-add maps), forests, and cameras without a diagonal block.  Each generator asserts the shape it promises,
so that a silent change to it fails loudly.  CPU only."""
import numpy as np
import scipy.sparse as sps
from scipy.sparse.csgraph import connected_components

from helpers import ba_b200
from spchol_emulation import Symbolic, covisibility_blocks

syn = ba_b200.synthetic
# the device's symbolic phase (csrc/ba_gpu.cu build_spchol): leaves of 32 cameras, SPC_CAP_BLOCKS, SPC_MAX_OWN
GPU_LEAF, GPU_CAP, GPU_MAX_OWN = 32, 770, 24


def gpu_symbolic(p, leaf=GPU_LEAF):
    """The tree the device builds for problem p (same block list, same parameters)."""
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    return Symbolic(p.n_cam, bi, bj, leaf=leaf, cap=GPU_CAP, max_own=GPU_MAX_OWN)


def is_chain(sym):
    """No cut anywhere: the camera order is kept, and apart from the fixed camera (no block of S: a root of its own) every node is
    the only child of the next one, one node per level."""
    roots = int(np.sum(sym.node[:, 4] < 0))
    return np.array_equal(sym.perm, np.arange(sym.n_cam)) and roots == 2 and sym.n_levels == sym.n_nodes - 1


def _blocks(p):
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    return set(zip(bi.tolist(), bj.tolist()))


def n_components(p):
    """Connected components of the camera co-visibility graph (the fixed camera included, unobserved cameras alone)."""
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, -1)
    g = sps.coo_matrix((np.ones(len(bi)), (bi, bj)), shape=(p.n_cam, p.n_cam))
    return connected_components(g, directed=False)[0]


# ---------------------------------------------------------------- loop closures on a TUM-shaped sequence
def narrow_sequence(n_kf=120, seed=17):
    """Short tracks (about three keyframes, as tum_narrow) so that fronts with closure cameras still fit shared memory."""
    return syn.make_tum_sequence(n_kf, 60 * n_kf, 180 * n_kf, seed=seed)


def revisit(seq, closures, seed, per_cam=6):
    """A copy of `seq` where, for every closure (cameras A, cameras B), each camera of B observes `per_cam` landmarks of A and
    each camera of A observes `per_cam` landmarks of B.  The new observations are the truth landmark projected with the truth
    pose, with the pixel noise and depth quantisation of make_tum_sequence; the few that fall behind z = 0.2 are dropped.
    Observations stay camera-major, the seeded in-camera order of the old ones kept."""
    rng = np.random.default_rng(seed)
    K = seq.K
    new_kf, new_lm = [], []
    for A, B in closures:
        A, B = np.asarray(A), np.asarray(B)
        for src, dst in ((A, B), (B, A)):
            seen = np.unique(seq.lm[np.isin(seq.kf, src)])
            for c in dst:
                mine = set(seq.lm[seq.kf == c].tolist())
                cand = np.array([l for l in seen if l not in mine], dtype=np.int64)
                take = rng.choice(cand, size=min(per_cam, cand.size), replace=False)
                new_kf.append(np.full(take.size, c, dtype=np.int64))
                new_lm.append(take)
    kf, lm = np.concatenate(new_kf), np.concatenate(new_lm)
    uv, z = syn.project(seq.truth_pose[kf], seq.truth_pt[lm], K)
    front = z > 0.2
    # tum_trajectory keeps every camera in a 0.6 m box and within 0.05 rad per axis, landmarks lie 1-4 m deep: a keyframe sees
    # the landmarks of the others, the exceptions are few
    assert front.mean() > 0.9, front.mean()
    kf, lm, uv, z = kf[front], lm[front], uv[front], z[front]
    uv = (uv + 0.5 * rng.standard_normal(uv.shape)).astype(np.float32).astype(np.float64)
    dn = z + 0.003 * z * z * rng.standard_normal(z.shape)
    depth = (np.round(dn * 5000.0) / 5000.0).astype(np.float32).astype(np.float64)
    all_kf = np.concatenate([seq.kf.astype(np.int64), kf])
    order = np.argsort(all_kf, kind="stable")
    n_kf = seq.truth_pose.shape[0]
    kf_all = all_kf[order]
    out = syn.Sequence(seq.K.copy(), seq.truth_pose.copy(), seq.pose.copy(), seq.truth_pt.copy(), seq.pt.copy(),
                       kf_all.astype(np.int32), np.concatenate([seq.lm, lm.astype(np.int32)])[order],
                       np.concatenate([seq.uv, uv])[order], np.concatenate([seq.depth, depth])[order],
                       np.searchsorted(kf_all, np.arange(n_kf + 1)).astype(np.int64))
    assert np.all(np.diff(out.kf) >= 0)
    return out


def closure_problem(case, n_kf=120, seed=17):
    """REF / DEPTH window over all keyframes of a narrow sequence with loop closures:
    "a"  the first cameras <-> the last cameras: nested dissection finds no cut, the tree is one chain;
    "b"  a closure inside the first half: a wide separator there, an ordinary cut at the top;
    "c"  several closures, across the halves and inside them."""
    seq = narrow_sequence(n_kf, seed)
    n = n_kf
    closures = {"a": [(range(0, 3), range(n - 3, n))],
                "b": [(range(8, 10), range(n // 2 - 12, n // 2 - 10))],
                "c": [(range(2, 4), range(n - 30, n - 28)), (range(20, 22), range(n // 2 - 6, n // 2 - 4)),
                      (range(n // 2 + 8, n // 2 + 10), range(n - 5, n - 3))]}[case]
    p = syn.window_problem(revisit(seq, closures, seed + 1), 0, n - 1).problem
    blocks = _blocks(p)
    for A, B in closures:  # the closure blocks are present in S
        assert any((min(a, b), max(a, b)) in blocks for a in A for b in B if a != p.fixed_cam and b != p.fixed_cam)
    sym = gpu_symbolic(p)
    base = gpu_symbolic(syn.window_problem(seq, 0, n - 1).problem)
    if case == "a":
        assert is_chain(sym)
    else:
        assert not np.array_equal(sym.perm, np.arange(n)) and sym.n_levels < sym.n_nodes
        assert sym.info[7] > base.info[7]  # the closure widens a border
    return p


# ---------------------------------------------------------------- the street loop with wrapping tracks
def closed_street(n_cam=360, n_pt=3000, n_obs=15000, seed=41, extend=3):
    """The street loop of make_loop_problem (closed once n_cam >= 360), NS cost, except that tracks wrap modulo n_cam: every
    track that touches the first or the last `extend` cameras is continued across the seam by `extend` cameras.  The new
    observations project the truth point with the truth pose plus the loop's pixel noise."""
    assert n_cam >= 360
    rng = np.random.default_rng(seed)
    p = syn.make_loop_problem(n_cam, n_pt, n_obs, seed)
    truth_pose, truth_pt = p.meta["truth_pose"], p.meta["truth_pt"]
    lo = np.full(p.n_pt, n_cam, dtype=np.int64)
    hi = np.full(p.n_pt, -1, dtype=np.int64)
    np.minimum.at(lo, p.pt_idx, p.cam_idx)
    np.maximum.at(hi, p.pt_idx, p.cam_idx)
    new_cam, new_pt = [], []
    for q in np.flatnonzero(lo < extend):
        for k in range(1, extend + 1):
            new_cam.append(n_cam - k); new_pt.append(q)
    for q in np.flatnonzero(hi >= n_cam - extend):
        for k in range(extend):
            new_cam.append(k); new_pt.append(q)
    cam, pt = np.array(new_cam, dtype=np.int64), np.array(new_pt, dtype=np.int64)
    uv, z = syn.project(truth_pose[cam], truth_pt[pt], p.intr)
    assert np.min(z) > 0.5
    uv = uv + 0.5 * rng.standard_normal(uv.shape)
    all_cam = np.concatenate([p.cam_idx.astype(np.int64), cam])
    order = np.argsort(all_cam, kind="stable")
    q = p.copy()
    q.cam_idx = all_cam[order].astype(np.int32)
    q.pt_idx = np.concatenate([p.pt_idx, pt.astype(np.int32)])[order]
    q.uv2 = np.concatenate([p.uv2, uv])[order]
    assert q.depth is None
    blocks = _blocks(q)
    assert (1, n_cam - 1) in blocks  # tracks wrap (camera 0 is fixed: it has no block of S)
    sym = gpu_symbolic(q)
    assert is_chain(sym)  # a ring has no cut
    return q


# ---------------------------------------------------------------- forests
def two_maps(a, b):
    """Problems a and b side by side, sharing no point: camera fixed_cam of a is fixed, b's gauge is free."""
    q = a.copy()
    q.pose7 = np.concatenate([a.pose7, b.pose7])
    q.pt3 = np.concatenate([a.pt3, b.pt3])
    q.cam_idx = np.concatenate([a.cam_idx, b.cam_idx + a.n_cam]).astype(np.int32)
    q.pt_idx = np.concatenate([a.pt_idx, b.pt_idx + a.n_pt]).astype(np.int32)
    q.uv2 = np.concatenate([a.uv2, b.uv2])
    q.depth = None if a.depth is None else np.concatenate([a.depth, b.depth])
    assert n_components(q) == n_components(a) + n_components(b) == 2
    sym = gpu_symbolic(q)
    assert int(np.sum(sym.node[:, 4] < 0)) >= 2  # a forest: one root per map at least
    return q


def tum_window(n_kf, seed):
    seq = syn.make_tum_sequence(n_kf, 50 * n_kf, 300 * n_kf, seed=seed)
    return syn.window_problem(seq, 0, n_kf - 1).problem


# ---------------------------------------------------------------- ragged inputs
def ragged(p, empty_cam=None, one_obs_cam=None, once=0, unobserved=0, duplicates=0, seed=3):
    """A copy of p with any of: camera `empty_cam` without observations, camera `one_obs_cam` with a single one, `once` points
    seen once, `unobserved` points never seen, `duplicates` repeated (camera, point) observations (a shifted pixel, next to
    the original).  Camera-major order is kept."""
    rng = np.random.default_rng(seed)
    keep = np.ones(p.n_obs, dtype=bool)
    if empty_cam is not None:
        keep[p.cam_idx == empty_cam] = False
    if one_obs_cam is not None:
        keep[np.flatnonzero(p.cam_idx == one_obs_cam)[1:]] = False
    protect = np.isin(p.cam_idx, [c for c in (one_obs_cam,) if c is not None])
    pts = np.setdiff1d(np.arange(p.n_pt), p.pt_idx[protect])
    gone = rng.choice(pts, size=unobserved, replace=False)
    keep[np.isin(p.pt_idx, gone)] = False
    seen_once = rng.choice(np.setdiff1d(pts, gone), size=once, replace=False)
    for q in seen_once:
        keep[np.flatnonzero((p.pt_idx == q) & keep)[1:]] = False
    cam, pt, uv = p.cam_idx[keep], p.pt_idx[keep], p.uv2[keep]
    depth = None if p.depth is None else p.depth[keep]
    if duplicates:
        cand = np.flatnonzero(~np.isin(pt, seen_once) & (cam != (-1 if one_obs_cam is None else one_obs_cam)))
        dup = np.sort(rng.choice(cand, size=duplicates, replace=False))
        cam = np.insert(cam, dup + 1, cam[dup])
        pt = np.insert(pt, dup + 1, pt[dup])
        uv = np.insert(uv, dup + 1, uv[dup] + 0.25, axis=0)
        if depth is not None:
            depth = np.insert(depth, dup + 1, depth[dup])
    q = p.copy()
    q.cam_idx, q.pt_idx, q.uv2, q.depth = cam.astype(np.int32), pt.astype(np.int32), uv, depth
    assert np.all(np.diff(q.cam_idx) >= 0)
    per_cam = np.bincount(q.cam_idx, minlength=q.n_cam)
    per_pt = np.bincount(q.pt_idx, minlength=q.n_pt)
    if empty_cam is not None:
        assert per_cam[empty_cam] == 0
    if one_obs_cam is not None:
        assert per_cam[one_obs_cam] == 1
    assert np.all(per_pt[gone] == 0) and np.sum(per_pt == 0) >= unobserved
    assert np.all(per_pt[seen_once] == 1)
    pairs = q.cam_idx.astype(np.int64) * q.n_pt + q.pt_idx
    assert q.n_obs - np.unique(pairs).size >= duplicates
    return q
