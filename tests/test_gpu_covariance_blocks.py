"""ba_gpu_covariance_blocks / GpuSolver.covariance_blocks: the covariance of ANY pair of parameter blocks (camera pairs that
share no point, camera-point, point-point, intrinsics) by sparse forward solves on the supernodal Cholesky.  The independent
reference is numpy from the ORACLE's Jacobians at the state downloaded from the GPU (test_gpu_covariance's Hessian and reduced
system; at cfg1 the dense inverse of the whole Hessian)."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla

import irregular_problems as ip
from helpers import ba_b200, mode_opts
from spchol_emulation import covisibility_blocks
from test_gpu_covariance import TOL, TOL_INTR, _hessian, _pairs, _reduced, _rel
from test_gpu_spchol_border import N_KF_BIG, _big_sequence, _problem

pytestmark = pytest.mark.gpu
capi = ba_b200.capi
DIM = {"cam": 6, "pt": 3, "intr": 4}


def _solver(mode, **kw):
    g, _ = mode_opts(mode, **kw)
    return ba_b200.GpuSolver(**g)


class _Ref:
    """Sigma of the whole Hessian from the oracle's Jacobians: Sigma_RR (equilibrated dense inverse of the reduced system),
    Sigma(R, p) = -Sigma_RR W_p V_p^-1, Sigma(p, q) = delta_pq V_p^-1 + V_p^-1 W_p^T Sigma_RR W_q V_q^-1."""

    def __init__(self, p, mode, pose, pt, intr, full=False):
        H, self.nR, self.nk, self.slot = _hessian(p, mode, pose, pt, intr)
        S, self.Vi, Hrp = _reduced(H, self.nR, p.n_pt)
        Sd = S.toarray()
        d = 1.0 / np.sqrt(np.diag(Sd))
        self.Srr = d[:, None] * np.linalg.inv(d[:, None] * Sd * d[None, :]) * d[None, :]
        self.Hrp = Hrp.toarray()
        self.Hi = np.linalg.inv(H.toarray()) if full else None

    def _cols(self, k, i):
        """Columns of block (k, i) in the reduced unknowns (None: a constant block)."""
        if k == "cam":
            return None if self.slot[i] < 0 else 6 * self.slot[i] + np.arange(6)
        return None if self.nk == 0 else self.nR - 4 + np.arange(4)

    def block(self, a, b):
        (ka, ia), (kb, ib) = a, b
        out = np.zeros((DIM[ka], DIM[kb]))
        if self.Hi is not None:  # the dense inverse of the whole Hessian
            ra, rb = self._full(ka, ia), self._full(kb, ib)
            return out if ra is None or rb is None else self.Hi[np.ix_(ra, rb)]
        if ka == "pt" and kb == "pt":
            Wa, Wb = self.Hrp[:, 3 * ia:3 * ia + 3], self.Hrp[:, 3 * ib:3 * ib + 3]
            return (self.Vi[ia] if ia == ib else 0.0) + self.Vi[ia] @ Wa.T @ self.Srr @ Wb @ self.Vi[ib]
        if kb == "pt":
            ca = self._cols(ka, ia)
            return out if ca is None else -self.Srr[ca] @ self.Hrp[:, 3 * ib:3 * ib + 3] @ self.Vi[ib]
        if ka == "pt":
            return self.block(b, a).T
        ca, cb = self._cols(ka, ia), self._cols(kb, ib)
        return out if ca is None or cb is None else self.Srr[np.ix_(ca, cb)]

    def _full(self, k, i):
        if k == "pt":
            return self.nR + 3 * i + np.arange(3)
        return self._cols(k, i)


def _err(got, ref):
    return _rel(np.concatenate([g.reshape(-1) for g in got]), np.concatenate([r.reshape(-1) for r in ref]))


def _check(name, mode, groups, got, ref):
    """groups: {label: request list}; got: the blocks in the order of the concatenated groups."""
    errs, o = {}, 0
    for label, req in groups.items():
        errs[label] = _err(got[o:o + len(req)], [ref.block(a, b) for a, b in req])
        o += len(req)
    print("covariance_blocks max relative error %s %s: %s" % (name, mode, " ".join("%s=%.2e" % kv for kv in sorted(errs.items()))))
    for label, e in errs.items():
        # REF: every block carries the intrinsics border (X T^-1 X^T), the ill-conditioned direction of the system
        assert e <= (TOL_INTR if mode == "REF" else TOL), (label, e)


def _run(p, mode, req, iters=4, solver=4):
    s = _solver(mode, solver=solver, max_num_iterations=iters)
    try:
        s.upload(p)
        if iters:
            s.solve()
        got = s.covariance_blocks(req)
        state = tuple(x.copy() for x in s.download())
    finally:
        s.close()
    return got, state


def _far_pairs(p):
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    blocks = set(zip(bi.tolist(), bj.tolist()))
    free = [c for c in range(p.n_cam) if c != p.fixed_cam]
    return [(a, b) for a in free for b in free if a < b and (a, b) not in blocks]


def _sample(rng, n, k):
    return rng.choice(n, size=min(n, k), replace=False)


# ---------------------------------------------------------------- 1. cfg1: every block kind against the dense inverse of H
@pytest.mark.parametrize("mode", ["REF", "DEPTH"])
def test_cfg1_every_kind_against_dense_inverse(mode):
    p = _problem("cfg1")
    rng = np.random.default_rng(1)
    cams = [("cam", c) for c in range(p.n_cam)]
    pts = [("pt", i) for i in range(p.n_pt)]
    K = ("intr", 0)
    groups = dict(cam_cam=[(a, b) for a in cams for b in cams],
                  cam_pt=[(a, b) for a in cams for b in pts],
                  pt_cam=[(b, a) for a in cams[:2] for b in pts[:50]],
                  cam_intr=[(a, K) for a in cams] + [(K, a) for a in cams],
                  intr=[(K, K)],
                  pt_intr=[(b, K) for b in pts] + [(K, b) for b in pts[:20]],
                  pt_diag=[(b, b) for b in pts],
                  pt_pt=[(pts[i], pts[j]) for i, j in zip(rng.integers(0, p.n_pt, 300), rng.integers(0, p.n_pt, 300))])
    req = [r for g in groups.values() for r in g]
    got, (pose, pt, intr) = _run(p, mode, req)
    _check("cfg1", mode, groups, got, _Ref(p, mode, pose, pt, intr, full=True))


# ---------------------------------------------------------------- 2. pairs that share no point, camera-point, point-point
@pytest.mark.parametrize("mode", ["REF", "DEPTH"])
@pytest.mark.parametrize("name", ["window20", "tum0.1"])
def test_far_pairs_and_points_against_numpy(name, mode):
    p = _problem(name)
    rng = np.random.default_rng(2)
    far = _far_pairs(p)
    if name == "window20":  # (every camera pair of the window shares a point: then every pair)
        assert not far
        far = [(a, b) for a in range(p.n_cam) for b in range(a + 1, p.n_cam) if p.fixed_cam not in (a, b)]
    assert far
    if len(far) > 2000:  # the farthest pairs, then a seeded sample (tum0.1 has fewer: all of them)
        far.sort(key=lambda ab: ab[1] - ab[0])
        keep = far[-200:]
        far = keep + [far[i] for i in _sample(rng, len(far) - 200, 1800)]
    groups = dict(far=[(("cam", a), ("cam", b)) for a, b in far],
                  far_t=[(("cam", b), ("cam", a)) for a, b in far[:100]],
                  cam_pt=[(("cam", int(c)), ("pt", int(q))) for c, q in zip(rng.integers(0, p.n_cam, 1000), rng.integers(0, p.n_pt, 1000))],
                  pt_pt=[(("pt", int(a)), ("pt", int(b))) for a, b in zip(rng.integers(0, p.n_pt, 1000), rng.integers(0, p.n_pt, 1000))],
                  pt_intr=[(("pt", int(a)), ("intr", 0)) for a in rng.integers(0, p.n_pt, 200)])
    req = [r for g in groups.values() for r in g]
    got, (pose, pt, intr) = _run(p, mode, req)
    _check(name, mode, groups, got, _Ref(p, mode, pose, pt, intr))


# ---------------------------------------------------------------- 3. loop closures
@pytest.mark.parametrize("name", ["closure_a", "closure_b", "closure_c"])
def test_closures(name):
    p = ip.closure_problem(name[-1])
    far = _far_pairs(p)
    across = [(a, b) for a, b in far if b - a > p.n_cam // 2][:400]  # across the closures
    free = [c for c in range(p.n_cam) if c != p.fixed_cam]
    groups = dict(across=[(("cam", a), ("cam", b)) for a, b in across],
                  ends=[(("cam", free[0]), ("cam", p.n_cam - 1)), (("cam", p.n_cam - 1), ("cam", free[0]))])
    req = [r for g in groups.values() for r in g]
    got, (pose, pt, intr) = _run(p, "REF", req)
    _check(name, "REF", groups, got, _Ref(p, "REF", pose, pt, intr))


# ---------------------------------------------------------------- 4. one camera's full row beyond the dense limit
def test_big_sequence_row_against_sparse_lu():
    seq = _big_sequence()
    p = ba_b200.synthetic.window_problem(seq, 0, N_KF_BIG - 1).problem
    c0 = N_KF_BIG // 2
    req = [(("cam", c0), ("cam", c)) for c in range(p.n_cam)]  # more sources than one pass holds
    s = _solver("REF")  # AUTO
    try:
        s.upload(p)
        got = s.covariance_blocks(req)
        rng = np.random.default_rng(4)
        one = {int(c): s.covariance_blocks([req[c]])[0] for c in _sample(rng, p.n_cam, 12)}
        pose, pt, intr = (x.copy() for x in s.download())
    finally:
        s.close()
    for c, blk in one.items():  # one block per call: the same bits as inside the row
        assert np.array_equal(blk, got[c]), c
    H, nR, nk, slot = _hessian(p, "REF", pose, pt, intr)
    S, _, _ = _reduced(H, nR, p.n_pt)
    E = np.zeros((nR, 6))
    E[6 * slot[c0] + np.arange(6), np.arange(6)] = 1.0
    col = spla.splu(S).solve(E)  # Sigma[:, c0]
    ref = [np.zeros((6, 6)) if slot[c] < 0 else col[6 * slot[c]:6 * slot[c] + 6].T for c in range(p.n_cam)]
    e = _err(got, ref)
    print("covariance_blocks max relative error big%d row %d: %.2e" % (N_KF_BIG, c0, e))
    assert e <= TOL_INTR
    assert not got[p.fixed_cam].any()


# ---------------------------------------------------------------- 5. agreement with ba_gpu_covariance
def test_agrees_with_selected_inversion():
    p = ip.closure_problem("c")
    pr = _pairs(p)
    s = _solver("REF", solver=4)
    try:
        s.upload(p)
        cov = s.covariance(points=True, pairs=pr)
        K = ("intr", 0)
        req = ([(("cam", c), ("cam", c)) for c in range(p.n_cam)] + [(("cam", int(a)), ("cam", int(b))) for a, b in pr]
               + [(("cam", c), K) for c in range(p.n_cam)] + [(K, K)] + [(("pt", i), ("pt", i)) for i in range(p.n_pt)])
        got = s.covariance_blocks(req)
    finally:
        s.close()
    n, m = p.n_cam, len(pr)
    err = dict(cam=_err(got[:n], cov["cam"]), pairs=_err(got[n:n + m], cov["pairs"]),
               cam_intr=_err(got[n + m:2 * n + m], cov["cam_intr"]), intr=_err([got[2 * n + m]], [cov["intr"]]),
               pt=_err(got[2 * n + m + 1:], cov["pt"]))
    for k, e in err.items():
        print("covariance_blocks against ba_gpu_covariance closure_c %s: %.2e" % (k, e))
    for k, e in err.items():
        assert e <= (1e-9 if k == "pt" else 1e-10), (k, e)


# ---------------------------------------------------------------- 6. call-level properties
def _mixed_requests(p, seed):
    rng = np.random.default_rng(seed)
    K = ("intr", 0)
    req = [(("cam", int(a)), ("cam", int(b))) for a, b in zip(rng.integers(0, p.n_cam, 60), rng.integers(0, p.n_cam, 60))]
    req += [(("cam", int(a)), ("pt", int(b))) for a, b in zip(rng.integers(0, p.n_cam, 60), rng.integers(0, p.n_pt, 60))]
    req += [(("pt", int(a)), ("pt", int(b))) for a, b in zip(rng.integers(0, p.n_pt, 60), rng.integers(0, p.n_pt, 60))]
    req += [(("pt", int(a)), K) for a in rng.integers(0, p.n_pt, 10)] + [(("cam", 3), K), (K, K)]
    req += [(("cam", c), ("cam", c)) for c in range(p.n_cam)] + [(("pt", int(a)),) * 2 for a in rng.integers(0, p.n_pt, 40)]
    return req


def test_determinism_permutation_transpose_definiteness():
    p = _problem("tum0.1")
    req = _mixed_requests(p, 6)
    perm = np.random.default_rng(7).permutation(len(req))
    s = _solver("REF", solver=4, max_num_iterations=3)
    try:
        s.upload(p)
        s.solve()
        a = s.covariance_blocks(req)
        b = s.covariance_blocks(req)
        c = s.covariance_blocks([req[i] for i in perm])
        t = s.covariance_blocks([(y, x) for x, y in req])
    finally:
        s.close()
    for i in range(len(req)):
        assert np.array_equal(a[i], b[i]), i
        assert np.array_equal(c[list(perm).index(i)], a[i]), i
        assert np.array_equal(t[i], a[i].T), i
        x, y = req[i]
        if x == y and not (x[0] == "cam" and x[1] == p.fixed_cam):
            assert np.array_equal(a[i], a[i].T) and np.linalg.eigvalsh(a[i]).min() > 0.0, req[i]


@pytest.mark.parametrize("name", ["window20", "closure_a"])
def test_auto_and_sparse_cholesky_bit_identical(name):
    p = ip.closure_problem("a") if name == "closure_a" else _problem(name)
    req = _mixed_requests(p, 8)
    got = []
    for solver in (0, 4):
        g, _ = _run(p, "REF", req, iters=0, solver=solver)
        got.append(g)
    for i, (x, y) in enumerate(zip(*got)):
        assert np.array_equal(x, y), req[i]


def test_fixed_camera_and_constant_intrinsics_are_zero():
    p = _problem("window20")
    f = p.fixed_cam
    K = ("intr", 0)
    req = [(("cam", f), ("cam", f)), (("cam", f), ("cam", f + 1)), (("cam", f + 2), ("cam", f)), (("cam", f), ("pt", 0)),
           (("pt", 1), ("cam", f)), (("cam", f), K), (("cam", 3), K), (K, K), (("pt", 5), K), (K, ("pt", 5))]
    ref_got, _ = _run(p, "REF", req, iters=2)
    for r, g in zip(req, ref_got):
        assert g.shape == (DIM[r[0][0]], DIM[r[1][0]])
        assert g.any() == (("cam", f) not in r), r
    dep_got, _ = _run(p, "DEPTH", req, iters=2)
    for r, g in zip(req, dep_got):
        assert g.any() == (("cam", f) not in r and K not in r), r


def test_rejections():
    lib = capi.load()
    s = _solver("REF", solver=4)
    try:
        with pytest.raises(ba_b200.BAError) as e:
            s.covariance_blocks([])
        assert e.value.code == capi.BA_ERR_STATE
        p = _problem("window20")
        s.upload(p)
        assert s.covariance_blocks([]) == []
        for bad in ([(("cam", -1), ("cam", 0))], [(("cam", p.n_cam), ("cam", 0))], [(("pt", p.n_pt), ("cam", 0))],
                    [(("intr", 1), ("cam", 0))], [(("cam", 0), ("pt", -1))]):
            with pytest.raises(ba_b200.BAError) as e:
                s.covariance_blocks(bad)
            assert e.value.code == capi.BA_ERR_INVALID, bad
        a = (capi.CovBlock * 1)()
        a[0].kind, a[0].index = 3, 0  # unknown kind
        assert lib.ba_gpu_covariance_blocks(s._ctx, 1, a, a, capi.dp(np.zeros(36))) == capi.BA_ERR_INVALID
        assert lib.ba_gpu_covariance_blocks(s._ctx, -1, None, None, None) == capi.BA_ERR_INVALID
        assert lib.ba_gpu_covariance_blocks(s._ctx, 1, None, None, None) == capi.BA_ERR_INVALID
    finally:
        s.close()
    for case in ("gauge", "NS", "INTR"):
        p = _problem("cfg1")
        if case == "gauge":
            p.fixed_cam = -1
        s = _solver("REF" if case == "gauge" else case)
        try:
            s.upload(p)
            with pytest.raises(ba_b200.BAError) as e:
                s.covariance_blocks([(("cam", 1), ("cam", 2))])
        finally:
            s.close()
        assert e.value.code == capi.BA_ERR_UNSUPPORTED
        assert {"gauge": "fixed camera", "NS": "depth prior", "INTR": "INTR"}[case] in str(e.value)


SINGULAR = {"two_maps": "camera", "one_obs_cam": "camera", "empty_cam": "camera", "unobserved_pt": "point"}


@pytest.mark.parametrize("name", sorted(SINGULAR))
def test_rank_deficient_rejected(name):
    p = {"two_maps": lambda: ip.two_maps(ip.tum_window(12, 5), ip.tum_window(10, 6)),
         "one_obs_cam": lambda: ip.ragged(ip.tum_window(12, 5), one_obs_cam=7),
         "empty_cam": lambda: ip.ragged(ip.tum_window(12, 5), empty_cam=7),
         "unobserved_pt": lambda: ip.ragged(ip.tum_window(12, 5), unobserved=3)}[name]()
    s = _solver("REF", solver=4)
    try:
        s.upload(p)
        with pytest.raises(ba_b200.BAError) as e:
            s.covariance_blocks([(("cam", 1), ("cam", p.n_cam - 1))])
        piv = s.covariance_pivots()
    finally:
        s.close()
    assert e.value.code == capi.BA_ERR_NUMERIC
    assert SINGULAR[name] in str(e.value)
    if SINGULAR[name] == "camera":
        assert piv["cam"] < capi.BA_COV_MIN_PIVOT_RATIO


def test_solve_blocks_solve_equals_solve_solve():
    p = _problem("tum0.1")
    req = _mixed_requests(p, 9)
    out = []
    for with_cov in (False, True):
        s = _solver("REF", solver=4, max_num_iterations=4)
        try:
            s.upload(p)
            s.solve()
            if with_cov:
                s.covariance_blocks(req)
            summ = s.solve()
            pose, pt, intr = s.download()
            out.append((summ.final_cost, summ.num_iterations, pose.copy(), pt.copy(), intr.copy(), [t["cost"] for t in s.trace()]))
        finally:
            s.close()
    a, b = out
    assert a[0] == b[0] and a[1] == b[1] and a[5] == b[5]
    for x, y in zip(a[2:5], b[2:5]):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("solver", [0, 4])
def test_covariance_after_blocks_is_unaffected(solver):
    p = _problem("window20")
    pr = _pairs(p)
    res = []
    for with_blocks in (False, True):
        s = _solver("REF", solver=solver, max_num_iterations=3)
        try:
            s.upload(p)
            s.solve()
            if with_blocks:
                s.covariance_blocks(_mixed_requests(p, 10))
            res.append(s.covariance(points=True, pairs=pr))
        finally:
            s.close()
    for k in ("cam", "cam_intr", "intr", "pt", "pairs"):
        assert np.array_equal(res[0][k], res[1][k]), k
