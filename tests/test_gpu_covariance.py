"""ba_gpu_covariance / GpuSolver.covariance: the inverse of the undamped Gauss-Newton Hessian per block (ceres::Covariance in the
tangent space, loss applied) by selected inversion over the supernodal Cholesky tree.  The independent reference is numpy,
built from the ORACLE's Jacobians at the state downloaded from the GPU: the dense reduced system with the intrinsics border,
inverted, and the point formula Sigma_pp = V^-1 + V^-1 W_p^T Sigma_RR W_p V^-1 (at cfg1 also the dense inverse of the whole
Hessian)."""
import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

from helpers import ba_b200, mode_opts, ora
from spchol_emulation import covisibility_blocks
from test_gpu_spchol_border import N_KF_BIG, _big_sequence, _problem

pytestmark = pytest.mark.gpu
capi = ba_b200.capi
TOL = 1e-8
# blocks that involve the intrinsics (camera-intrinsics, intrinsics): the intrinsics columns are orders of magnitude larger than the pose
# columns and their covariance is the ill-conditioned direction of the system; measured maxima on a B200: 1.2e-8 (tum0.1, REF) and
# 4.4e-8 (2,800 keyframes) against 3e-10 .. 6e-9 for the camera, pair and point blocks
TOL_INTR = 1e-7


def _solver(mode, **kw):
    g, _ = mode_opts(mode, **kw)
    return ba_b200.GpuSolver(**g)


def _hessian(p, mode, pose, pt, intr):
    """(H sparse over [free cameras | intrinsics | points], n_R, slot of every camera) from the oracle's Jacobians."""
    _, o = mode_opts(mode)
    opts = ora.default_options(**o)
    q = ora.Problem(pose, pt, p.cam_idx, p.pt_idx, p.uv2, p.depth, intr, p.intr_prior, p.fixed_cam)
    ev = ora.evaluate(q, opts)
    assert ev["rc"] == 0
    nk = 4 if o["optimize_intrinsics"] else 0
    slot = np.full(p.n_cam, -1)
    free = [c for c in range(p.n_cam) if c != p.fixed_cam]
    slot[free] = np.arange(len(free))
    nR = 6 * len(free) + nk
    n_obs, R = ev["Jc"].shape[:2]
    rows, cols, vals = [], [], []
    obs_row = np.arange(n_obs)[:, None] * R + np.arange(R)[None, :]
    cam = p.cam_idx.astype(np.int64)
    # camera columns (free cameras only)
    m = slot[cam] >= 0
    for k in range(6):
        rows.append(obs_row[m].reshape(-1)); cols.append(np.repeat(6 * slot[cam[m]] + k, R)); vals.append(ev["Jc"][m][:, :, k].reshape(-1))
    for k in range(3):
        rows.append(obs_row.reshape(-1)); cols.append(np.repeat(nR + 3 * p.pt_idx.astype(np.int64) + k, R)); vals.append(ev["Jp"][:, :, k].reshape(-1))
    if nk:
        for k in range(4):
            rows.append(obs_row[:, :2].reshape(-1)); cols.append(np.full(2 * n_obs, 6 * len(free) + k)); vals.append(ev["Jk"][:, :, k].reshape(-1))
    J = sps.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n_obs * R, nR + 3 * p.n_pt))
    H = (J.T @ J).tocsr()
    if nk:
        H = H + sps.csr_matrix((np.full(4, opts.weight_intrinsics), (np.arange(4) + 6 * len(free), np.arange(4) + 6 * len(free))),
                               shape=H.shape)
    return H.tocsr(), nR, nk, slot


def _reduced(H, nR, n_pt):
    """Sparse reduced system S = H_RR - H_Rp V^-1 H_pR and the point blocks V^-1 [n_pt, 3, 3]."""
    Hrr, Hrp = H[:nR, :nR], H[:nR, nR:]
    V = np.stack([H[nR + 3 * i:nR + 3 * i + 3, nR + 3 * i:nR + 3 * i + 3].toarray() for i in range(n_pt)])
    Vi = np.linalg.inv(V)
    Vib = sps.block_diag(list(Vi), format="csr")
    return (Hrr - Hrp @ Vib @ Hrp.T).tocsc(), Vi, Hrp


def _reference(p, mode, pose, pt, intr):
    H, nR, nk, slot = _hessian(p, mode, pose, pt, intr)
    S, Vi, Hrp = _reduced(H, nR, p.n_pt)
    Sd = S.toarray()
    d = 1.0 / np.sqrt(np.diag(Sd))  # (equilibrated: the intrinsics columns are orders of magnitude larger than the pose columns)
    Srr = d[:, None] * np.linalg.inv(d[:, None] * Sd * d[None, :]) * d[None, :]
    nc = nR - nk
    out = dict(cam=np.zeros((p.n_cam, 6, 6)), cam_intr=np.zeros((p.n_cam, 6, 4)), intr=np.zeros((4, 4)))
    for c in range(p.n_cam):
        if slot[c] >= 0:
            out["cam"][c] = Srr[6 * slot[c]:6 * slot[c] + 6, 6 * slot[c]:6 * slot[c] + 6]
            if nk:
                out["cam_intr"][c] = Srr[6 * slot[c]:6 * slot[c] + 6, nc:]
    if nk:
        out["intr"] = Srr[nc:, nc:]
    K = (Hrp.T @ Srr).T  # Sigma_RR W  [nR, 3 n_pt]
    Hd = Hrp.toarray().reshape(nR, p.n_pt, 3)
    Mp = np.einsum("ipr,ips->prs", Hd, K.reshape(nR, p.n_pt, 3))
    out["pt"] = Vi + Vi @ Mp @ Vi
    out["pair"] = lambda a, b: (np.zeros((6, 6)) if slot[a] < 0 or slot[b] < 0 else
                                Srr[6 * slot[a]:6 * slot[a] + 6, 6 * slot[b]:6 * slot[b] + 6])
    out["H"], out["nR"], out["slot"] = H, nR, slot
    return out


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300))


def _pairs(p):
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    return np.stack([np.concatenate([bi, bj]), np.concatenate([bj, bi])], axis=1).astype(np.int32)


# ---------------------------------------------------------------- 1. against the oracle's Hessian
@pytest.mark.parametrize("mode", ["REF", "DEPTH"])
@pytest.mark.parametrize("name", ["cfg1", "window20", "tum0.1"])
def test_matches_oracle_reference(name, mode):
    p = _problem(name)
    s = _solver(mode, max_num_iterations=4)
    s.upload(p)
    s.solve()
    pose, pt, intr = (x.copy() for x in s.download())
    pr = _pairs(p)
    got = s.covariance(points=True, pairs=pr)
    s.close()
    ref = _reference(p, mode, pose, pt, intr)
    err = dict(cam=_rel(got["cam"], ref["cam"]), pt=_rel(got["pt"], ref["pt"]),
               pairs=_rel(got["pairs"], np.stack([ref["pair"](a, b) for a, b in pr])))
    if mode == "REF":
        err.update(cam_intr=_rel(got["cam_intr"], ref["cam_intr"]), intr=_rel(got["intr"], ref["intr"]))
    else:
        assert not got["cam_intr"].any() and not got["intr"].any()
    if name == "cfg1":  # the dense inverse of the whole Hessian: cameras, intrinsics and every point block
        Hi = np.linalg.inv(ref["H"].toarray())
        nR, slot = ref["nR"], ref["slot"]
        full_pt = np.stack([Hi[nR + 3 * i:nR + 3 * i + 3, nR + 3 * i:nR + 3 * i + 3] for i in range(p.n_pt)])
        full_cam = np.stack([Hi[6 * slot[c]:6 * slot[c] + 6, 6 * slot[c]:6 * slot[c] + 6] if slot[c] >= 0 else np.zeros((6, 6))
                             for c in range(p.n_cam)])
        err.update(full_pt=_rel(got["pt"], full_pt), full_cam=_rel(got["cam"], full_cam))
    print("covariance max relative error %s %s: %s" % (name, mode, " ".join("%s=%.2e" % kv for kv in sorted(err.items()))))
    for k, v in err.items():
        assert v <= (TOL_INTR if k in ("cam_intr", "intr") else TOL), (k, v)


# ---------------------------------------------------------------- 2. same bits under AUTO and solver = 4
@pytest.mark.parametrize("name", ["window20", "tum0.1"])
def test_auto_and_sparse_cholesky_bit_identical(name):
    p = _problem(name)
    pr = _pairs(p)
    res = []
    for solver in (0, 4):
        s = _solver("REF", solver=solver)
        s.upload(p)
        res.append((s.covariance(points=True, pairs=pr), s.spchol_info()))
        s.close()
    (a, ia), (b, ib) = res
    assert ia == {} and ib["nodes"] >= 1  # AUTO: the dense explicit solver is in force
    for k in ("cam", "cam_intr", "intr", "pt", "pairs"):
        assert np.array_equal(a[k], b[k]), k


# ---------------------------------------------------------------- 3. fixed camera, rejections
@pytest.mark.parametrize("fixed", [0, 5, "last"])
def test_fixed_camera_blocks_are_zero(fixed):
    p = _problem("window20")
    p.fixed_cam = p.n_cam - 1 if fixed == "last" else fixed
    s = _solver("REF", max_num_iterations=3)
    s.upload(p)
    s.solve()
    pose, pt, intr = (x.copy() for x in s.download())
    f = p.fixed_cam
    pr = np.array([[f, f], [f, (f + 1) % p.n_cam], [(f + 1) % p.n_cam, f]], dtype=np.int32)
    got = s.covariance(points=False, pairs=pr)
    s.close()
    assert got["pt"] is None
    assert not got["cam"][f].any() and not got["cam_intr"][f].any() and not got["pairs"].any()
    ref = _reference(p, "REF", pose, pt, intr)
    assert _rel(got["cam"], ref["cam"]) <= TOL and _rel(got["cam_intr"], ref["cam_intr"]) <= TOL_INTR


@pytest.mark.parametrize("case", ["gauge", "NS", "INTR"])
def test_rejected_when_the_hessian_is_singular(case):
    p = _problem("cfg1")
    mode = "REF" if case == "gauge" else case
    if case == "gauge":
        p.fixed_cam = -1
    s = _solver(mode)
    s.upload(p)
    with pytest.raises(ba_b200.BAError) as e:
        s.covariance()
    s.close()
    assert e.value.code == capi.BA_ERR_UNSUPPORTED
    why = {"gauge": "fixed camera", "NS": "depth prior", "INTR": "INTR"}[case]
    assert why in str(e.value)


def test_state_and_invalid_pairs():
    s = _solver("REF", solver=4)
    with pytest.raises(ba_b200.BAError) as e:
        s.covariance()
    assert e.value.code == capi.BA_ERR_STATE
    p = _problem("tum0.1")
    s.upload(p)
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    blocks = set(zip(bi.tolist(), bj.tolist()))
    far = next((a, b) for a in range(1, p.n_cam) for b in range(a + 1, p.n_cam) if (a, b) not in blocks)
    for bad, code in (([far], capi.BA_ERR_INVALID), ([[0, p.n_cam]], capi.BA_ERR_INVALID)):
        with pytest.raises(ba_b200.BAError) as e:
            s.covariance(points=False, pairs=np.array(bad, dtype=np.int32))
        assert e.value.code == code
    s.close()


# ---------------------------------------------------------------- 4. determinism, symmetry, definiteness
def test_repeated_calls_bit_identical_symmetric_positive_definite():
    p = _problem("tum0.1")
    s = _solver("REF", solver=4, max_num_iterations=3)
    s.upload(p)
    s.solve()
    pr = _pairs(p)
    a = s.covariance(points=True, pairs=pr)
    b = s.covariance(points=True, pairs=pr)
    s.close()
    for k in ("cam", "cam_intr", "intr", "pt", "pairs"):
        assert np.array_equal(a[k], b[k]), k
    free = [c for c in range(p.n_cam) if c != p.fixed_cam]
    cam = a["cam"][free]
    assert np.array_equal(cam, cam.transpose(0, 2, 1)) and np.array_equal(a["pt"], a["pt"].transpose(0, 2, 1))
    assert np.linalg.eigvalsh(cam).min() > 0.0 and np.linalg.eigvalsh(a["pt"]).min() > 0.0
    assert np.linalg.eigvalsh(a["intr"]).min() > 0.0


# ---------------------------------------------------------------- 5. a later solve is unaffected
@pytest.mark.parametrize("name,solver", [("window20", 0), ("tum0.1", 4)])
def test_solve_covariance_solve_equals_solve_solve(name, solver):
    p = _problem(name)
    out = []
    for with_cov in (False, True):
        s = _solver("REF", solver=solver, max_num_iterations=4)
        s.upload(p)
        s.solve()
        if with_cov:
            s.covariance(points=True, pairs=_pairs(p))
        summ = s.solve()
        pose, pt, intr = s.download()
        out.append((summ.final_cost, summ.num_iterations, pose.copy(), pt.copy(), intr.copy(), [t["cost"] for t in s.trace()]))
        s.close()
    a, b = out
    assert a[0] == b[0] and a[1] == b[1] and a[5] == b[5]
    for x, y in zip(a[2:5], b[2:5]):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------- 6. beyond the dense explicit limit
def test_big_sequence_columns_against_sparse_lu():
    seq = _big_sequence()
    p = ba_b200.synthetic.window_problem(seq, 0, N_KF_BIG - 1).problem
    s = _solver("REF")  # AUTO: the sparse Cholesky with the border is in force
    s.upload(p)
    cams = [1, 2, N_KF_BIG // 2, N_KF_BIG - 1]
    bi, bj = covisibility_blocks(p.cam_idx, p.pt_idx, p.n_cam, p.fixed_cam)
    pr = np.array([(a, b) for a, b in zip(bi, bj) if a in cams or b in cams], dtype=np.int32)
    got = s.covariance(points=False, pairs=pr)
    pose, pt, intr = (x.copy() for x in s.download())
    s.close()
    H, nR, nk, slot = _hessian(p, "REF", pose, pt, intr)
    S, _, _ = _reduced(H, nR, p.n_pt)
    lu = spla.splu(S)
    cols = {}
    for c in cams:
        E = np.zeros((nR, 6))
        E[6 * slot[c] + np.arange(6), np.arange(6)] = 1.0
        cols[c] = lu.solve(E)  # Sigma[:, c]
    ref_cam = np.stack([cols[c][6 * slot[c]:6 * slot[c] + 6] for c in cams])
    ref_ci = np.stack([cols[c][nR - 4:].T for c in cams])
    ref_pairs = np.stack([cols[b][6 * slot[a]:6 * slot[a] + 6] if b in cols else cols[a][6 * slot[b]:6 * slot[b] + 6].T
                          for a, b in pr])
    err = dict(cam=_rel(got["cam"][cams], ref_cam), cam_intr=_rel(got["cam_intr"][cams], ref_ci), pairs=_rel(got["pairs"], ref_pairs))
    print("covariance max relative error big%d REF: %s" % (N_KF_BIG, " ".join("%s=%.2e" % kv for kv in sorted(err.items()))))
    for k, v in err.items():
        assert v <= (TOL_INTR if k in ("cam_intr", "intr") else TOL), (k, v)
