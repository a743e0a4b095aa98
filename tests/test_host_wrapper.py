"""The compiled C++ drop-in (host/OptimizationUtils_gpu.cpp): windowOptimize /
countConstraints with the reference's signatures (headers/OptimizationUtils.h:42,
55), driven through the flat harness libba_host.so."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import ROOT, ba_b200, ora, pose_err

HOST_LIB = os.path.join(os.path.dirname(ba_b200.capi.LIB_PATH), "libba_host.so")
syn = ba_b200.synthetic
se3 = ba_b200.se3


def _lib():
    ba_b200.capi.load()  # libba_gpu.so first (dependency)
    L = C.CDLL(HOST_LIB)
    L.ba_host_count_constraints.restype = C.c_int
    L.ba_host_window_optimize.restype = C.c_int
    return L


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def test_host_library_exports_and_count():
    L = _lib()
    assert hasattr(L, "ba_host_window_optimize") and hasattr(L, "ba_host_count_constraints")
    assert hasattr(ba_b200.hostlib.load(), "ba_host_sliding_sequence")
    # a schedule that cannot run is refused before any GPU call (window larger than the sequence)
    with pytest.raises(RuntimeError):
        ba_b200.hostlib.sliding_sequence(syn.make_tum_sequence(4, 40, 160, seed=1), window_size=8)
    seq = syn.make_tum_sequence(12, 200, 1200, seed=4)
    seq.depth[::7] = 0.0          # inadmissible observations (depth <= 1e-15 are skipped, :265)
    seq.depth[3::11] = -1.0
    kf_ptr = seq.kf_ptr.astype(np.int32)
    n = L.ba_host_count_constraints(12, _ptr(kf_ptr, C.c_int32), _ptr(seq.depth, C.c_double), 2, 9)
    assert n == ba_b200.count_constraints(seq, 2, 9)
    a, b = kf_ptr[2], kf_ptr[10]
    assert n == int(np.count_nonzero(seq.depth[a:b] > 1e-15))


@pytest.mark.gpu
@pytest.mark.parametrize("n_kf,kf_i,kf_f,iters", [(30, 8, 27, 10), (60, 0, 59, 6)], ids=["window", "global-blocked-cholesky"])
def test_window_optimize_cpp_dropin(n_kf, kf_i, kf_f, iters):
    """windowOptimize through the compiled C++ drop-in: a sliding window, and the reference's global optimisation
    over all keyframes (src/main.cpp:179-182; reduced dimension 358 -> blocked Cholesky)."""
    L = _lib()
    seq = syn.make_tum_sequence(n_kf, 100 * n_kf, 600 * n_kf, seed=13)
    seq.depth[5::97] = 0.0  # a few inadmissible observations
    pose = seq.pose.copy()
    lm_pt = seq.pt.copy()
    lm_id = np.arange(seq.pt.shape[0], dtype=np.int32)
    kf_ptr = seq.kf_ptr.astype(np.int32)
    uv = seq.uv.astype(np.float32)
    n_max = int(kf_ptr[kf_f + 1] - kf_ptr[kf_i])
    out_n = C.c_int32(0)
    out_count = C.c_int32(0)
    out_cam = np.zeros(n_max, dtype=np.int32); out_lm = np.zeros(n_max, dtype=np.int32)
    ref_cam = np.zeros(n_max, dtype=np.int32); ref_lm = np.zeros(n_max, dtype=np.int32)
    intr0 = seq.K.copy(); intr = seq.K.copy(); costs = np.zeros(2)
    rc = L.ba_host_window_optimize(n_kf, _ptr(pose, C.c_double), _ptr(kf_ptr, C.c_int32), _ptr(seq.lm, C.c_int32),
                                   _ptr(uv, C.c_float), _ptr(seq.depth, C.c_double), lm_id.shape[0], _ptr(lm_id, C.c_int32),
                                   _ptr(lm_pt, C.c_double), kf_i, kf_f, iters, _ptr(intr0, C.c_double), _ptr(intr, C.c_double),
                                   C.byref(out_n), _ptr(out_cam, C.c_int32), _ptr(out_lm, C.c_int32), _ptr(ref_cam, C.c_int32),
                                   _ptr(ref_lm, C.c_int32), C.byref(out_count), _ptr(costs, C.c_double))
    assert rc == 0
    n = out_n.value
    assert n == out_count.value == ba_b200.count_constraints(seq, kf_i, kf_f)
    # bit-exact enumeration: what went to the GPU == an independent walk of the same containers
    assert np.array_equal(out_cam[:n], ref_cam[:n]) and np.array_equal(out_lm[:n], ref_lm[:n])
    assert np.all(np.diff(out_cam[:n]) >= 0)
    # oracle on the problem in exactly that order
    key = {(int(k), int(l)): i for i, (k, l) in enumerate(zip(seq.kf, seq.lm))}
    rows = np.array([key[(kf_i + int(c), int(l))] for c, l in zip(out_cam[:n], out_lm[:n])])
    uniq, first = np.unique(out_lm[:n], return_index=True)
    lm_order = uniq[np.argsort(first, kind="stable")]
    new_of = {int(l): i for i, l in enumerate(lm_order)}
    T0 = seq.pose[kf_i]
    T0inv = se3.inverse(T0)
    p = ba_b200.BAProblem(se3.mul(np.broadcast_to(T0inv, (kf_f - kf_i + 1, 7)), seq.pose[kf_i:kf_f + 1]),
                          se3.act(T0inv, seq.pt[lm_order]), out_cam[:n], [new_of[int(l)] for l in out_lm[:n]],
                          seq.uv[rows], seq.depth[rows], seq.K, seq.K, 0)
    op = ora.Problem(p.pose7, p.pt3, p.cam_idx, p.pt_idx, p.uv2, p.depth, p.intr, p.intr_prior, 0)
    rc, osum, _ = ora.solve(op, ora.default_options(max_num_iterations=iters))
    assert rc == 0
    assert abs(costs[0] - osum.initial_cost) <= 1e-12 * osum.initial_cost
    assert abs(costs[1] - osum.final_cost) <= (1e-8 if n_kf <= 30 else 1e-7) * osum.final_cost
    want_pose = se3.mul(np.broadcast_to(T0, op.pose7.shape), op.pose7)
    dt, dr = pose_err(pose[kf_i:kf_f + 1], want_pose)
    assert dt < 1e-6 and dr < 1e-6
    assert np.max(np.abs(lm_pt[lm_order] - se3.act(T0, op.pt3))) < 1e-5
    assert np.max(np.abs(intr - op.intr)) < 1e-5
    # untouched outside the window / for landmarks not observed in it
    assert np.array_equal(pose[:kf_i], seq.pose[:kf_i]) and np.array_equal(pose[kf_f + 1:], seq.pose[kf_f + 1:])
    others = np.setdiff1d(lm_id, lm_order)
    assert np.array_equal(lm_pt[others], seq.pt[others])


@pytest.mark.gpu
def test_sliding_sequence_cpp_dropin_matches_python_mirror():
    """The reference's schedule (src/main.cpp:161-175: a window over the last 20 keyframes every 10 keyframes, plus
    the leftover window) through the compiled windowOptimize == the same schedule through the Python mirror.  The two
    enumerate the observations in different orders (std::unordered_map iteration vs array order), so the sums differ
    in the last bits: poses agree to 1e-6 m / 1e-6 rad after 6 warm-started windows."""
    n_kf, W, F, iters = 65, 20, 10, 8
    a = syn.make_tum_sequence(n_kf, 100 * n_kf, 600 * n_kf, seed=21)
    b = syn.make_tum_sequence(n_kf, 100 * n_kf, 600 * n_kf, seed=21)
    ia = a.K.copy()
    res = ba_b200.hostlib.sliding_sequence(a, W, F, max_num_iterations=iters, fixed_iterations=True, intrinsics_optimized=ia)
    assert res["windows"] == 6 and res["lm_iterations"] == 6 * iters   # sizes 20, 30, ..., 60 and the leftover (45..64)
    assert res["ms"]["total"] >= res["ms"]["upload"] + res["ms"]["solve"] + res["ms"]["download"] > 0.0
    gp = ba_b200.CeresGlobalProblem(max_num_iterations=iters, window_size=W, frame_frequency=F)
    sw = ba_b200.GpuSolver(gp.gpu_options(function_tolerance=0.0, parameter_tolerance=0.0, gradient_tolerance=0.0))
    ib = b.K.copy()
    ends = [s for s in range(1, n_kf + 1) if s % F == 0 and s >= W] + ([n_kf] if n_kf % F else [])
    for s_ in ends:
        assert ba_b200.window_optimize(gp, s_ - W, s_ - 1, b, b.K, ib, solver=sw)
    sw.close()
    dt, dr = pose_err(a.pose, b.pose)
    assert dt < 1e-6 and dr < 1e-6
    assert np.max(np.abs(a.pt - b.pt)) < 1e-5
    assert np.max(np.abs(ia - ib)) < 1e-5
    moved = np.max(np.abs(a.pose[:, 4:] - syn.make_tum_sequence(n_kf, 100 * n_kf, 600 * n_kf, seed=21).pose[:, 4:]))
    assert moved > 1e-4   # the windows did change the trajectory


def test_window_optimize_missing_landmark_leaves_inputs_untouched():
    """A keyframe that references a landmark id absent from the map made the reference throw (map.at,
    src/OptimizationUtils.cpp:270); the drop-in returns false BEFORE any GPU call and undoes the in-place frame change
    (:248, :274): poses and landmarks are bit-identical afterwards.  Runs without a GPU."""
    L = _lib()
    seq = syn.make_tum_sequence(12, 240, 1440, seed=9)
    pose = seq.pose.copy()
    kf_ptr = seq.kf_ptr.astype(np.int32)
    uv = seq.uv.astype(np.float32)
    # the map lacks the landmark of an observation in the middle of the window
    victim = int(seq.lm[kf_ptr[5] + 3])
    lm_id = np.array([l for l in range(seq.pt.shape[0]) if l != victim], dtype=np.int32)
    lm_pt = seq.pt[lm_id].copy()
    lm_pt0 = lm_pt.copy()
    intr0 = seq.K.copy(); intr = seq.K.copy()
    rc = L.ba_host_window_optimize(12, _ptr(pose, C.c_double), _ptr(kf_ptr, C.c_int32), _ptr(seq.lm, C.c_int32),
                                   _ptr(uv, C.c_float), _ptr(seq.depth, C.c_double), lm_id.shape[0], _ptr(lm_id, C.c_int32),
                                   _ptr(lm_pt, C.c_double), 2, 9, 5, _ptr(intr0, C.c_double), _ptr(intr, C.c_double),
                                   None, None, None, None, None, None, None)
    assert rc == -1
    assert np.array_equal(pose, seq.pose) and np.array_equal(lm_pt, lm_pt0) and np.array_equal(intr, seq.K)


# ---------------------------------------------------------------- the build INTEGRATION.md prescribes
HOST_DIR = os.path.join(ROOT, "3dsmc-bundle-adjustment_b200", "host")


@pytest.mark.parametrize("src", ["OptimizationUtils_gpu.cpp", "TrajectoryIO.cpp", "ba_host_capi.cpp"])
def test_wrapper_compiles_with_reference_headers_macro(src):
    """-DBA_USE_REFERENCE_HEADERS (include "OptimizationUtils.h" instead of the compat types) against a shim that only
    has the members the reference's vendored Sophus / Eigen really offer (tests/ref_header_shim): no SE3d(const double*)."""
    import subprocess
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Wextra", "-Werror", "-DBA_USE_REFERENCE_HEADERS",
           "-I", os.path.join(ROOT, "tests", "ref_header_shim"), os.path.join(HOST_DIR, src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_reference_arm_program_compiles_against_the_reference_interface():
    """bench/ceres_baseline.cpp (the reference's schedule through windowOptimize, linked either with the reference's own
    OptimizationUtils.cpp + Ceres or with this drop-in) uses only what the reference's headers declare."""
    import subprocess
    src = os.path.join(ROOT, "bench", "ceres_baseline.cpp")
    for extra in (["-DBA_USE_REFERENCE_HEADERS", "-I", os.path.join(ROOT, "tests", "ref_header_shim")], []):
        r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Wextra", "-Werror"] + extra + [src], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]


def test_no_raw_pointer_se3_constructor_anywhere():
    """Sophus::SE3 has no constructor from `const double*` (headers/sophus/se3.hpp:407-455): neither the compat class
    nor the wrapper may rely on one; raw storage goes through data() (se3_raw.h)."""
    import re
    compat = open(os.path.join(HOST_DIR, "compat", "reference_types.h")).read()
    assert re.search(r"SE3d\s*\(\s*const\s+double\s*\*", compat) is None
    for f in ("OptimizationUtils_gpu.cpp", "TrajectoryIO.cpp", "ba_host_capi.cpp"):
        s = open(os.path.join(HOST_DIR, f)).read()
        assert re.search(r"SE3d\s*\(\s*(pose7|p7|initial7)", s) is None, f


# ---------------------------------------------------------------- device-resident store (SURVEY.md 8f row N1)
@pytest.mark.gpu
@pytest.mark.parametrize("growing, window", [(False, 20), (True, 20), (False, 70)],
                         ids=["complete-maps", "maps-grow-between-windows", "complete-maps-window70"])
def test_device_store_sliding_windows_bit_identical(growing, window):
    """The reference's schedule (a 20-keyframe window every 10 keyframes, warm-started) through the compiled drop-in, once
    with every window walked and uploaded in full and once through the device-resident store (only new / grown keyframes
    and new landmarks are uploaded; enumeration and frame changes on the device): poses, landmarks and intrinsics must
    be equal BIT FOR BIT after the whole sequence.  With growing maps the second half of every keyframe's map arrives with
    the next keyframe (the "old_frame" inserts of src/Map3D.cpp:52): such a keyframe is uploaded twice.  70-keyframe
    windows take the blocked dense factorisation."""
    hostlib = ba_b200.hostlib
    out = []
    for store in (False, True):
        seq = syn.make_config(2, scale=0.1)   # 80 keyframes, 8000 landmarks
        intr = seq.K.copy()
        r = hostlib.sliding_sequence(seq, window, 10, max_num_iterations=6, fixed_iterations=True, intrinsics_optimized=intr,
                                     device_store=store, growing_maps=growing)
        out.append((seq.pose.copy(), seq.pt.copy(), intr.copy(), r))
    a, b = out
    assert a[3]["windows"] == b[3]["windows"] == (80 - window) // 10 + 1 and a[3]["lm_iterations"] == b[3]["lm_iterations"]
    assert a[3]["store_windows"] == 0 and b[3]["store_windows"] == b[3]["windows"]   # every window of the second run took the store
    assert np.array_equal(a[0], b[0]), float(np.max(np.abs(a[0] - b[0])))
    assert np.array_equal(a[1], b[1]), float(np.max(np.abs(a[1] - b[1])))
    assert np.array_equal(a[2], b[2])
    assert not np.array_equal(a[0], syn.make_config(2, scale=0.1).pose)   # the windows did move the poses


@pytest.mark.gpu
def test_device_store_c_abi_direct():
    """ba_store_* through ctypes: one window assembled on the device equals upload / solve / download of the host-built
    arrays (synthetic.window_problem does the frame change with numpy: equal to round-off, not bit for bit)."""
    import ctypes as C
    cap = ba_b200.capi
    lib = cap.load()
    seq = syn.make_tum_sequence(30, 3000, 18000, seed=9)
    s = ba_b200.GpuSolver(max_num_iterations=6)
    st = C.c_void_p()
    assert lib.ba_store_create(s._ctx, C.byref(st)) == 0
    try:
        for k in range(30):
            a, b = int(seq.kf_ptr[k]), int(seq.kf_ptr[k + 1])
            ids = np.ascontiguousarray(seq.lm[a:b], dtype=np.int32)
            uvf = np.ascontiguousarray(seq.uv[a:b], dtype=np.float32)
            dep = np.ascontiguousarray(seq.depth[a:b], dtype=np.float64)
            assert lib.ba_store_set_keyframe(st, k, b - a, cap.ip(ids), uvf.ctypes.data_as(C.POINTER(C.c_float)), cap.dp(dep)) == 0
        pose = np.ascontiguousarray(seq.pose, dtype=np.float64)
        assert lib.ba_store_set_poses(st, 0, 30, cap.dp(pose)) == 0
        ids = np.arange(seq.pt.shape[0], dtype=np.int32)
        pts = np.ascontiguousarray(seq.pt, dtype=np.float64)
        assert lib.ba_store_set_landmarks(st, len(ids), cap.ip(ids), cap.dp(pts)) == 0
        intr, prior = seq.K.copy(), seq.K.copy()
        summ = cap.Summary()
        pose_out = np.zeros((20, 7))
        lm_of_pt = np.zeros(20000, dtype=np.int32)
        pt_out = np.zeros((20000, 3))
        n_pt, n_obs = C.c_int32(0), C.c_int32(0)
        ms = np.zeros(3)
        rc = lib.ba_store_window_solve(st, 10, 29, cap.dp(prior), cap.dp(intr), C.byref(summ), cap.dp(pose_out), 20000, C.byref(n_pt),
                                       cap.ip(lm_of_pt), cap.dp(pt_out), C.byref(n_obs), cap.dp(ms))
        assert rc == 0, lib.ba_gpu_last_error(s._ctx)
    finally:
        lib.ba_store_destroy(st)
    win = syn.window_problem(seq, 10, 29)
    assert n_obs.value == win.problem.n_obs and n_pt.value == win.problem.n_pt
    assert np.array_equal(lm_of_pt[:n_pt.value], win.lm_ids)          # first-appearance order, bit-exact
    s2 = ba_b200.GpuSolver(max_num_iterations=6)
    s2.upload(win.problem)
    summ2 = s2.solve()
    pose2, pt2, intr2 = s2.download()
    s2.close()
    s.close()
    assert summ.num_iterations == summ2.num_iterations
    assert abs(summ.final_cost - summ2.final_cost) <= 1e-9 * summ2.final_cost
    world = ba_b200.se3.mul(np.broadcast_to(win.T0, pose2.shape), pose2)
    assert np.max(np.abs(world - pose_out)) < 1e-9
    assert np.max(np.abs(ba_b200.se3.act(win.T0, pt2) - pt_out[:n_pt.value])) < 1e-8
    assert np.max(np.abs(intr - intr2)) < 1e-7
