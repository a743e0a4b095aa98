"""Host-side handle on the GPU solver: thin, numpy-in / numpy-out, everything
numeric happens behind the C-ABI (ba_gpu_create / upload / solve / download).

`BAProblem` is the flat form of what the reference's windowOptimize assembles
for ceres::Problem (src/OptimizationUtils.cpp:236-299): poses in Sophus storage
order, points in order of first appearance, observations in the canonical
camera-major order.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import capi


class BAError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("ba_gpu error %d: %s" % (code, msg))
        self.code = code


@dataclass
class BAProblem:
    pose7: np.ndarray                 # [n_cam,7] (qx,qy,qz,qw,tx,ty,tz) camera->world
    pt3: np.ndarray                   # [n_pt,3]
    cam_idx: np.ndarray               # [n_obs] int32, non-decreasing
    pt_idx: np.ndarray                # [n_obs] int32
    uv2: np.ndarray                   # [n_obs,2]
    depth: Optional[np.ndarray]       # [n_obs] or None
    intr: np.ndarray                  # fx fy cx cy
    intr_prior: Optional[np.ndarray] = None
    fixed_cam: int = 0
    meta: dict = field(default_factory=dict)

    def __post_init__(self):
        self.pose7 = capi.f64(self.pose7).reshape(-1, 7).copy()
        self.pt3 = capi.f64(self.pt3).reshape(-1, 3).copy()
        self.cam_idx = capi.i32(self.cam_idx).copy()
        self.pt_idx = capi.i32(self.pt_idx).copy()
        self.uv2 = capi.f64(self.uv2).reshape(-1, 2).copy()
        self.depth = None if self.depth is None else capi.f64(self.depth).copy()
        self.intr = capi.f64(self.intr).copy()
        self.intr_prior = self.intr.copy() if self.intr_prior is None else capi.f64(self.intr_prior).copy()

    n_cam = property(lambda self: self.pose7.shape[0])
    n_pt = property(lambda self: self.pt3.shape[0])
    n_obs = property(lambda self: self.cam_idx.shape[0])

    def copy(self):
        return BAProblem(self.pose7, self.pt3, self.cam_idx, self.pt_idx, self.uv2, self.depth, self.intr,
                         self.intr_prior, self.fixed_cam, dict(self.meta))


def default_options(**kw):
    o = capi.Options()
    capi.load().ba_gpu_default_options(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise AttributeError("unknown ba_gpu option %r" % k)
        setattr(o, k, v)
    return o


class GpuSolver:
    """One context == one CUDA stream on one device; not thread-safe."""

    def __init__(self, options=None, **kw):
        self.lib = capi.load()
        self.options = options if options is not None else default_options(**kw)
        self._ctx = C.c_void_p()
        rc = self.lib.ba_gpu_create(C.byref(self.options), C.byref(self._ctx))
        if rc:
            raise BAError(rc, self.lib.ba_gpu_last_error(None).decode())
        self._shape = None

    def close(self):
        if self._ctx:
            self.lib.ba_gpu_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise BAError(rc, self.lib.ba_gpu_last_error(self._ctx).decode())
        return rc

    def set_options(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.options, k):
                raise AttributeError(k)
            setattr(self.options, k, v)
        self._check(self.lib.ba_gpu_set_options(self._ctx, C.byref(self.options)))

    def upload(self, p: BAProblem):
        self._check(self.lib.ba_gpu_upload(
            self._ctx, p.n_cam, capi.dp(p.pose7), p.fixed_cam, p.n_pt, capi.dp(p.pt3), p.n_obs, capi.ip(p.cam_idx),
            capi.ip(p.pt_idx), capi.dp(p.uv2), capi.dp(p.depth), capi.dp(p.intr), capi.dp(p.intr_prior)))
        self._shape = (p.n_cam, p.n_pt, p.n_obs)

    def solve(self):
        s = capi.Summary()
        self._check(self.lib.ba_gpu_solve(self._ctx, C.byref(s)))
        return s

    def trace(self):
        cap = self.options.max_num_iterations + 2
        buf = (capi.IterRecord * cap)()
        n = self._check(self.lib.ba_gpu_get_trace(self._ctx, buf, cap))
        return [{f[0]: getattr(buf[i], f[0]) for f in capi.IterRecord._fields_} for i in range(n)]

    def download(self, out=None):
        """(pose7 [n_cam,7], pt3 [n_pt,3], intr4).  `out` = a (pose, pt, intr) tuple of preallocated contiguous float64
        arrays to receive the result -- e.g. views of pinned host memory, which the device writes at PCIe speed (a
        pageable destination of the 48 MB of config-5 points takes ~11 ms instead of ~1)."""
        n_cam, n_pt, _ = self._shape
        if out is None:
            out = (np.zeros((n_cam, 7)), np.zeros((n_pt, 3)), np.zeros(4))
        pose, pt, intr = out
        assert pose.shape == (n_cam, 7) and pt.shape == (n_pt, 3) and intr.shape == (4,)
        self._check(self.lib.ba_gpu_download(self._ctx, capi.dp(pose), capi.dp(pt), capi.dp(intr)))
        return pose, pt, intr

    # ---- test / measurement hooks
    def eval(self):
        n_cam, n_pt, n = self._shape
        R = 2 + (1 if self.options.use_depth_prior else 0)
        out = dict(r=np.zeros((n, R)), Jc=np.zeros((n, R, 6)), Jp=np.zeros((n, R, 3)), Jk=np.zeros((n, 2, 4)),
                   g_c=np.zeros((n_cam, 6)), g_p=np.zeros((n_pt, 3)), g_k=np.zeros(4))
        cost = C.c_double(0.0)
        self._check(self.lib.ba_gpu_eval(self._ctx, capi.dp(out["r"]), capi.dp(out["Jc"]), capi.dp(out["Jp"]),
                                         capi.dp(out["Jk"]), C.cast(C.byref(cost), capi.c_double_p), capi.dp(out["g_c"]),
                                         capi.dp(out["g_p"]), capi.dp(out["g_k"])))
        out["cost"] = cost.value
        return out

    def indices(self):
        n_cam, n_pt, n = self._shape
        perm = np.zeros(n, dtype=np.int32)
        pt_rowptr = np.zeros(n_pt + 1, dtype=np.int32)
        cam_rowptr = np.zeros(n_cam + 1, dtype=np.int32)
        self._check(self.lib.ba_gpu_get_indices(self._ctx, capi.ip(perm), capi.ip(pt_rowptr), capi.ip(cam_rowptr)))
        return perm, pt_rowptr, cam_rowptr

    def schur_matvec(self, radius, x):
        x = capi.f64(x).reshape(-1)
        y = np.zeros_like(x)
        self._check(self.lib.ba_gpu_schur_matvec(self._ctx, float(radius), capi.dp(x), capi.dp(y)))
        return y

    def schur_solve(self, radius, rhs):
        """(S + D^2)^-1 rhs through the sparse Cholesky in force (test hook)."""
        rhs = capi.f64(rhs).reshape(-1)
        y = np.zeros_like(rhs)
        self._check(self.lib.ba_gpu_schur_solve(self._ctx, float(radius), capi.dp(rhs), capi.dp(y)))
        return y

    def covariance(self, points=True, pairs=None):
        """Covariance of the estimate at the current state (after solve(), or right after upload()): the inverse of the
        undamped Gauss-Newton Hessian per block in its tangent space, as ceres::Covariance (loss applied).  Needs the depth
        prior and a fixed camera.  pairs: [n, 2] camera indices of co-visible cameras (or a == b).
        -> {"cam": [n_cam,6,6], "cam_intr": [n_cam,6,4], "intr": [4,4], "pt": [n_pt,3,3] (None if not points),
            "pairs": [n,6,6]}"""
        if self._shape is None:  # (before upload: the library reports BA_ERR_STATE)
            self._check(self.lib.ba_gpu_covariance(self._ctx, None, None, None, None, 0, None, None, None))
        n_cam, n_pt, _ = self._shape
        pr = np.zeros((0, 2), dtype=np.int32) if pairs is None else np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        a, b = np.ascontiguousarray(pr[:, 0]), np.ascontiguousarray(pr[:, 1])
        out = dict(cam=np.zeros((n_cam, 6, 6)), cam_intr=np.zeros((n_cam, 6, 4)), intr=np.zeros((4, 4)),
                   pt=np.zeros((n_pt, 3, 3)) if points else None, pairs=np.zeros((len(a), 6, 6)))
        self._check(self.lib.ba_gpu_covariance(self._ctx, capi.dp(out["cam"]), capi.dp(out["cam_intr"]), capi.dp(out["intr"]),
                                               capi.dp(out["pt"]), len(a), capi.ip(a), capi.ip(b), capi.dp(out["pairs"])))
        return out

    def spchol_info(self):
        """Structure of the sparse Cholesky of the last upload ({} when another solver is in force)."""
        info = (C.c_int64 * 24)()
        self._check(self.lib.ba_gpu_spchol_info(self._ctx, info))
        if info[1] == 0:
            return {}
        keys = ["n_cam", "nodes", "levels", "panel_blocks", "update_blocks", "max_front_blocks", "max_own", "max_border",
                "max_children", "flops", "critical_path_block_ops", "symbolic_us", "parts", "distributed", "top_cameras",
                "exchange_bytes", "s_exchange_blocks"]
        return {k: int(info[i]) for i, k in enumerate(keys)}

    def phase_times(self):
        """{phase name: ms} of the last solve (CUDA events recorded while it ran); empty for the windowed solver."""
        ms = np.zeros(11)
        self._check(self.lib.ba_gpu_phase_times(self._ctx, capi.dp(ms)))
        out = {self.lib.ba_gpu_phase_name(k).decode(): float(ms[k]) for k in range(1, 11)}
        return out if sum(out.values()) > 0 else {}

    def se3_plus(self, pose7, delta6):
        pose7 = capi.f64(pose7).reshape(-1, 7)
        delta6 = capi.f64(delta6).reshape(-1, 6)
        out = np.zeros_like(pose7)
        self._check(self.lib.ba_gpu_se3_plus(self._ctx, pose7.shape[0], capi.dp(pose7), capi.dp(delta6), capi.dp(out)))
        return out

    def time_kernel(self, which, warmup=3, iters=20, flush_l2=False):
        ms = C.c_float(0.0)
        self._check(self.lib.ba_gpu_time_kernel(self._ctx, which, warmup, iters, 1 if flush_l2 else 0, C.byref(ms)))
        return ms.value

    def launch_count(self):
        return int(self.lib.ba_gpu_launch_count(self._ctx))

    def backproject(self, uv, depth_img, intr, pose7=None):
        """Batched getLocalPoints3D (src/Map3D.cpp:76-97) [+ world-frame landmark initialisation (:44)
        when pose7 is given]: uv [n,2] float32 pixels, depth_img [H,W] float32 metres.
        Returns local [n,3] (and world [n,3])."""
        import ctypes as C
        uv = np.ascontiguousarray(uv, dtype=np.float32).reshape(-1, 2)
        img = np.ascontiguousarray(depth_img, dtype=np.float32)
        k = capi.f64(intr)
        n = uv.shape[0]
        local = np.empty((n, 3), dtype=np.float64)
        world = np.empty((n, 3), dtype=np.float64) if pose7 is not None else None
        p = capi.f64(pose7) if pose7 is not None else None
        fp = C.POINTER(C.c_float)
        self._check(self.lib.ba_gpu_backproject(self._ctx, n, uv.ctypes.data_as(fp), img.ctypes.data_as(fp), img.shape[1], img.shape[0],
                                                capi.dp(k), capi.dp(p), capi.dp(local), capi.dp(world)))
        return (local, world) if pose7 is not None else local

    def sparse_stats(self):
        """(row entries, stored upper blocks) of the block-sparse Schur complement; zeros for other solvers."""
        import ctypes as C
        npairs, nblk, nent = C.c_int64(0), C.c_int32(0), C.c_int32(0)
        self._check(self.lib.ba_gpu_sparse_stats(self._ctx, C.byref(npairs), C.byref(nblk), C.byref(nent)))
        return int(nent.value), int(nblk.value)

    def sparse_pairs(self):
        """Same-point observation pairs behind the block-sparse Schur complement (0 for other solvers)."""
        import ctypes as C
        npairs, nblk, nent = C.c_int64(0), C.c_int32(0), C.c_int32(0)
        self._check(self.lib.ba_gpu_sparse_stats(self._ctx, C.byref(npairs), C.byref(nblk), C.byref(nent)))
        return int(npairs.value)

    def jacobian_store_used(self):
        """BA_JAC_* in force after the last upload (what BA_JAC_AUTO resolved to)."""
        rc = int(self.lib.ba_gpu_jacobian_store_used(self._ctx))
        if rc < 0:
            self._check(rc)
        return rc

    def comm_init(self, id128: bytes, rank: int, n_ranks: int):
        self._check(self.lib.ba_gpu_comm_init(self._ctx, id128, rank, n_ranks))


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = capi.load().ba_gpu_comm_unique_id(buf)
    if rc:
        raise BAError(rc, capi.load().ba_gpu_last_error(None).decode())
    return buf.raw
