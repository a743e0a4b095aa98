"""ctypes binding of the COMPILED C++ drop-in (host/OptimizationUtils_gpu.cpp, built as
libba_host.so next to libba_gpu.so): windowOptimize / countConstraints with the reference's
signatures (headers/OptimizationUtils.h:42, 55), reached through the flat harness of
host/ba_host_capi.cpp.  Used by the tests and by bench.py's sliding-sequence measurement; a C++
caller links OptimizationUtils_gpu.cpp directly (INTEGRATION.md).
"""
import ctypes as C
import os

import numpy as np

from . import capi

HOST_LIB_PATH = os.path.join(os.path.dirname(capi.LIB_PATH), "libba_host.so")
_lib = None


def load():
    """dlopen libba_host.so (and its dependency libba_gpu.so); raises if either is missing."""
    global _lib
    if _lib is None:
        capi.load()
        if not os.path.exists(HOST_LIB_PATH):
            raise OSError("libba_host.so is not built: run `make -C 3dsmc-bundle-adjustment_b200/host`")
        L = C.CDLL(HOST_LIB_PATH)
        L.ba_host_count_constraints.restype = C.c_int
        L.ba_host_window_optimize.restype = C.c_int
        L.ba_host_sliding_sequence.restype = C.c_int
        _lib = L
    return _lib


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def sliding_sequence(seq, window_size, frame_frequency=10, max_num_iterations=75, fixed_iterations=False, do_global=False,
                     intrinsics_initial=None, intrinsics_optimized=None, device_store=False, growing_maps=False):
    """The reference's optimisation schedule (src/main.cpp:161-182) over the whole sequence `seq`
    (synthetic.Sequence) through the compiled windowOptimize.  Mutates seq.pose, seq.pt and
    intrinsics_optimized in place (as windowOptimize does with the caller's containers) and returns
    a dict: windows, lm_iterations and the accumulated host wall clock per phase in milliseconds.
    device_store=True routes the calls through the device-resident keyframe / landmark store (ba_host_device_store);
    growing_maps=True inserts the second half of every keyframe's global_points_map when the next keyframe arrives (the
    "old_frame" inserts of src/Map3D.cpp:52), so that keyframes change between two windows."""
    L = load()
    n_kf = int(seq.pose.shape[0])
    kf_ptr = np.ascontiguousarray(seq.kf_ptr, dtype=np.int32)
    lm = np.ascontiguousarray(seq.lm, dtype=np.int32)
    uv = np.ascontiguousarray(seq.uv, dtype=np.float32)
    depth = np.ascontiguousarray(seq.depth, dtype=np.float64)
    pose = np.ascontiguousarray(seq.pose, dtype=np.float64)
    pt = np.ascontiguousarray(seq.pt, dtype=np.float64)
    lm_id = np.arange(pt.shape[0], dtype=np.int32)
    intr0 = np.array(seq.K if intrinsics_initial is None else intrinsics_initial, dtype=np.float64)
    intr = np.array(seq.K if intrinsics_optimized is None else intrinsics_optimized, dtype=np.float64)
    ms = np.zeros(7)
    n_it = C.c_int64(0)
    rc = L.ba_host_sliding_sequence(n_kf, _ptr(pose, C.c_double), _ptr(kf_ptr, C.c_int32), _ptr(lm, C.c_int32), _ptr(uv, C.c_float),
                                    _ptr(depth, C.c_double), int(pt.shape[0]), _ptr(lm_id, C.c_int32), _ptr(pt, C.c_double),
                                    int(window_size), int(frame_frequency), int(bool(do_global)), int(max_num_iterations),
                                    int(bool(fixed_iterations)), _ptr(intr0, C.c_double), _ptr(intr, C.c_double),
                                    _ptr(ms, C.c_double), C.byref(n_it), int(bool(device_store)) | (2 if growing_maps else 0))
    if rc < 0:
        raise RuntimeError("ba_host_sliding_sequence failed (see stderr)")
    seq.pose[...] = pose
    seq.pt[...] = pt
    if intrinsics_optimized is not None:
        intrinsics_optimized[:] = intr
    keys = ("total", "extract", "upload", "solve", "download", "write_back")
    return {"windows": rc, "lm_iterations": int(n_it.value), "ms": dict(zip(keys, ms.tolist())), "intrinsics": intr,
            "store_windows": int(ms[6])}
