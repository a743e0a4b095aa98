"""ctypes binding of the C-ABI in include/ba_gpu.h (libba_gpu.so, built in-tree).

The library is the product; this file is plumbing.  There is no CPU fallback:
`load()` raises if the shared object is missing, and `ba_gpu_create` fails
without a CUDA device.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libba_gpu.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "ba_gpu.h")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)

BA_OK, BA_ERR_INVALID, BA_ERR_CUDA, BA_ERR_STATE, BA_ERR_UNSUPPORTED, BA_ERR_NUMERIC, BA_ERR_COMM = 0, -1, -2, -3, -4, -5, -6
BA_SOLVER_AUTO, BA_SOLVER_EXPLICIT_CHOLESKY, BA_SOLVER_IMPLICIT_PCG, BA_SOLVER_SPARSE_SCHUR_PCG = 0, 1, 2, 3
BA_SOLVER_SPARSE_SCHUR_CHOLESKY = 4
BA_COV_MIN_PIVOT_RATIO = 1e-9  # ba_gpu_covariance's relative pivot test (include/ba_gpu.h)
BA_COV_CAMERA, BA_COV_POINT, BA_COV_INTRINSICS = 0, 1, 2  # ba_cov_block kinds
BA_JAC_AUTO, BA_JAC_PLANES, BA_JAC_FACTORED, BA_JAC_TILED = 0, 1, 2, 3
BA_KERNEL_LINEARIZE, BA_KERNEL_SCHUR_MATVEC, BA_KERNEL_SCHUR_PASS1, BA_KERNEL_SCHUR_PASS2 = 0, 1, 2, 3
TERMINATION = {0: "NO_CONVERGENCE", 1: "GRADIENT", 2: "PARAMETER", 3: "FUNCTION", 4: "MIN_RADIUS", 5: "FAILURE"}


class Options(C.Structure):
    """== ba_gpu_options; first block keeps the names of ceresGlobalProblem
    (headers/BundleAdjustmentConfig.h:47-50, 64-65)."""
    _fields_ = [
        ("HUB_P_REPR", C.c_double), ("WEIGHT_INTRINSICS", C.c_double), ("WEIGHT_UNPR", C.c_double),
        ("HUB_P_UNPR", C.c_double), ("max_num_iterations", C.c_int32), ("eta", C.c_double),
        ("use_depth_prior", C.c_int32), ("optimize_intrinsics", C.c_int32), ("solver", C.c_int32),
        ("explicit_max_dim", C.c_int32), ("n_obs_total", C.c_int64),
        ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double), ("parameter_tolerance", C.c_double),
        ("initial_trust_region_radius", C.c_double), ("max_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double), ("min_relative_decrease", C.c_double),
        ("min_lm_diagonal", C.c_double), ("max_lm_diagonal", C.c_double),
        ("max_num_consecutive_invalid_steps", C.c_int32), ("jacobi_scaling", C.c_int32),
        ("max_linear_solver_iterations", C.c_int32), ("min_linear_solver_iterations", C.c_int32),
        ("residual_reset_period", C.c_int32), ("device", C.c_int32), ("poll_interval", C.c_int32),
        ("persistent_pcg", C.c_int32), ("jacobian_store", C.c_int32),
        ("sparse_max_pairs_per_obs", C.c_int32),
    ]


class CovBlock(C.Structure):
    """== ba_cov_block: (kind, index) of a parameter block for ba_gpu_covariance_blocks."""
    _fields_ = [("kind", C.c_int32), ("index", C.c_int32)]


class IterRecord(C.Structure):
    _fields_ = [
        ("iteration", C.c_int32), ("step_is_valid", C.c_int32), ("step_is_successful", C.c_int32),
        ("linear_iters", C.c_int32), ("cost", C.c_double), ("cost_change", C.c_double),
        ("gradient_max_norm", C.c_double), ("step_norm", C.c_double), ("relative_decrease", C.c_double),
        ("radius", C.c_double), ("model_cost_change", C.c_double),
    ]


class Summary(C.Structure):
    _fields_ = [
        ("termination", C.c_int32), ("num_iterations", C.c_int32), ("num_successful", C.c_int32),
        ("num_unsuccessful", C.c_int32), ("initial_cost", C.c_double), ("final_cost", C.c_double),
        ("total_linear_iters", C.c_int64), ("solver_used", C.c_int32), ("reduced_dim", C.c_int32),
        ("solve_ms", C.c_double), ("kernel_launches", C.c_int64),
    ]


EXPORTS = [
    "ba_gpu_default_options", "ba_gpu_create", "ba_gpu_destroy", "ba_gpu_last_error", "ba_gpu_set_options",
    "ba_gpu_upload", "ba_gpu_solve", "ba_gpu_get_trace", "ba_gpu_download", "ba_gpu_eval", "ba_gpu_get_indices",
    "ba_gpu_schur_matvec", "ba_gpu_se3_plus", "ba_gpu_time_kernel", "ba_gpu_launch_count", "ba_gpu_comm_unique_id",
    "ba_gpu_comm_init", "ba_gpu_jacobian_store_used", "ba_gpu_sparse_stats", "ba_gpu_backproject",
    "ba_gpu_schur_solve", "ba_gpu_spchol_info", "ba_gpu_covariance", "ba_gpu_covariance_blocks",
    "ba_gpu_covariance_pivots", "ba_gpu_phase_times", "ba_gpu_phase_name",
    "ba_store_create", "ba_store_destroy", "ba_store_clear", "ba_store_set_keyframe", "ba_store_set_keyframes", "ba_store_set_poses", "ba_store_set_landmarks",
    "ba_store_window_solve",
    "ba_sparse_symbolic_create", "ba_sparse_symbolic_info", "ba_sparse_symbolic_get", "ba_sparse_symbolic_destroy",
    "ba_sparse_symbolic_partition", "ba_sparse_symbolic_queue",
]

_LIB = None


def load():
    """Loads libba_gpu.so; raises (never falls back) if it is not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libba_gpu.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C 3dsmc-bundle-adjustment_b200/csrc`); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.ba_gpu_default_options.argtypes = [C.POINTER(Options)]
    L.ba_gpu_default_options.restype = None
    L.ba_gpu_create.argtypes = [C.POINTER(Options), C.POINTER(vp)]
    L.ba_gpu_destroy.argtypes = [vp]
    L.ba_gpu_destroy.restype = None
    L.ba_gpu_last_error.argtypes = [vp]
    L.ba_gpu_last_error.restype = C.c_char_p
    L.ba_gpu_set_options.argtypes = [vp, C.POINTER(Options)]
    L.ba_gpu_upload.argtypes = [vp, C.c_int32, c_double_p, C.c_int32, C.c_int32, c_double_p, C.c_int32, c_int32_p,
                                c_int32_p, c_double_p, c_double_p, c_double_p, c_double_p]
    L.ba_gpu_solve.argtypes = [vp, C.POINTER(Summary)]
    L.ba_gpu_get_trace.argtypes = [vp, C.POINTER(IterRecord), C.c_int32]
    L.ba_gpu_download.argtypes = [vp, c_double_p, c_double_p, c_double_p]
    L.ba_gpu_eval.argtypes = [vp] + [c_double_p] * 8
    L.ba_gpu_get_indices.argtypes = [vp, c_int32_p, c_int32_p, c_int32_p]
    L.ba_gpu_schur_matvec.argtypes = [vp, C.c_double, c_double_p, c_double_p]
    L.ba_gpu_se3_plus.argtypes = [vp, C.c_int32, c_double_p, c_double_p, c_double_p]
    L.ba_gpu_time_kernel.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float)]
    L.ba_gpu_launch_count.argtypes = [vp]
    L.ba_gpu_launch_count.restype = C.c_int64
    L.ba_gpu_backproject.argtypes = [vp, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, C.c_int32, c_double_p,
                                     c_double_p, c_double_p, c_double_p]
    L.ba_gpu_jacobian_store_used.argtypes = [vp]
    L.ba_gpu_sparse_stats.argtypes = [vp, C.POINTER(C.c_int64), c_int32_p, c_int32_p]
    L.ba_gpu_comm_unique_id.argtypes = [C.c_char_p]
    L.ba_gpu_comm_init.argtypes = [vp, C.c_char_p, C.c_int32, C.c_int32]
    L.ba_gpu_phase_times.argtypes = [vp, c_double_p]
    L.ba_gpu_phase_name.argtypes = [C.c_int32]
    L.ba_gpu_phase_name.restype = C.c_char_p
    L.ba_gpu_schur_solve.argtypes = [vp, C.c_double, c_double_p, c_double_p]
    L.ba_gpu_spchol_info.argtypes = [vp, C.POINTER(C.c_int64)]
    L.ba_gpu_covariance.argtypes = [vp, c_double_p, c_double_p, c_double_p, c_double_p, C.c_int32, c_int32_p, c_int32_p,
                                    c_double_p]
    L.ba_gpu_covariance_blocks.argtypes = [vp, C.c_int32, C.POINTER(CovBlock), C.POINTER(CovBlock), c_double_p]
    L.ba_gpu_covariance_pivots.argtypes = [vp, c_double_p]
    L.ba_store_create.argtypes = [vp, C.POINTER(vp)]
    L.ba_store_destroy.argtypes = [vp]
    L.ba_store_destroy.restype = None
    L.ba_store_clear.argtypes = [vp]
    L.ba_store_set_keyframe.argtypes = [vp, C.c_int32, C.c_int32, c_int32_p, C.POINTER(C.c_float), c_double_p]
    L.ba_store_set_keyframes.argtypes = [vp, C.c_int32, c_int32_p, c_int32_p, c_int32_p, C.POINTER(C.c_float), c_double_p]
    L.ba_store_set_poses.argtypes = [vp, C.c_int32, C.c_int32, c_double_p]
    L.ba_store_set_landmarks.argtypes = [vp, C.c_int32, c_int32_p, c_double_p]
    L.ba_store_window_solve.argtypes = [vp, C.c_int32, C.c_int32, c_double_p, c_double_p, C.POINTER(Summary), c_double_p, C.c_int32,
                                        c_int32_p, c_int32_p, c_double_p, c_int32_p, c_double_p]
    L.ba_sparse_symbolic_create.argtypes = [C.c_int32, C.c_int32, c_int32_p, c_int32_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.ba_sparse_symbolic_info.argtypes = [vp, C.POINTER(C.c_int64)]
    L.ba_sparse_symbolic_get.argtypes = [vp, C.c_int32, c_int32_p]
    L.ba_sparse_symbolic_destroy.argtypes = [vp]
    L.ba_sparse_symbolic_partition.argtypes = [vp, C.c_int32, c_int32_p, c_double_p]
    L.ba_sparse_symbolic_queue.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_int32_p] + [c_int32_p] * 5
    L.ba_sparse_symbolic_destroy.restype = None
    for name in EXPORTS:
        if name not in ("ba_gpu_destroy", "ba_gpu_default_options", "ba_gpu_last_error", "ba_gpu_launch_count",
                        "ba_sparse_symbolic_destroy", "ba_gpu_phase_name", "ba_store_destroy"):
            getattr(L, name).restype = C.c_int
    _LIB = L
    return L


def dp(a):
    return a.ctypes.data_as(c_double_p) if a is not None else None


def ip(a):
    return a.ctypes.data_as(c_int32_p) if a is not None else None


def f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(shape) if shape is not None else a


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)
