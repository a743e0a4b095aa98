/*
 * ba_gpu.h -- C ABI of the B200-native windowed bundle-adjustment solver.
 *
 * Drop-in boundary for the Ceres Problem/Solve path of
 * martinxluptak/3dsmc-bundle-adjustment (citations relative to the reference):
 *
 *   ba_gpu_create   <- ceres::Problem + Solver::Options construction
 *                      src/OptimizationUtils.cpp:218-226,
 *                      headers/BundleAdjustmentConfig.h:44-67
 *   ba_gpu_upload   <- AddParameterBlock / AddResidualBlock /
 *                      SetParameterBlockConstant
 *                      src/OptimizationUtils.cpp:236-241, 251-254, 275, 279-294, 299
 *   ba_gpu_solve    <- ceres::Solve            src/OptimizationUtils.cpp:300
 *   ba_gpu_download <- Ceres writing the optimum back into the caller-owned
 *                      pose / point / intrinsics blocks
 *                      (pose.data() :251, map_point.point.data() :275,
 *                       intrinsics_optimized.data() :236)
 *
 * Plain pointers and sizes only; no C++/torch types. All doubles are IEEE fp64,
 * all indices int32. Every function returns 0 on success and a negative
 * BA_ERR_* code on failure (never throws, never aborts);
 * ba_gpu_last_error() gives the message.  A context is not thread-safe; use one
 * per host thread.  There is NO CPU fallback: without a CUDA device
 * ba_gpu_create fails with BA_ERR_CUDA.
 */
#ifndef BA_GPU_H
#define BA_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ba_gpu_ctx ba_gpu_ctx;

enum {
  BA_OK = 0,
  BA_ERR_INVALID = -1,  /* bad argument / unsorted or out-of-range indices */
  BA_ERR_CUDA = -2,     /* CUDA runtime error (message has the detail) */
  BA_ERR_STATE = -3,    /* call order (e.g. solve before upload) */
  BA_ERR_UNSUPPORTED = -4, /* option combination not implemented */
  BA_ERR_NUMERIC = -5,  /* non-finite cost at the initial point */
  BA_ERR_COMM = -6      /* NCCL error */
};

enum {
  BA_SOLVER_AUTO = 0,              /* dense explicit if reduced dim <= explicit_max_dim, or with free intrinsics
                                      up to reduced dim 16,384; free intrinsics beyond 16,384 (one GPU): the
                                      sparse Cholesky with the intrinsics border (_SPARSE_SCHUR_CHOLESKY;
                                      BA_ERR_UNSUPPORTED with the reason when its fronts do not fit);
                                      else block-sparse S if the co-visibility is sparse (NS mode), factorised
                                      exactly (_SPARSE_SCHUR_CHOLESKY) when its fronts fit, else with PCG;
                                      else implicit */
  BA_SOLVER_EXPLICIT_CHOLESKY = 1, /* explicit Schur complement + dense Cholesky
                                      (== Ceres DENSE_SCHUR / SPARSE_SCHUR step) */
  BA_SOLVER_IMPLICIT_PCG = 2,      /* matrix-free Schur + block-Jacobi PCG
                                      (== Ceres ITERATIVE_SCHUR + SCHUR_JACOBI) */
  BA_SOLVER_SPARSE_SCHUR_PCG = 3,  /* explicit BLOCK-SPARSE Schur complement (6x6 blocks, symmetric
                                      storage, device-built structure) + the same PCG
                                      (== ITERATIVE_SCHUR with use_explicit_schur_complement;
                                      the matrix Ceres SPARSE_SCHUR factorises). NS mode only. */
  BA_SOLVER_SPARSE_SCHUR_CHOLESKY = 4 /* the same block-sparse S factorised EXACTLY by a supernodal multifrontal
                                      Cholesky over a nested-dissection tree of the camera sequence
                                      (== Ceres SPARSE_SCHUR, the reference's own setting,
                                      headers/BundleAdjustmentConfig.h:62).  Every cost mode: with depth
                                      prior and / or free intrinsics (REF, the reference's cost) S comes from
                                      the planes store and the four intrinsics columns are a dense border,
                                      solved by a 4x4 Schur complement between the forward and the backward
                                      substitution; one GPU, jacobian_store AUTO or PLANES.  BA_ERR_UNSUPPORTED
                                      when a front does not fit shared memory (AUTO on an NS problem then
                                      keeps PCG). */
};

enum {
  BA_JAC_AUTO = 0,     /* NS mode + implicit PCG: tiled if the index locality allows, else factored;
                          planes otherwise */
  BA_JAC_PLANES = 1,   /* materialised r, Jc (2x6), Jp (2x3) planes: 160 B/obs per ordering */
  BA_JAC_FACTORED = 2, /* r + (X/Z, Y/Z, 1/Z, w): 48 B/obs; Jacobian entries rebuilt in registers
                          (NS mode + implicit PCG only); two-pass Schur product */
  BA_JAC_TILED = 3     /* factored store + a tile-local camera-major copy of (X/Z, Y/Z, 1/Z, w): the
                          Schur product is ONE pass, 36 B/obs (needs point tiles that span <= 64
                          cameras and hold <= 2048 observations; BA_ERR_UNSUPPORTED otherwise) */
};

enum {
  BA_TERM_NO_CONVERGENCE = 0, /* max_num_iterations reached */
  BA_TERM_GRADIENT = 1,
  BA_TERM_PARAMETER = 2,
  BA_TERM_FUNCTION = 3,
  BA_TERM_MIN_RADIUS = 4,
  BA_TERM_FAILURE = 5
};

/* Knobs. The first block keeps the reference's names
 * (ceresGlobalProblem, headers/BundleAdjustmentConfig.h:47-50, 64-65). */
typedef struct ba_gpu_options {
  double HUB_P_REPR;        /* Huber delta, reprojection      (:47) */
  double WEIGHT_INTRINSICS; /* intrinsics prior weight         (:48) */
  double WEIGHT_UNPR;       /* depth-prior weight              (:49) */
  double HUB_P_UNPR;        /* Huber delta, depth prior        (:50) */
  int32_t max_num_iterations; /* options.max_num_iterations    (:64) */
  double eta;               /* options.eta (PCG forcing term)  (:65) */
  /* cost model: REF mode = (1,1) is the reference's cost; NS mode = (0,0) is
   * reprojection only with fixed intrinsics (north-star subset) */
  int32_t use_depth_prior;
  int32_t optimize_intrinsics;
  int32_t solver;           /* BA_SOLVER_* */
  int32_t explicit_max_dim; /* AUTO switch point (reduced system dimension) */
  int64_t n_obs_total;      /* weight normaliser 1/N; 0 -> n_obs of the upload
                               (set to the global count when point-sharded) */
  /* Ceres 2.0.0 trust-region defaults (SURVEY.md Appendix A) */
  double function_tolerance, gradient_tolerance, parameter_tolerance;
  double initial_trust_region_radius, max_trust_region_radius, min_trust_region_radius;
  double min_relative_decrease, min_lm_diagonal, max_lm_diagonal;
  int32_t max_num_consecutive_invalid_steps;
  int32_t jacobi_scaling;
  int32_t max_linear_solver_iterations, min_linear_solver_iterations;
  int32_t residual_reset_period;
  /* execution */
  int32_t device;          /* CUDA ordinal; <0 = current device */
  int32_t poll_interval;   /* host polls the device-side LM / PCG termination
                              flag every this many iterations (>=1) */
  int32_t persistent_pcg;  /* block-sparse solver: 0 = one launch per PCG step; 1 = the whole PCG solve of an
                              LM iteration in one persistent cooperative kernel; with several GPUs (peer access,
                              <= 8 ranks) the block-CSR product is ROW-SHARDED over the ranks and exchanged
                              through flag-in-data slots in NVLink peer memory inside the kernel;
                              2 = persistent, replicated on every rank (no exchange inside PCG) */
  int32_t jacobian_store;  /* BA_JAC_AUTO / _PLANES / _FACTORED / _TILED */
  int32_t sparse_max_pairs_per_obs; /* BA_SOLVER_AUTO on a large NS-mode problem (one GPU) picks the
                              block-sparse Schur solver when the number of same-point observation
                              pairs is at most this many per observation, else the implicit one */
} ba_gpu_options;

/* Per-iteration record, written by the device-side LM controller. Mirrors
 * ceres::IterationSummary for the fields the parity tests compare. */
typedef struct ba_gpu_iter {
  int32_t iteration, step_is_valid, step_is_successful, linear_iters;
  double cost, cost_change, gradient_max_norm, step_norm, relative_decrease,
      radius, model_cost_change;
} ba_gpu_iter;

typedef struct ba_gpu_summary {
  int32_t termination, num_iterations, num_successful, num_unsuccessful;
  double initial_cost, final_cost;
  int64_t total_linear_iters;
  int32_t solver_used;       /* the BA_SOLVER_* that ran (what AUTO resolved to) */
  int32_t reduced_dim;
  double solve_ms;           /* CUDA-event time of ba_gpu_solve on its stream */
  int64_t kernel_launches;   /* kernels launched by this solve */
} ba_gpu_summary;

void ba_gpu_default_options(ba_gpu_options *o);

int ba_gpu_create(const ba_gpu_options *o, ba_gpu_ctx **ctx);
void ba_gpu_destroy(ba_gpu_ctx *ctx);
/* ctx may be NULL: message of the last failed ba_gpu_create on this thread */
const char *ba_gpu_last_error(const ba_gpu_ctx *ctx);
/* replaces the options of an existing context (takes effect at next upload) */
int ba_gpu_set_options(ba_gpu_ctx *ctx, const ba_gpu_options *o);

/* Host buffers in, canonical reference order (SURVEY.md 8a): observation k is
 * the k-th admissible (keyframe, landmark) pair of the reference's loop
 * (src/OptimizationUtils.cpp:244, 257) => cam_idx non-decreasing.
 *   pose7 [n_cam*7]  (qx,qy,qz,qw,tx,ty,tz), camera->world, Sophus storage
 *                    order (headers/sophus/se3.hpp:356-365)
 *   fixed_cam        index of the constant pose (:299), or -1
 *   pt3   [n_pt*3]   world points; pt_idx = order of first appearance (:271-276)
 *   uv2   [n_obs*2]  pixels; depth [n_obs] metres or NULL (required iff
 *                    use_depth_prior)
 *   intr4 (fx,fy,cx,cy) initial value; intr_prior4 = intrinsics_initial (:238) */
int ba_gpu_upload(ba_gpu_ctx *ctx, int32_t n_cam, const double *pose7,
                  int32_t fixed_cam, int32_t n_pt, const double *pt3,
                  int32_t n_obs, const int32_t *cam_idx, const int32_t *pt_idx,
                  const double *uv2, const double *depth, const double intr4[4],
                  const double intr_prior4[4]);

int ba_gpu_solve(ba_gpu_ctx *ctx, ba_gpu_summary *summary);
/* copies up to cap trace records of the last solve; returns the count */
int ba_gpu_get_trace(ba_gpu_ctx *ctx, ba_gpu_iter *out, int32_t cap);

int ba_gpu_download(ba_gpu_ctx *ctx, double *pose7, double *pt3, double intr4[4]);

/* ---- test hooks (parity tests call these through ctypes) ---- */
/* Linearisation at the current device state, transposed back to the canonical
 * row-major per-observation layout of the oracle: R = 2 + use_depth_prior.
 *   r [n_obs*R], Jc [n_obs*R*6], Jp [n_obs*R*3], Jk [n_obs*2*4],
 *   g_c [n_cam*6], g_p [n_pt*3], g_k [4]; any pointer may be NULL. */
int ba_gpu_eval(ba_gpu_ctx *ctx, double *r, double *Jc, double *Jp, double *Jk,
                double *cost, double *g_c, double *g_p, double *g_k);
/* Device-built index arrays: stable point-major permutation and CSR pointers */
int ba_gpu_get_indices(ba_gpu_ctx *ctx, int32_t *perm_pt_major,
                       int32_t *pt_rowptr, int32_t *cam_rowptr);
/* y = S x (reduced camera system at the current state, given radius), unscaled
 * coordinates, x,y [n_cam*6] host buffers. Runs the implicit-Schur kernels. */
int ba_gpu_schur_matvec(ba_gpu_ctx *ctx, double radius, const double *x, double *y);
/* y = (S + D^2)^-1 rhs through the sparse Cholesky of the last upload (BA_SOLVER_SPARSE_SCHUR_CHOLESKY in force, NS mode:
 * BA_ERR_UNSUPPORTED with depth prior or free intrinsics, as for ba_gpu_schur_matvec then), same conventions as
 * ba_gpu_schur_matvec: ba_gpu_schur_matvec(radius, ba_gpu_schur_solve(radius, b)) == b */
int ba_gpu_schur_solve(ba_gpu_ctx *ctx, double radius, const double *rhs, double *y);
/* Covariance of the estimate at the current device state (after ba_gpu_solve, or right after ba_gpu_upload):
 * the inverse of the undamped Gauss-Newton Hessian of the cost in force, per block in its tangent space
 * (== ceres::Covariance, GetCovarianceBlockInTangentSpace, loss applied).  Constant blocks have zero covariance.
 *   cov_cam      [n_cam*36]  6x6 row-major per camera, columns ordered as Jc of ba_gpu_eval   (nullable)
 *   cov_cam_intr [n_cam*24]  6x4 camera-intrinsics cross-covariance                            (nullable)
 *   cov_intr     [16]        4x4                                                                (nullable)
 *   cov_pt       [n_pt*9]    3x3 per point                                                      (nullable)
 *   n_pairs, cam_a, cam_b -> cov_pairs [n_pairs*36]: Cov(delta_a, delta_b) for cameras that share a point (or a == b)
 * Selected inversion over the supernodal tree of BA_SOLVER_SPARSE_SCHUR_CHOLESKY, whichever solver the upload resolved to
 * (the first call after an upload builds that tree when another solver is in force).  A later ba_gpu_solve is unaffected.
 * BA_ERR_UNSUPPORTED: no depth prior (scale free), fixed_cam < 0 (gauge free), more than one rank, or a front that does not
 * fit; BA_ERR_INVALID: a pair that is not co-visible, an index out of range.
 * BA_ERR_NUMERIC: the Hessian is singular or numerically rank-deficient: a point's 3x3 block is singular (a point without
 * observations), or a scalar pivot of the Jacobi-scaled camera system, or of the 4x4 intrinsics system T = C - Z^T Z, is below
 * BA_COV_MIN_PIVOT_RATIO times its column's diagonal before elimination (a camera with too few observations to fix its pose,
 * cameras not connected to the fixed one).  In an exactly rank-deficient Hessian such a pivot is rounding, of either sign, and
 * the inverse would be of order 1e16: the relative test rejects it whatever the rounding.  This is the analogue of Ceres'
 * Covariance::Options::min_reciprocal_condition_number.  The LM step (ba_gpu_solve) does not apply it: there the damping
 * makes the system definite. */
#define BA_COV_MIN_PIVOT_RATIO 1e-9
int ba_gpu_covariance(ba_gpu_ctx *ctx, double *cov_cam, double *cov_cam_intr, double cov_intr[4 * 4], double *cov_pt,
                      int32_t n_pairs, const int32_t *cam_a, const int32_t *cam_b, double *cov_pairs);
/* Covariance of ANY n pairs of parameter blocks (ceres::Covariance::Compute(pairs), GetCovarianceBlockInTangentSpace):
 * camera pairs that share no point, camera-point, point-point, camera-intrinsics, intrinsics, and the blocks
 * ba_gpu_covariance returns.  Same Hessian, conventions and preconditions as ba_gpu_covariance (the same factorisation and
 * relative pivot test; ba_gpu_covariance_pivots reports this call too), without the selected inversion: with A = L L^T,
 * (A^-1)_ab = (L^-1 E_a)^T (L^-1 E_b), a dot product over the common part of the two cameras' root paths in the tree.
 *   a[i], b[i] -> out: Cov(a[i], b[i]), dim(a[i]) x dim(b[i]) row-major (dims 6 / 3 / 4), the blocks back to back in order
 * A block with the fixed camera, or with constant intrinsics (DEPTH cost), is zero.  The bits of a block do not depend on the
 * other requests, and Cov(b, a) is exactly Cov(a, b)^T.  A later ba_gpu_solve or ba_gpu_covariance is unaffected.
 * BA_ERR_INVALID: n < 0, a null array with n > 0, an unknown kind, an index out of range, an intrinsics index other than 0;
 * otherwise the codes of ba_gpu_covariance.  n == 0 runs the factorisation and its pivot test only. */
enum { BA_COV_CAMERA = 0, BA_COV_POINT = 1, BA_COV_INTRINSICS = 2 };
typedef struct ba_cov_block {
  int32_t kind;  /* BA_COV_* */
  int32_t index; /* camera or point; 0 for the intrinsics */
} ba_cov_block;
int ba_gpu_covariance_blocks(ba_gpu_ctx *ctx, int32_t n, const ba_cov_block *a, const ba_cov_block *b, double *out);
/* smallest pivot / diagonal ratio of the last ba_gpu_covariance or ba_gpu_covariance_blocks call (also a rejected one):
 * ratio[0] over the camera system, ratio[1] over the intrinsics (0 when they are constant); compare with
 * BA_COV_MIN_PIVOT_RATIO */
int ba_gpu_covariance_pivots(const ba_gpu_ctx *ctx, double ratio[2]);
/* structure of the sparse Cholesky of the last upload (zeros when another solver is in force): info[0..10] as
 * ba_sparse_symbolic_info, info[11] = host microseconds of the symbolic phase, info[12] = parts of the subtree-to-rank
 * partition in force (1: one queue), info[13] = 1 when the factorisation is distributed over the ranks of the communicator
 * (every rank its own subtrees, top part replicated), info[14] = cameras of the top part, info[15] = bytes of update matrices +
 * right-hand-side updates exchanged per solve, info[16] = blocks of S summed over ranks per LM iteration (of all stored blocks
 * when the factorisation is replicated) */
int ba_gpu_spchol_info(const ba_gpu_ctx *ctx, int64_t info[24]);
/* out7[i] = pose7[i] * exp(delta6[i]) on the device (Sophus semantics) */
int ba_gpu_se3_plus(ba_gpu_ctx *ctx, int32_t n, const double *pose7,
                    const double *delta6, double *out7);

/* ---- the step before BA: batched back-projection and landmark initialisation ----
 * Replaces the per-key-point loop of getLocalPoints3D (src/Map3D.cpp:76-97) and the world-frame
 * transform of addNewLandmark (src/Map3D.cpp:44).  Host buffers:
 *   uv2f [n*2] float pixels (cv::KeyPoint::pt); depth_img [height*width] float metres, row-major
 *   (depth_frame.at<float>(trunc(v), trunc(u))); intr4 (fx,fy,cx,cy);
 *   local3 [n*3] = (z (u-cx)/fx, z (v-cy)/fy, z)            (nullable)
 *   world3 [n*3] = pose7 * local3, needs pose7 (qx..tz)     (nullable)
 * Bit-exact with the reference's plain fp64 arithmetic (no FMA contraction).  A key point outside the
 * image -> BA_ERR_INVALID (cv::Mat::at would read out of bounds). */
int ba_gpu_backproject(ba_gpu_ctx *ctx, int32_t n, const float *uv2f, const float *depth_img, int32_t width,
                       int32_t height, const double intr4[4], const double *pose7, double *local3, double *world3);

/* ---- measurement hooks (bench.py) ---- */
enum {
  BA_KERNEL_LINEARIZE = 0,    /* camera-major residual+Jacobian kernel */
  BA_KERNEL_SCHUR_MATVEC = 1, /* one implicit-Schur product (both passes) */
  BA_KERNEL_SCHUR_PASS1 = 2,  /* point-major pass  t = V^-1 W^T x only */
  BA_KERNEL_SCHUR_PASS2 = 3   /* camera-major pass y = U x - W t only */
  /* with the tiled store MATVEC is the single fused kernel and PASS1/PASS2 time the
     two-pass kernels over the same data */
};
/* Launches kernel `which` `iters` times on the context stream between two CUDA
 * events (after `warmup` untimed launches); *ms_avg = mean ms per launch. If
 * flush_l2 != 0 a >L2-sized buffer is rewritten before every timed launch and
 * each launch is timed by its own event pair. */
int ba_gpu_time_kernel(ba_gpu_ctx *ctx, int32_t which, int32_t warmup,
                       int32_t iters, int32_t flush_l2, float *ms_avg);
/* Where the time of the last ba_gpu_solve went (large-problem solvers: implicit / block-sparse): milliseconds per
 * phase, summed over the LM iterations, from CUDA events recorded on the solver stream at the phase boundaries
 * while the solve ran (not a separate profiling run).  All zero for the windowed explicit solver (graph replay). */
enum {
  BA_PHASE_START = 0, BA_PHASE_ITER0 = 1, BA_PHASE_POINT_INVERSE = 2, BA_PHASE_RHS = 3, BA_PHASE_SCHUR = 4,
  BA_PHASE_FACTOR = 5,        /* sparse Cholesky: factorisation (forward substitution fused); PCG solvers: the whole PCG */
  BA_PHASE_SUBSTITUTION = 6,  /* sparse Cholesky: backward substitution */
  BA_PHASE_BACKSUB = 7, BA_PHASE_CANDIDATE = 8, BA_PHASE_CONTROL = 9, BA_PHASE_RELINEARIZE = 10, BA_PHASE_COUNT = 11
};
int ba_gpu_phase_times(const ba_gpu_ctx *ctx, double ms[BA_PHASE_COUNT]);
const char *ba_gpu_phase_name(int32_t phase);
/* kernels launched by this context since creation */
int64_t ba_gpu_launch_count(const ba_gpu_ctx *ctx);
/* BA_JAC_* in force after the last upload (what BA_JAC_AUTO resolved to) */
int ba_gpu_jacobian_store_used(const ba_gpu_ctx *ctx);
/* block-sparse Schur structure of the last upload (BA_SOLVER_SPARSE_SCHUR_PCG / _CHOLESKY in any cost mode; zeros for the
 * other solvers): same-point observation pairs, stored upper blocks, row entries (each off-diagonal block appears twice) */
int ba_gpu_sparse_stats(const ba_gpu_ctx *ctx, int64_t *n_pairs, int32_t *n_blocks, int32_t *n_entries);

/* ---- device-resident keyframe / landmark store for sliding windows (SURVEY.md 8f row N1) ----
 * Replaces, for the optimiser's purposes, the host containers the reference re-walks for every window
 * (std::vector<KeyFrame> + Map3D, headers/CommonTypes.h:15-43, filled by src/Map3D.cpp:7-74; walked at
 * src/OptimizationUtils.cpp:244-294): observation lists, world poses and world points live in HBM, a window uploads
 * only what is new or grew.  One store per solver context (its stream, its options), not thread-safe.
 *   set_keyframe   the list of keyframe kf in the iteration order of its global_points_map: landmark ids in [0, 2^24),
 *                  float pixels (cv::KeyPoint::pt), local depths points3d_local[localId].z; replaces an earlier list
 *   set_poses      world poses of keyframes kf0 .. kf0 + n - 1
 *   set_landmarks  world points by landmark id (new landmarks; the store itself keeps optimised points up to date)
 *   window_solve   windowOptimize (:215-313) on the resident data: admissible observations (depth > 1e-15) of
 *                  kf_i..kf_f in canonical order, point ids by first appearance, frame of keyframe kf_i, first pose
 *                  constant, solve, back to the world frame.  Same bits as ba_gpu_upload / solve / download on the
 *                  host-built arrays.  ms3 (nullable): enumeration + index build, solve, write-back in milliseconds. */
typedef struct ba_store ba_store;
int ba_store_create(ba_gpu_ctx *ctx, ba_store **out);
void ba_store_destroy(ba_store *st); /* before ba_gpu_destroy of its context */
int ba_store_clear(ba_store *st);    /* forget all keyframes / landmarks, keep the device buffers */
int ba_store_set_keyframe(ba_store *st, int32_t kf, int32_t n, const int32_t *landmark_id, const float *uv2f, const double *depth);
/* several keyframes in one call (lists back to back, cnt[k] entries for keyframe kf[k]): three copies per call */
int ba_store_set_keyframes(ba_store *st, int32_t n_kf, const int32_t *kf, const int32_t *cnt, const int32_t *landmark_id,
                           const float *uv2f, const double *depth);
int ba_store_set_poses(ba_store *st, int32_t kf0, int32_t n, const double *pose7);
int ba_store_set_landmarks(ba_store *st, int32_t n, const int32_t *id, const double *xyz);
int ba_store_window_solve(ba_store *st, int32_t kf_i, int32_t kf_f, const double intr_prior4[4], double intr4[4],
                          ba_gpu_summary *summary, double *pose7_out, int32_t lm_cap, int32_t *n_pt, int32_t *landmark_of_pt,
                          double *pt3_out, int32_t *n_obs, double ms3[3]);

/* ---- symbolic phase of the sparse Cholesky of S (host only, no device needed; CPU tests drive it) ----
 * n_blk stored upper blocks (blk_i <= blk_j) of the reduced camera matrix; nested-dissection ordering of the camera
 * sequence, elimination tree, supernodes whose front panel fits cap_blocks 6x6 blocks, levels, extend-add maps
 * (csrc/ba_sparse_symbolic.h).  info[0..10] = n_cam, nodes, levels, panel blocks, update blocks, largest front (blocks),
 * largest own / border count, most children, flops, critical-path block operations; info[12 + w] = length of array w.
 * Arrays (int32): 0 perm, 1 pos, 2 node records (16 ints), 3 border lists, 4 children, 5 rel, 6 inv, 7 entries of S
 * (4 ints), 8 level_ptr, 9 level_nodes.  BA_ERR_UNSUPPORTED when a front cannot fit. */
typedef struct ba_spsym ba_spsym;
int ba_sparse_symbolic_create(int32_t n_cam, int32_t n_blk, const int32_t *blk_i, const int32_t *blk_j, int32_t leaf_cams,
                              int32_t cap_blocks, int32_t max_own, ba_spsym **out);
int ba_sparse_symbolic_info(const ba_spsym *h, int64_t info[24]);
int ba_sparse_symbolic_get(const ba_spsym *h, int32_t which, int32_t *dst);
/* Subtree-to-rank partition the multi-GPU factorisation uses for `parts` ranks (csrc/ba_sparse_symbolic.h, spsym_partition):
 * part[node] = owning rank, -1 = top part (factorised by every rank).  work[0..2] = block operations of the whole tree, of the
 * top part, of the most loaded rank.  Returns the number of parts in force (1: tree too small, the solve stays replicated). */
int ba_sparse_symbolic_partition(const ba_spsym *h, int32_t parts, int32_t *part, double work[3]);
/* Work queue of a persistent tree kernel on n_sm SMs (csrc/ba_sparse_symbolic.h): which = 0 the sparse Cholesky's
 * (spq_cholesky) for `parts` parts and the items rank `rank` runs (-1: one GPU runs every part), which = 1 the selected
 * inversion's (spq_selinv; parts and rank unused).  info[0..3] = items, then (which = 0) qB, qB_n and the number of top-part
 * cameras.  Arrays, each may be NULL: queue (node, kind per item; kind >= 0 tile, -1 factor / prepare, -2 solve, -3 finish),
 * tiles (per node), and for which = 0 qA (parts + 1), cnt_init (3 nodes + 16) and topcams.  Returns the parts in force. */
int ba_sparse_symbolic_queue(const ba_spsym *h, int32_t which, int32_t parts, int32_t rank, int32_t n_sm, int32_t info[4],
                             int32_t *queue, int32_t *tiles, int32_t *qA, int32_t *cnt_init, int32_t *topcams);

void ba_sparse_symbolic_destroy(ba_spsym *h);

/* ---- multi-GPU: one process per GPU, points sharded (SURVEY.md 8e) ---- */
/* rank 0 makes the id (128 bytes), the launcher broadcasts it, every rank
 * calls comm_init before upload. Uses NCCL (dlopen'ed libnccl.so.2). */
int ba_gpu_comm_unique_id(char id128[128]);
int ba_gpu_comm_init(ba_gpu_ctx *ctx, const char id128[128], int32_t rank,
                     int32_t n_ranks);

#ifdef __cplusplus
}
#endif
#endif
