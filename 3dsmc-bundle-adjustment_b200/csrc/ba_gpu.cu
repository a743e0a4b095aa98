// ba_gpu.cu -- C-ABI of the B200-native windowed bundle-adjustment solver
// (include/ba_gpu.h).  Host orchestration only: every floating-point operation of
// the solve runs in the sm_100a kernels of ba_kernels.cuh; the host enqueues
// whole LM iterations and polls a device-side termination flag.
//
// Boundary replaced: the ceres::Problem / ceres::Solve calls of
// src/OptimizationUtils.cpp:218-300 (reference paths relative to /root/reference).
// There is NO CPU fallback: without a CUDA device ba_gpu_create fails.
#include "../../include/ba_gpu.h"
#include "ba_kernels.cuh"
#include "ba_kernels_fact.cuh"
#include "ba_kernels_tile.cuh"
#include "ba_kernels_sparse.cuh"
#include "ba_kernels_dist.cuh"
#include "ba_kernels_chol.cuh"
#include "ba_kernels_spchol.cuh"
#include "ba_kernels_selinv.cuh"
#include "ba_kernels_store.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>

#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

// ------------------------------------------------------------------ NCCL (dlopen)
typedef struct ncclComm *ncclComm_t;
typedef struct {
  char internal[128];
} ncclUniqueId;
typedef int ncclResult_t;
enum { ncclSum_ = 0, ncclMax_ = 2 };
enum { ncclUint64_ = 5, ncclFloat64_ = 8 };
struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static bool nccl_load(std::string *err) {
  if (g_nccl.lib) return true;
  const char *names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char *n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) {
    *err = std::string("dlopen libnccl.so.2 failed: ") + dlerror();
    return false;
  }
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(g_nccl.lib, "ncclAllGather");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(g_nccl.lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.AllGather) {
    *err = "libnccl is missing required symbols";
    return false;
  }
  return true;
}

// ------------------------------------------------------------------ context
struct Buf {
  void *p = nullptr;
  size_t cap = 0;
};

struct ba_gpu_ctx {
  ba_gpu_options opt;
  int device = 0, n_sm = 148;
  cudaStream_t stream = nullptr;
  // second stream for the independent branches of an LM iteration (fork / join by events): the windowed
  // problems are chains of ~25 latency-bound small kernels, several of which do not depend on each other
  cudaStream_t stream2 = nullptr, cur = nullptr;
  cudaStream_t stream3 = nullptr;  // blocked Cholesky look-ahead: bulk of the trailing update
  cudaEvent_t ev_panel = nullptr, ev_trsm = nullptr, ev_col[2] = {nullptr, nullptr}, ev_bulk2[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_mid = nullptr;
  bool forking = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  int64_t launches = 0;
  bool uploaded = false, linearized = false;
  std::vector<Buf *> bufs;

  // sizes
  int n_cam = 0, n_pt = 0, n_obs = 0, fixed_cam = -1, n_free = 0, n_items = 0;
  int depth = 0, nk = 0;  // cost-model switches in force
  int solver = 0, n_red = 0;
  int nblk_obs = 0, nblk_ent = 0, nblk_cam = 0, nblk_pt = 0, n_tiles = 0, nblk_item = 0, pl_tile_pts = BA_TILE_PTS, pl_tiles = 0;
  CostParams cp;
  LmOptions lo;

  // problem
  Buf pose, pose_c, pt, pt_c, intr, intr_c, intr_prior;
  Buf cam_idx, pt_idx, uv, depthv;
  Buf perm, pt_rowptr, cam_rowptr, pt_cnt, cam_cnt, cursor, err_flag;
  Buf pm_cam, pm_pt, pm_uv, pm_depth;
  Buf items, item_ptr, item_cnt, cam_slot;
  // Jacobian planes (materialised store) / factored store
  Buf jcm, jpm;
  JPlanes Jc_, Jp_;
  bool fact = false, planes_ready = false;
  Buf fcm, fpm, geo, camx, Vs, ts, tgs, ys, tile_lo, tile_span;
  bool staged = false;
  FPlanes Fc_, Fp_;
  // tile-fused product (ba_kernels_tile.cuh)
  Buf tmeta, tseg, tout, taux, tm_cam, tm_pt, tm_uv, ftm, cam_tmin, cam_tmax, tcnt, tpart_ptr, part6t;
  bool tiled = false;
  int tile_npt = 0, n_tparts = 0;
  double2 *Tg0 = nullptr, *Tg1 = nullptr;
  // explicit block-sparse Schur complement (ba_kernels_sparse.cuh)
  Buf sp_cnt, sp_off, sp_keys, sp_vals, sp_keys2, sp_pairs, sp_ukeys, sp_ucnt, sp_nruns, sb_ptr, sb_i, sb_j, row_ucnt, row_tcnt,
      row_ustart, row_tstart, sp_tkeys, sp_tvals, sp_tkeys2, sp_tvals2, ent_ptr, ent, Sblk, ysp, cub_tmp, dsq, row_pq;
  int n_sblk = 0, n_sblk_local = 0, n_ent = 0, pcg_grid = 0, sp_ctas_per_sm = 1;
  Buf sp_pair_pt, chol_v, chol_linv, chol_lsub, chol_slots;
  // one LM iteration of the windowed explicit solver as an instantiated CUDA graph (every decision is taken on the
  // device, so the node parameters never change between iterations); upload / set_options mark it stale and the next
  // solve re-captures and updates the executable in place (cudaGraphExecUpdate: destroying and re-instantiating it cost
  // 0.2 + 0.1 ms per window)
  cudaGraphExec_t lm_graph = nullptr;
  int64_t lm_graph_launches = 0;
  bool lm_graph_off = false, lm_graph_stale = true;
  bool spmv6 = false;  // BA_SPMV6=1: six-lanes-per-block product kernel in the launch-per-step PCG / product hook (experiment)
  bool sps_simt = false;  // BA_SPS_SIMT=1: values of S by k_sp_schur_simt instead of the DMMA kernel (A/B comparisons only)
  bool pdl = false, pdl_off = false;  // programmatic dependent launches inside the windowed LM iteration (BA_NO_PDL=1: off)
  int legacy_chol = 0;  // BA_LEGACY_CHOL=1: left-looking single-CTA Cholesky, =2: shared-memory L D L^T, =3: grid-barrier blocked substitution (A/B timing only)
  Buf sp_lkeys, sp_gid, sp_gather, sp_gsorted, sp_diag, sp_scal;
  // row-sharded persistent PCG over NVLink peer memory (ba_kernels_dist.cuh)
  Buf my_rows, row_flag, row_pos, ipc_stage;
  void *xch = nullptr;          // own exchange buffer (cudaMalloc, cudaIpc-exported)
  size_t xch_cap = 0;
  int xch_ncam = 0;
  void *xch_peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  PcgFan fan;
  bool dist_pcg = false;
  int n_my_rows = 0, dist_grid = 0;
  long long n_pairs = 0;
  // exact sparse Cholesky of S (ba_sparse_symbolic.h / ba_kernels_spchol.cuh)
  bool src_on_device = false;   // the arrays handed to the current upload live in device memory (ba_store_window_solve)
  bool spchol = false;          // the block-sparse solver factorises S instead of running PCG
  SpSymbolic sym;               // host-side structure of the last upload
  Buf spn_node, spn_bord, spn_children, spn_rel, spn_inv, spn_aent, spn_perm, spn_levels;
  Buf spc_panel, spc_U, spc_z, spc_linv, spc_ypos, spc_prof, spc_queue, spc_tiles, spc_cnt, spc_cnt_init, spc_topcams;
  int spc_n_items = 0;
  // subtree-to-rank partition (spsym_partition): phase A = the subtrees of one part (queue items spc_qA[p] .. spc_qA[p + 1]),
  // phase B = top part + backward substitution (spc_qB, spc_qB_n).  spc_dist: part p runs on rank p and the head of spc_U
  // (update matrices of the subtree roots + right-hand-side updates, spc_xchg doubles) is summed over ranks in between;
  // on one GPU (BA_SPCHOL_PARTS, tests) the parts run one after the other.
  int spc_parts = 1, spc_qA[BA_MAX_RANKS + 1] = {0}, spc_qB = 0, spc_qB_n = 0, spc_n_topcams = 0;
  bool spc_dist = false;
  size_t spc_xchg = 0, spc_ru_off = 0;
  // distributed factorisation: a rank assembles only its own subtrees and the top part, so only the blocks of S some rank
  // contributes to WITHOUT factorising them (shard borders, top part) are summed over ranks: spc_nx block ids in spc_xidx
  Buf spc_xidx, spc_xbuf;
  int spc_nx = 0;
  bool sp_full_next = false;  // the next enqueue_sparse_values() completes ALL of S on every rank (product hook)
  bool spc_tree = true;         // one persistent launch with dependency counters (BA_SPCHOL_LEVELS=1: one launch per tree level)
  size_t spc_smem_factor = 0, spc_smem_solve = 0, spc_smem_update = 0;
  double sym_ms = 0.0;          // host time of the symbolic phase (last upload)
  // sparse Cholesky of the REF / depth-prior / free-intrinsics cost (solver = EXPLICIT_CHOLESKY's linearisation and W / WV,
  // the block-sparse S and the tree instead of the dense S): right-hand-side rows of the tree (5 with the intrinsics border),
  // B by camera [24 n_cam], Z = L^-1 B by position [24 n_cam], the corner C + b_k [20], the per-CTA border partials
  bool sp_ref = false;
  int spc_nrhs = 1;
  Buf spb_B, spb_Z, spb_kk, spb_part;
  // covariance (ba_gpu_covariance, ba_kernels_selinv.cuh), built by the first call after an upload: selected-inversion queue,
  // Y scratch (panel-shaped), X = A^-1 B by position [4 x 6 n_cam], T^-1, Sigma on the stored blocks of S, Sigma_ck (scaled),
  // block -> front records, camera -> position, outputs
  bool cov_ready = false;
  int cov_n_items = 0;
  size_t cov_smem = 0;
  Buf cov_Y, cov_X, cov_zq, cov_yscr, cov_Tinv, cov_S, cov_ck, cov_brec, cov_pos, cov_queue, cov_tiles, cov_cnt, cov_cam, cov_ci,
      cov_pt, cov_pin, cov_pout, cov_bad, cov_piv;
  double cov_ratio[2] = {0.0, 0.0};  // smallest pivot / diagonal of the last covariance call: cameras, intrinsics (0: none)
  // phase timing of the large-problem solvers: CUDA events on the solver stream at the phase boundaries of every LM
  // iteration of the last solve (a few dozen event records per iteration: < 0.1 % of a multi-millisecond iteration)
  std::vector<cudaEvent_t> ph_ev;
  std::vector<int> ph_id;
  int ph_n = 0;
  bool ph_on = false;
  double ph_ms[BA_PHASE_COUNT] = {0};
  Buf p2, pcg_bar, wb_rho, wb_Q, bp_buf, err_flag_bp, row_keys, row_keys2, row_ids, row_order;
  // scaling / diag / gradient / blocks
  Buf sc, sp, sk, dc, dp, dk, gc, gp, gk, U, Uck, Ukk, V, Vinv, Wk, tg, t, yc, yp, yk, rk, Jkk;
  Buf one_c, one_p, one_k;
  // PCG
  Buf b, x, r, z, p, q, Minv;
  // partials
  Buf part_blk, part6, part21, part_ex, part_kk;
  Buf pc_lin, pc_cand, pc_mcc, pe_gmax, pe_xn, pe_step, pcam_rho, pcam_bb, pcam_pq, pcam_Q;
  // multi-GPU staging (dense per-camera sums, scalars, identity item_ptr)
  Buf red_blk, red6, red21, scal, ident;
  // explicit solver
  Buf W, WV, S, rhs, blk_i, blk_j, blk_cam, pair_ptr, pair_a, pair_b;
  Buf ex_keys, ex_keys2, ex_vals, ex_vals2, blk_cnt;  // device-built pair list (windows)
  int n_blk = 0;
  int ex_band_cams = -1;  // largest camera-slot distance of a non-empty block of the dense explicit S (-1: unknown = dense)
  // controller
  Buf st, trace;
  LmState *h_st = nullptr;  // pinned
  ba_gpu_summary last_summary;
  std::vector<BaIterRec> h_trace;
  // L2 flush scratch for ba_gpu_time_kernel
  Buf flush;
  // multi-GPU
  ncclComm_t comm = nullptr;
  int rank = 0, n_ranks = 1;
  int64_t collectives = 0;
  bool comm_error = false;
};

static thread_local std::string g_create_err;

static int fail(ba_gpu_ctx *c, int code, const char *fmt, ...) {
  char tmp[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tmp, sizeof(tmp), fmt, ap);
  va_end(ap);
  if (c)
    c->err = tmp;
  else
    g_create_err = tmp;
  return code;
}

#define CK(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(ctx, BA_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                       __FILE__, __LINE__);                                               \
  } while (0)

static int buf_reserve(ba_gpu_ctx *ctx, Buf &b, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (b.cap >= bytes) return 0;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  const size_t want = bytes + bytes / 8 + 256;  // head-room for sliding windows
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) return fail(ctx, BA_ERR_CUDA, "cudaMalloc(%zu): %s", want, cudaGetErrorString(e));
  b.cap = want;
  if (std::find(ctx->bufs.begin(), ctx->bufs.end(), &b) == ctx->bufs.end()) ctx->bufs.push_back(&b);
  return 0;
}
#define RES(buf, bytes)                                      \
  do {                                                       \
    int rc_ = buf_reserve(ctx, ctx->buf, (size_t)(bytes));   \
    if (rc_) return rc_;                                     \
  } while (0)

template <class T>
static T *P(const Buf &b) {
  return reinterpret_cast<T *>(b.p);
}
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
// dense explicit Schur complement: n^2 doubles (2 GiB at the limit), blocked Cholesky above 1024
#define BA_EXPLICIT_MAX_DIM 16384
static size_t tile_smem_bytes(int npt) {
  return ((size_t)6 * (npt * BA_THREADS + 8) + 3 * BA_TILE_PTS + BA_TILE_MAXSPAN * BA_TILE_QREC + BA_TILE_MAXSPAN * 6) * 8;
}

// ctx->pdl (windowed explicit LM iteration only): programmatic stream serialisation -- the kernel's CTAs may be made
// resident before the previous kernel of the stream has finished; every kernel launched in that region starts with
// pdl_wait() (ba_kernels.cuh; tests/test_cabi_cpu.py audits the sources)
#define LAUNCH(kern, grid, block, smem, ...)                                          \
  do {                                                                                \
    if ((grid) > 0) {                                                                 \
      if (ctx->pdl) {                                                                 \
        cudaLaunchConfig_t cfg_ = {};                                                 \
        cfg_.gridDim = dim3(grid);                                                    \
        cfg_.blockDim = dim3(block);                                                  \
        cfg_.dynamicSmemBytes = (smem);                                               \
        cfg_.stream = ctx->cur;                                                       \
        cudaLaunchAttribute at_[1];                                                   \
        at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;               \
        at_[0].val.programmaticStreamSerializationAllowed = 1;                        \
        cfg_.attrs = at_;                                                             \
        cfg_.numAttrs = 1;                                                            \
        cudaLaunchKernelEx(&cfg_, kern, __VA_ARGS__);                                 \
      } else {                                                                        \
        kern<<<(grid), (block), (smem), ctx->cur>>>(__VA_ARGS__);                     \
      }                                                                               \
      ctx->launches++;                                                                \
    }                                                                                 \
  } while (0)

// dispatch on the cost-model switches (template parameters of the kernels)
#define DISPATCH_DK(D, K, ...)          \
  do {                                  \
    if ((D) && (K)) {                   \
      constexpr int DD = 1, KK = 4;     \
      __VA_ARGS__;                      \
    } else if ((D)) {                   \
      constexpr int DD = 1, KK = 0;     \
      __VA_ARGS__;                      \
    } else if ((K)) {                   \
      constexpr int DD = 0, KK = 4;     \
      __VA_ARGS__;                      \
    } else {                            \
      constexpr int DD = 0, KK = 0;     \
      __VA_ARGS__;                      \
    }                                   \
  } while (0)
#define DISPATCH_D(D, ...)          \
  do {                              \
    if ((D)) {                      \
      constexpr int DD = 1;         \
      __VA_ARGS__;                  \
    } else {                        \
      constexpr int DD = 0;         \
      __VA_ARGS__;                  \
    }                               \
  } while (0)

// ------------------------------------------------------------------ options
extern "C" void ba_gpu_default_options(ba_gpu_options *o) {
  memset(o, 0, sizeof(*o));
  // headers/BundleAdjustmentConfig.h:47-50, 64-65
  o->HUB_P_REPR = 1e-3;
  o->WEIGHT_INTRINSICS = 1e-6;
  o->WEIGHT_UNPR = 10.0;
  o->HUB_P_UNPR = 1e-3;
  o->max_num_iterations = 75;
  o->eta = 1e-6;
  o->use_depth_prior = 1;
  o->optimize_intrinsics = 1;
  o->solver = BA_SOLVER_AUTO;
  o->explicit_max_dim = 160;
  o->n_obs_total = 0;
  // ceres 2.0.0 Solver::Options defaults
  o->function_tolerance = 1e-6;
  o->gradient_tolerance = 1e-10;
  o->parameter_tolerance = 1e-8;
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->max_num_consecutive_invalid_steps = 5;
  o->jacobi_scaling = 1;
  o->max_linear_solver_iterations = 500;
  o->min_linear_solver_iterations = 0;
  o->residual_reset_period = 10;
  o->device = -1;
  o->poll_interval = 10;
  o->persistent_pcg = 1;
  o->jacobian_store = BA_JAC_AUTO;
  o->sparse_max_pairs_per_obs = 16;
}

static int check_options(ba_gpu_ctx *ctx, const ba_gpu_options *o) {
  if (!(o->HUB_P_REPR > 0.0) || !(o->HUB_P_UNPR > 0.0) || !(o->WEIGHT_UNPR >= 0.0) || !(o->WEIGHT_INTRINSICS >= 0.0))
    return fail(ctx, BA_ERR_INVALID, "Huber deltas must be > 0 and weights >= 0");
  if (o->max_num_iterations < 0 || o->max_num_iterations > 10000000 || o->poll_interval < 1)
    return fail(ctx, BA_ERR_INVALID, "bad iteration options (0 <= max_num_iterations <= 10^7, poll_interval >= 1)");
  if (o->solver < BA_SOLVER_AUTO || o->solver > BA_SOLVER_SPARSE_SCHUR_CHOLESKY) return fail(ctx, BA_ERR_INVALID, "bad solver");
  if (o->jacobian_store < BA_JAC_AUTO || o->jacobian_store > BA_JAC_TILED) return fail(ctx, BA_ERR_INVALID, "bad jacobian_store");
  if (!(o->initial_trust_region_radius > 0.0)) return fail(ctx, BA_ERR_INVALID, "bad trust-region radius");
  return 0;
}

extern "C" void ba_gpu_destroy(ba_gpu_ctx *ctx);
extern "C" int ba_gpu_create(const ba_gpu_options *o, ba_gpu_ctx **out) {
  if (!o || !out) return fail(nullptr, BA_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, BA_ERR_CUDA, "no CUDA device (%s); this library has no CPU fallback",
                e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
  ba_gpu_ctx *ctx = new ba_gpu_ctx();
  int rc = check_options(ctx, o);
  if (rc) {
    g_create_err = ctx->err;
    delete ctx;
    return rc;
  }
  ctx->opt = *o;
  int dev = o->device;
  if (dev < 0) cudaGetDevice(&dev);
  ctx->device = dev;
  auto bail = [&](const char *what, cudaError_t ce) {
    fail(nullptr, BA_ERR_CUDA, "%s: %s", what, cudaGetErrorString(ce));
    ba_gpu_destroy(ctx);  // releases whatever was created so far (streams, events, pinned state)
    return BA_ERR_CUDA;
  };
  if ((e = cudaSetDevice(dev)) != cudaSuccess) return bail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
  ctx->n_sm = prop.multiProcessorCount;
  if (prop.major < 10) {
    fail(nullptr, BA_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
    ba_gpu_destroy(ctx);
    return BA_ERR_CUDA;
  }
  // main / side stream at the highest priority, a third one at the lowest for the bulk of the blocked Cholesky's trailing
  // update: the CTAs of the critical chain (next column, diagonal tile, panel) are dispatched ahead of the queued bulk
  int prio_least = 0, prio_greatest = 0;
  cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
  if ((e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_greatest)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_greatest)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithPriority(&ctx->stream3, cudaStreamNonBlocking, prio_least)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_panel, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_trsm, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  for (int i = 0; i < 2; ++i) {
    if ((e = cudaEventCreateWithFlags(&ctx->ev_col[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_bulk2[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  }
  ctx->cur = ctx->stream;
  if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_mid, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaMallocHost((void **)&ctx->h_st, sizeof(LmState))) != cudaSuccess) return bail("cudaMallocHost", e);
  ctx->legacy_chol = getenv("BA_LEGACY_CHOL") ? atoi(getenv("BA_LEGACY_CHOL")) : 0;
  ctx->lm_graph_off = getenv("BA_NO_LM_GRAPH") != nullptr;
  ctx->pdl_off = getenv("BA_NO_PDL") != nullptr;
  ctx->spmv6 = getenv("BA_SPMV6") != nullptr;
  ctx->sps_simt = getenv("BA_SPS_SIMT") && atoi(getenv("BA_SPS_SIMT")) != 0;
  cudaFuncSetAttribute(k_sp_schur, cudaFuncAttributeMaxDynamicSharedMemorySize, BA_SPS_SMEM);
  cudaFuncSetAttribute(k_cholesky_solve<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024);
  cudaFuncSetAttribute(k_ldlt_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt_smem_bytes(BA_LDLT_MAX_N));
  cudaFuncSetAttribute(k_ldlt2_solve<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt2_smem_bytes(31));
  cudaFuncSetAttribute(k_ldlt2_solve<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt2_smem_bytes(63));
  cudaFuncSetAttribute(k_ldlt2_solve<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt2_smem_bytes(95));
  cudaFuncSetAttribute(k_ldlt2_solve<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt2_smem_bytes(127));
  cudaFuncSetAttribute(k_ldlt2_solve<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldlt2_smem_bytes(BA_LDLT2_MAX_N));
  cudaFuncSetAttribute(k_chol_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_UPD_SMEM);
  cudaFuncSetAttribute(k_chol_trsm, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * CH_NB * CH_LD * 8);
  cudaFuncSetAttribute(k_chol_trsm2, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * CH_NB * CH_LD * 8);
  cudaFuncSetAttribute(k_chol_potrf2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_potrf2_smem_bytes());
  cudaFuncSetAttribute(kt_schur_fused<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(2));
  cudaFuncSetAttribute(kt_schur_fused<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(3));
  cudaFuncSetAttribute(kt_schur_fused<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(4));
  cudaFuncSetAttribute(kt_schur_fused<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(6));
  cudaFuncSetAttribute(kt_schur_fused<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(8));
  *out = ctx;
  return BA_OK;
}

static void drop_lm_graph(ba_gpu_ctx *ctx) {
  if (ctx->lm_graph) cudaGraphExecDestroy(ctx->lm_graph);
  ctx->lm_graph = nullptr;
}

extern "C" void ba_gpu_destroy(ba_gpu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  drop_lm_graph(ctx);
  if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->comm);
  for (int k = 0; k < 8; ++k)
    if (ctx->xch_peer[k] && k != ctx->rank) cudaIpcCloseMemHandle(ctx->xch_peer[k]);
  if (ctx->xch) cudaFree(ctx->xch);
  for (Buf *b : ctx->bufs)
    if (b->p) cudaFree(b->p);
  if (ctx->h_st) cudaFreeHost(ctx->h_st);
  if (ctx->stream2) cudaStreamSynchronize(ctx->stream2);
  if (ctx->stream3) {
    cudaStreamSynchronize(ctx->stream3);
    cudaStreamDestroy(ctx->stream3);
  }
  for (cudaEvent_t e : ctx->ph_ev) cudaEventDestroy(e);
  if (ctx->ev_panel) cudaEventDestroy(ctx->ev_panel);
  if (ctx->ev_trsm) cudaEventDestroy(ctx->ev_trsm);
  for (int i = 0; i < 2; ++i) {
    if (ctx->ev_col[i]) cudaEventDestroy(ctx->ev_col[i]);
    if (ctx->ev_bulk2[i]) cudaEventDestroy(ctx->ev_bulk2[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_mid) cudaEventDestroy(ctx->ev_mid);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" const char *ba_gpu_last_error(const ba_gpu_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int ba_gpu_set_options(ba_gpu_ctx *ctx, const ba_gpu_options *o) {
  if (!ctx || !o) return BA_ERR_INVALID;
  int rc = check_options(ctx, o);
  if (rc) return rc;
  const int dev = ctx->opt.device;
  ctx->opt = *o;
  ctx->opt.device = dev;
  ctx->uploaded = false;
  ctx->lm_graph_stale = true;
  return BA_OK;
}

extern "C" int64_t ba_gpu_launch_count(const ba_gpu_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int ba_gpu_sparse_stats(const ba_gpu_ctx *ctx, int64_t *n_pairs, int32_t *n_blocks, int32_t *n_entries) {
  if (!ctx || !ctx->uploaded) return BA_ERR_STATE;
  // block-sparse S in force: the NS solvers (PCG and Cholesky: ctx->solver == SPARSE_SCHUR_PCG) and the sparse Cholesky with
  // depth prior / free intrinsics (ctx->sp_ref)
  const bool sp = ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG || ctx->sp_ref;
  if (n_pairs) *n_pairs = sp ? ctx->n_pairs : 0;
  if (n_blocks) *n_blocks = sp ? ctx->n_sblk : 0;
  if (n_entries) *n_entries = sp ? ctx->n_ent : 0;
  return BA_OK;
}
extern "C" int ba_gpu_jacobian_store_used(const ba_gpu_ctx *ctx) {
  if (!ctx || !ctx->uploaded) return BA_ERR_STATE;
  return ctx->tiled ? BA_JAC_TILED : (ctx->fact ? BA_JAC_FACTORED : BA_JAC_PLANES);
}

// ------------------------------------------------------------------ upload
static void set_planes(JPlanes &J, double *base, size_t n_pad, int depth, int nk) {
  // every plane is n_pad double2 (or double) long and 256-byte aligned
  size_t off = 0;
  auto take2 = [&]() {
    double2 *p = reinterpret_cast<double2 *>(base + off);
    off += 2 * n_pad;
    return p;
  };
  auto take1 = [&]() {
    double *p = base + off;
    off += n_pad;
    return p;
  };
  memset(&J, 0, sizeof(J));
  J.r = take2();
  for (int k = 0; k < 6; ++k) J.Jc[k] = take2();
  for (int k = 0; k < 3; ++k) J.Jp[k] = take2();
  if (depth) {
    J.r3 = take1();
    for (int k = 0; k < 6; ++k) J.Jc3[k] = take1();
    for (int k = 0; k < 3; ++k) J.Jp3[k] = take1();
  }
  if (nk) {
    J.Jk[0] = take2();
    J.Jk[1] = take2();
  }
}
static size_t planes_doubles(size_t n_pad, int depth, int nk) { return n_pad * (20 + (depth ? 10 : 0) + (nk ? 4 : 0)); }

__global__ void k_fill(double *p, size_t n, double v) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void k_slots(int n_cam, int fixed_cam, int32_t *slot) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n_cam) slot[c] = (c == fixed_cam) ? -1 : (fixed_cam >= 0 && c > fixed_cam ? c - 1 : c);
}

// host-side pair list of the explicit Schur complement: for every block pair
// (i <= j) of free-camera slots the (obs_a, obs_b) pairs that share a point, in
// point-major order.  Pure index plumbing; values never touch the host.
static int build_pair_list(ba_gpu_ctx *ctx, const int32_t *cam_idx, const int32_t *pt_idx) {
  const int n_obs = ctx->n_obs, n_pt = ctx->n_pt, nf = ctx->n_free;
  std::vector<int32_t> rowptr((size_t)n_pt + 1, 0), perm((size_t)n_obs);
  for (int i = 0; i < n_obs; ++i) rowptr[pt_idx[i] + 1]++;
  for (int p = 0; p < n_pt; ++p) rowptr[p + 1] += rowptr[p];
  {
    std::vector<int32_t> cur(rowptr.begin(), rowptr.end() - 1);
    for (int i = 0; i < n_obs; ++i) perm[cur[pt_idx[i]]++] = i;
  }
  auto slot = [&](int c) { return c == ctx->fixed_cam ? -1 : (ctx->fixed_cam >= 0 && c > ctx->fixed_cam ? c - 1 : c); };
  const size_t nb_all = (size_t)nf * (nf + 1) / 2;
  auto bidx = [&](int i, int j) { return (size_t)i * nf - (size_t)i * (i - 1) / 2 + (j - i); };
  std::vector<int64_t> cnt(nb_all + 1, 0);
  for (int p = 0; p < n_pt; ++p)
    for (int a = rowptr[p]; a < rowptr[p + 1]; ++a) {
      const int sa = slot(cam_idx[perm[a]]);
      if (sa < 0) continue;
      for (int b = rowptr[p]; b < rowptr[p + 1]; ++b) {
        const int sb = slot(cam_idx[perm[b]]);
        if (sb < sa) continue;
        cnt[bidx(sa, sb) + 1]++;
      }
    }
  // keep every diagonal block (damping only when a camera has no observation)
  std::vector<int32_t> bi, bj, bc, pptr;
  std::vector<int64_t> start(nb_all, -1);
  int64_t total = 0;
  std::vector<int> slot_cam(nf);
  for (int c = 0; c < ctx->n_cam; ++c)
    if (slot(c) >= 0) slot_cam[slot(c)] = c;
  for (int i = 0; i < nf; ++i)
    for (int j = i; j < nf; ++j) {
      const size_t k = bidx(i, j);
      if (cnt[k + 1] == 0 && i != j) continue;
      start[k] = total;
      bi.push_back(i);
      bj.push_back(j);
      bc.push_back(slot_cam[i]);
      pptr.push_back((int32_t)total);
      total += cnt[k + 1];
    }
  if (total > 0x7fffffff) return fail(ctx, BA_ERR_UNSUPPORTED, "explicit Schur pair list too large");
  pptr.push_back((int32_t)total);
  std::vector<int32_t> pa((size_t)total), pb((size_t)total);
  std::vector<int64_t> cur(start);
  for (int p = 0; p < n_pt; ++p)
    for (int a = rowptr[p]; a < rowptr[p + 1]; ++a) {
      const int sa = slot(cam_idx[perm[a]]);
      if (sa < 0) continue;
      for (int b = rowptr[p]; b < rowptr[p + 1]; ++b) {
        const int sb = slot(cam_idx[perm[b]]);
        if (sb < sa) continue;
        const int64_t w = cur[bidx(sa, sb)]++;
        pa[w] = perm[a];
        pb[w] = perm[b];
      }
    }
  ctx->n_blk = (int)bi.size();
  ctx->ex_band_cams = 0;
  for (size_t b = 0; b < bi.size(); ++b) ctx->ex_band_cams = std::max(ctx->ex_band_cams, bj[b] - bi[b]);
  RES(blk_i, bi.size() * 4);
  RES(blk_j, bi.size() * 4);
  RES(blk_cam, bi.size() * 4);
  RES(pair_ptr, pptr.size() * 4);
  RES(pair_a, pa.size() * 4);
  RES(pair_b, pb.size() * 4);
  CK(cudaMemcpyAsync(ctx->blk_i.p, bi.data(), bi.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->blk_j.p, bj.data(), bj.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->blk_cam.p, bc.data(), bc.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->pair_ptr.p, pptr.data(), pptr.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  if (total) {
    CK(cudaMemcpyAsync(ctx->pair_a.p, pa.data(), pa.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->pair_b.p, pb.data(), pb.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));  // host vectors die here
  return 0;
}

// materialised Jacobian planes, allocated on demand (always for the explicit /
// REF path; lazily for the un-scaled evaluation hook when the store is factored)
static int ensure_planes(ba_gpu_ctx *ctx) {
  if (ctx->planes_ready) return 0;
  const size_t n_pad = ((size_t)ctx->n_obs + 31) / 32 * 32 + 32;
  RES(jcm, planes_doubles(n_pad, ctx->depth, ctx->nk) * 8);
  RES(jpm, planes_doubles(n_pad, ctx->depth, ctx->nk) * 8);
  set_planes(ctx->Jc_, P<double>(ctx->jcm), n_pad, ctx->depth, ctx->nk);
  set_planes(ctx->Jp_, P<double>(ctx->jpm), n_pad, ctx->depth, ctx->nk);
  ctx->planes_ready = true;
  return 0;
}

// structure of the explicit block-sparse Schur complement (integer-only, device-built;
// the radix sort / scan / run-length steps are CUB library calls, setup only)
#define CUBCALL(fn, ...)                                                  \
  do {                                                                    \
    size_t tb_ = 0;                                                       \
    CK(fn(nullptr, tb_, __VA_ARGS__, ctx->stream));                       \
    RES(cub_tmp, tb_ + 16);                                               \
    CK(fn(ctx->cub_tmp.p, tb_, __VA_ARGS__, ctx->stream));                \
  } while (0)
static int nccl_allreduce(ba_gpu_ctx *ctx, double *buf, size_t n, bool is_max);
// host scalar combined over the ranks (setup only)
static int allreduce_host_scalar(ba_gpu_ctx *ctx, double *v, bool is_max) {
  if (ctx->n_ranks == 1) return 0;
  RES(sp_scal, 64);
  CK(cudaMemcpyAsync(ctx->sp_scal.p, v, 8, cudaMemcpyHostToDevice, ctx->stream));
  int rc = nccl_allreduce(ctx, P<double>(ctx->sp_scal), 1, is_max);
  if (rc) return rc;
  CK(cudaMemcpyAsync(v, ctx->sp_scal.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
// pair list of the dense explicit solver, device-built (windowed problems: the host loop of build_pair_list()
// plus its six host->device copies were the largest part of ba_gpu_upload).  Every block of the upper triangle is
// listed; k_schur_pairs skips the empty off-diagonal ones.
static int build_pair_list_device(ba_gpu_ctx *ctx) {
  const int n_pt = ctx->n_pt, nf = ctx->n_free;
  const int nb_all = nf * (nf + 1) / 2;
  cudaStream_t s = ctx->stream;
  RES(sp_cnt, ((size_t)n_pt + 2) * 8);
  RES(sp_off, ((size_t)n_pt + 2) * 8);
  LAUNCH(k_sp_count, cdiv(n_pt + 1, BA_THREADS), BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
         ctx->fixed_cam, P<long long>(ctx->sp_cnt));
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<long long>(ctx->sp_cnt), P<long long>(ctx->sp_off), n_pt + 1);
  long long n_pairs = 0;
  CK(cudaMemcpyAsync(&n_pairs, P<long long>(ctx->sp_off) + n_pt, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (n_pairs > 0x7fffffffLL) return fail(ctx, BA_ERR_UNSUPPORTED, "explicit Schur pair list too large");
  const size_t np1 = (size_t)n_pairs + 1;
  RES(ex_keys, np1 * 4);
  RES(ex_keys2, np1 * 4);
  RES(ex_vals, np1 * 8);
  RES(ex_vals2, np1 * 8);
  RES(blk_cnt, ((size_t)nb_all + 2) * 4);
  RES(blk_i, ((size_t)nb_all + 1) * 4);
  RES(blk_j, ((size_t)nb_all + 1) * 4);
  RES(blk_cam, ((size_t)nb_all + 1) * 4);
  RES(pair_ptr, ((size_t)nb_all + 2) * 4);
  RES(pair_a, np1 * 4);
  RES(pair_b, np1 * 4);
  CK(cudaMemsetAsync(ctx->blk_cnt.p, 0, ((size_t)nb_all + 2) * 4, s));
  LAUNCH(k_ex_emit, ctx->nblk_pt, BA_THREADS, 0, n_pt, nf, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->perm),
         ctx->fixed_cam, P<long long>(ctx->sp_off), P<uint32_t>(ctx->ex_keys), P<unsigned long long>(ctx->ex_vals),
         P<int32_t>(ctx->blk_cnt));
  if (n_pairs > 0) {
    int bits = 1;
    while (bits < 31 && (1 << bits) < nb_all) ++bits;
    CUBCALL(cub::DeviceRadixSort::SortPairs, P<uint32_t>(ctx->ex_keys), P<uint32_t>(ctx->ex_keys2),
            P<unsigned long long>(ctx->ex_vals), P<unsigned long long>(ctx->ex_vals2), (int)n_pairs, 0, bits);
  }
  LAUNCH(k_exclusive_scan, 1, 1024, 0, nb_all, P<int32_t>(ctx->blk_cnt), P<int32_t>(ctx->pair_ptr));
  LAUNCH(k_ex_finish, cdiv(std::max((int)n_pairs, nf * nf), BA_THREADS), BA_THREADS, 0, (int)n_pairs,
         P<unsigned long long>(ctx->ex_vals2), P<int32_t>(ctx->pair_a), P<int32_t>(ctx->pair_b), nf, ctx->fixed_cam,
         P<int32_t>(ctx->blk_i), P<int32_t>(ctx->blk_j), P<int32_t>(ctx->blk_cam));
  ctx->n_blk = nb_all;
  ctx->ex_band_cams = -1;  // (windows: every block of the upper triangle is listed; at most 7 tiles anyway)
  return 0;
}

static int sparse_count_pairs(ba_gpu_ctx *ctx, long long *n_pairs_out) {
  const int n_pt = ctx->n_pt;
  cudaStream_t s = ctx->stream;
  RES(sp_cnt, ((size_t)n_pt + 2) * 8);
  RES(sp_off, ((size_t)n_pt + 2) * 8);
  LAUNCH(k_sp_count, cdiv(n_pt + 1, BA_THREADS), BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
         ctx->fixed_cam, P<long long>(ctx->sp_cnt));
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<long long>(ctx->sp_cnt), P<long long>(ctx->sp_off), n_pt + 1);
  CK(cudaMemcpyAsync(n_pairs_out, P<long long>(ctx->sp_off) + n_pt, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}
static int build_sparse_structure(ba_gpu_ctx *ctx) {
  const int n_pt = ctx->n_pt, n_cam = ctx->n_cam;
  cudaStream_t s = ctx->stream;
  typedef unsigned long long u64;
  RES(sp_cnt, ((size_t)n_pt + 2) * 8);
  RES(sp_off, ((size_t)n_pt + 2) * 8);
  LAUNCH(k_sp_count, cdiv(n_pt + 1, BA_THREADS), BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
         ctx->fixed_cam, P<long long>(ctx->sp_cnt));
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<long long>(ctx->sp_cnt), P<long long>(ctx->sp_off), n_pt + 1);
  long long n_pairs = 0;
  CK(cudaMemcpyAsync(&n_pairs, P<long long>(ctx->sp_off) + n_pt, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (n_pairs > 0x7fffffffLL) return fail(ctx, BA_ERR_UNSUPPORTED, "sparse Schur: %lld observation pairs (limit 2^31-1)", n_pairs);
  ctx->n_pairs = n_pairs;
  const size_t np8 = ((size_t)n_pairs + 1) * 8;
  RES(sp_keys, np8);
  RES(sp_vals, np8);
  RES(sp_keys2, np8);
  RES(sp_pairs, np8);
  LAUNCH(k_sp_emit, ctx->nblk_pt, BA_THREADS, 0, n_pt, n_cam, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->perm),
         ctx->fixed_cam, P<long long>(ctx->sp_off), P<u64>(ctx->sp_keys), P<u64>(ctx->sp_vals));
  int bits = 1;
  while (bits < 64 && ((u64)1 << bits) < (u64)n_cam * (u64)n_cam) ++bits;
  CUBCALL(cub::DeviceRadixSort::SortPairs, P<u64>(ctx->sp_keys), P<u64>(ctx->sp_keys2), P<u64>(ctx->sp_vals), P<u64>(ctx->sp_pairs),
          (int)n_pairs, 0, bits);
  RES(sp_pair_pt, ((size_t)n_pairs + 1) * 4);
  LAUNCH(k_sp_pair_points, (int)((n_pairs + BA_THREADS - 1) / BA_THREADS), BA_THREADS, 0, n_pairs, P<u64>(ctx->sp_pairs),
         P<int32_t>(ctx->pt_idx), P<int32_t>(ctx->sp_pair_pt));
  {
    int per_sm = 0;
    if (ctx->sps_simt)
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sp_schur_simt, BA_THREADS, 0));
    else
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sp_schur, BA_THREADS, BA_SPS_SMEM));
    ctx->sp_ctas_per_sm = std::max(1, per_sm);
  }
  RES(sp_ukeys, np8);
  RES(sp_ucnt, ((size_t)n_pairs + 2) * 4);
  RES(sp_nruns, 16);
  CUBCALL(cub::DeviceRunLengthEncode::Encode, P<u64>(ctx->sp_keys2), P<u64>(ctx->sp_ukeys), P<int32_t>(ctx->sp_ucnt),
          P<int32_t>(ctx->sp_nruns), (int)n_pairs);
  int32_t n_blk = 0;
  CK(cudaMemcpyAsync(&n_blk, ctx->sp_nruns.p, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (n_pairs == 0) n_blk = 0;
  // pair list pointers of the LOCAL blocks
  ctx->n_sblk_local = n_blk;
  RES(sb_ptr, ((size_t)n_blk + 2) * 4);
  CK(cudaMemsetAsync(P<int32_t>(ctx->sp_ucnt) + n_blk, 0, 4, s));
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<int32_t>(ctx->sp_ucnt), P<int32_t>(ctx->sb_ptr), n_blk + 1);
  RES(sp_lkeys, ((size_t)n_blk + 1) * 8);
  RES(sp_gid, ((size_t)n_blk + 1) * 4);
  CK(cudaMemcpyAsync(ctx->sp_lkeys.p, ctx->sp_ukeys.p, (size_t)n_blk * 8, cudaMemcpyDeviceToDevice, s));
  if (ctx->n_ranks > 1) {
    // point-sharded: every rank holds the blocks its own points touch.  The block structure must be the
    // same everywhere (S is all-reduced, PCG runs replicated): all-gather the key lists, sort, unique.
    double mx = (double)n_blk;
    int rcm = allreduce_host_scalar(ctx, &mx, true);
    if (rcm) return rcm;
    const size_t slot = (size_t)mx + 1, all = slot * ctx->n_ranks;
    if (all > 0x7fffffffull) return fail(ctx, BA_ERR_UNSUPPORTED, "sparse Schur: too many blocks to gather");
    RES(sp_gather, (all + 1) * 8);
    RES(sp_gsorted, (all + 1) * 8);
    CK(cudaMemsetAsync(P<u64>(ctx->sp_gather) + slot * ctx->rank, 0xff, slot * 8, s));
    CK(cudaMemcpyAsync(P<u64>(ctx->sp_gather) + slot * ctx->rank, ctx->sp_lkeys.p, (size_t)n_blk * 8, cudaMemcpyDeviceToDevice, s));
    ncclResult_t nr = g_nccl.AllGather(P<u64>(ctx->sp_gather) + slot * ctx->rank, ctx->sp_gather.p, slot, ncclUint64_, ctx->comm, s);
    if (nr != 0) return fail(ctx, BA_ERR_COMM, "ncclAllGather: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
    ctx->collectives++;
    CUBCALL(cub::DeviceRadixSort::SortKeys, P<u64>(ctx->sp_gather), P<u64>(ctx->sp_gsorted), (int)all, 0, 64);
    RES(sp_ukeys, (all + 1) * 8);
    RES(sp_ucnt, (all + 2) * 4);
    CUBCALL(cub::DeviceRunLengthEncode::Encode, P<u64>(ctx->sp_gsorted), P<u64>(ctx->sp_ukeys), P<int32_t>(ctx->sp_ucnt),
            P<int32_t>(ctx->sp_nruns), (int)all);
    int32_t n_all = 0;
    CK(cudaMemcpyAsync(&n_all, ctx->sp_nruns.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    n_blk = n_all - 1;  // the padding key ~0 sorts last (every rank pads at least one slot)
    LAUNCH(k_sp_lookup, cdiv(ctx->n_sblk_local, BA_THREADS), BA_THREADS, 0, ctx->n_sblk_local, P<u64>(ctx->sp_lkeys), n_blk,
           P<u64>(ctx->sp_ukeys), P<int32_t>(ctx->sp_gid));
  } else {
    LAUNCH(k_iota, cdiv(n_blk + 1, 256), 256, 0, n_blk + 1, P<int32_t>(ctx->sp_gid));
  }
  ctx->n_sblk = n_blk;
  const size_t nb = (size_t)n_blk;
  RES(sb_i, (nb + 1) * 4);
  RES(sb_j, (nb + 1) * 4);
  RES(row_ucnt, ((size_t)n_cam + 2) * 4);
  RES(row_tcnt, ((size_t)n_cam + 2) * 4);
  RES(row_ustart, ((size_t)n_cam + 2) * 4);
  RES(row_tstart, ((size_t)n_cam + 2) * 4);
  RES(sp_tkeys, (nb + 1) * 8);
  RES(sp_tkeys2, (nb + 1) * 8);
  RES(sp_tvals, (nb + 1) * 4);
  RES(sp_tvals2, (nb + 1) * 4);
  CK(cudaMemsetAsync(ctx->row_ucnt.p, 0, ((size_t)n_cam + 2) * 4, s));
  CK(cudaMemsetAsync(ctx->row_tcnt.p, 0, ((size_t)n_cam + 2) * 4, s));
  LAUNCH(k_sp_blocks, cdiv(n_blk, BA_THREADS), BA_THREADS, 0, n_blk, n_cam, P<u64>(ctx->sp_ukeys), P<int32_t>(ctx->sb_i),
         P<int32_t>(ctx->sb_j), P<int32_t>(ctx->row_ucnt), P<int32_t>(ctx->row_tcnt), P<u64>(ctx->sp_tkeys), P<int32_t>(ctx->sp_tvals));
  if (n_blk > 0)
    CUBCALL(cub::DeviceRadixSort::SortPairs, P<u64>(ctx->sp_tkeys), P<u64>(ctx->sp_tkeys2), P<int32_t>(ctx->sp_tvals),
            P<int32_t>(ctx->sp_tvals2), n_blk, 0, 64);
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<int32_t>(ctx->row_ucnt), P<int32_t>(ctx->row_ustart), n_cam + 1);
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<int32_t>(ctx->row_tcnt), P<int32_t>(ctx->row_tstart), n_cam + 1);
  int32_t n_t = 0;
  CK(cudaMemcpyAsync(&n_t, P<int32_t>(ctx->row_tstart) + n_cam, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  ctx->n_ent = n_blk + n_t;
  RES(ent_ptr, ((size_t)n_cam + 2) * 4);
  RES(ent, ((size_t)ctx->n_ent + 1) * 8);
  LAUNCH(k_sp_entries, cdiv(n_cam + 1, BA_THREADS), BA_THREADS, 0, n_cam, P<int32_t>(ctx->row_ustart), P<int32_t>(ctx->row_tstart),
         P<int32_t>(ctx->sp_tvals2), P<int32_t>(ctx->sb_i), P<int32_t>(ctx->sb_j), P<int32_t>(ctx->ent_ptr),
         P<int2>(ctx->ent));
  // PCG row order: rows sorted by decreasing entry count, dealt round-robin to the persistent warps
  RES(row_keys, ((size_t)n_cam + 1) * 8);
  RES(row_keys2, ((size_t)n_cam + 1) * 8);
  RES(row_ids, ((size_t)n_cam + 1) * 4);
  RES(row_order, ((size_t)n_cam + 1) * 4);
  LAUNCH(k_sp_row_keys, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->ent_ptr), P<u64>(ctx->row_keys), P<int32_t>(ctx->row_ids));
  CUBCALL(cub::DeviceRadixSort::SortPairs, P<u64>(ctx->row_keys), P<u64>(ctx->row_keys2), P<int32_t>(ctx->row_ids),
          P<int32_t>(ctx->row_order), n_cam, 0, 64);
  RES(sp_diag, ((size_t)n_cam + 1) * 4);
  LAUNCH(k_sp_diag_index, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->row_ustart), P<int32_t>(ctx->sb_j),
         P<int32_t>(ctx->sp_diag));
  RES(Sblk, (nb + 1) * 288);
  RES(ysp, ((size_t)n_cam + 1) * 48);
  RES(p2, ((size_t)n_cam + 1) * 48);
  RES(row_pq, ((size_t)n_cam + 1) * 8);
  RES(wb_rho, ((size_t)cdiv(n_cam, 32) + 1) * 8);
  RES(wb_Q, ((size_t)cdiv(n_cam, 32) + 1) * 8);
  RES(dsq, ((size_t)n_cam + 1) * 48);
  RES(pcg_bar, 128);
  CK(cudaMemsetAsync(ctx->pcg_bar.p, 0, 128, s));
  {
    int per_sm = 0;
    CK(cudaFuncSetAttribute(k_pcg_sparse_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize, BA_WARPS * BA_PCG_SMEM_PER_WARP));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg_sparse_persistent, BA_THREADS, (size_t)BA_WARPS * BA_PCG_SMEM_PER_WARP));
    ctx->pcg_grid = ctx->n_sm * std::min(per_sm, 2);
  }
  CK(cudaGetLastError());
  return 0;
}

// symbolic phase of the exact sparse Cholesky (host: ordering, elimination tree, supernodes, maps) from the block structure of
// the last build_sparse_structure(); uploads the integer tables and sizes the numeric buffers.  BA_ERR_UNSUPPORTED when a front
// cannot fit one SM's shared memory (co-visibility without a sequential structure): the caller keeps PCG then.
static int build_spchol(ba_gpu_ctx *ctx) {
  cudaStream_t s = ctx->stream;
  const int n_cam = ctx->n_cam, n_blk = ctx->n_sblk;
  std::vector<int32_t> bi((size_t)n_blk + 1), bj((size_t)n_blk + 1);
  if (n_blk > 0) {
    CK(cudaMemcpyAsync(bi.data(), ctx->sb_i.p, (size_t)n_blk * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(bj.data(), ctx->sb_j.p, (size_t)n_blk * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  const auto t0 = std::chrono::steady_clock::now();
  const int leaf = getenv("BA_SPCHOL_LEAF") ? std::max(2, atoi(getenv("BA_SPCHOL_LEAF"))) : 32;
  ctx->sym = spsym_build(n_cam, n_blk, bi.data(), bj.data(), leaf, SPC_CAP_BLOCKS, SPC_MAX_OWN);
  ctx->sym_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  const SpSymbolic &S = ctx->sym;
  if (S.error == 1)
    return fail(ctx, BA_ERR_UNSUPPORTED, "sparse Cholesky: a front of the reduced camera system does not fit shared memory "
                                         "(co-visibility too wide); use BA_SOLVER_SPARSE_SCHUR_PCG or BA_SOLVER_IMPLICIT_PCG");
  if (S.error) return fail(ctx, BA_ERR_STATE, "sparse Cholesky: inconsistent symbolic structure (%d)", S.error);
  if ((double)S.panel_blocks * 288.0 + (double)S.u_blocks * 288.0 > 64e9)
    return fail(ctx, BA_ERR_UNSUPPORTED, "sparse Cholesky: factor would need %.1f GB", ((double)S.panel_blocks + (double)S.u_blocks) * 288e-9);
  auto up = [&](Buf &b, const std::vector<int32_t> &v) -> int {
    int rc = buf_reserve(ctx, b, (v.size() + 1) * 4);
    if (rc) return rc;
    if (!v.empty()) CK(cudaMemcpyAsync(b.p, v.data(), v.size() * 4, cudaMemcpyHostToDevice, s));
    return 0;
  };
  // subtree-to-rank partition: one part per rank (BA_SPCHOL_REPLICATED=1 keeps every rank factorising the whole tree);
  // on one GPU BA_SPCHOL_PARTS=n runs the n parts one after the other (tests of the queues and of the exchange layout)
  int want_parts = ctx->n_ranks > 1 ? (getenv("BA_SPCHOL_REPLICATED") ? 1 : ctx->n_ranks)
                                    : (getenv("BA_SPCHOL_PARTS") ? std::min(BA_MAX_RANKS, std::max(1, atoi(getenv("BA_SPCHOL_PARTS")))) : 1);
  if (getenv("BA_SPCHOL_LEVELS") || ctx->sp_ref) want_parts = 1;  // (the REF-cost path is single-GPU: one part)
  const int R = ctx->spc_nrhs;
  const SpPartition part = spsym_partition(S, want_parts);
  ctx->spc_parts = part.parts;
  ctx->spc_dist = ctx->n_ranks > 1 && part.parts == ctx->n_ranks;
  // layout of spc_U (6x6 blocks): [update matrices of the subtree roots | right-hand-side updates of every node | the other
  // update matrices]: the first two pieces are what the ranks exchange, one contiguous all-reduce.  (R rows of 6 nb per node)
  const int64_t ru_blocks = ((int64_t)S.bord.size() * 6 * R + 35) / 36 + 1;
  {
    SpSymbolic &W = ctx->sym;
    auto usize = [&](int id) { const int64_t nb = W.node[(size_t)id * SPSYM_NODE_INTS + SPN_NB]; return nb * nb; };
    auto is_cut = [&](int id) {
      const int par = W.node[(size_t)id * SPSYM_NODE_INTS + SPN_PARENT];
      return part.parts > 1 && part.part[id] >= 0 && par >= 0 && part.part[par] < 0;
    };
    int64_t off = 0;
    auto place = [&](int id) {
      W.node[(size_t)id * SPSYM_NODE_INTS + SPN_U_LO] = (int32_t)(off & 0x7fffffff);
      W.node[(size_t)id * SPSYM_NODE_INTS + SPN_U_HI] = (int32_t)(off >> 31);
      off += usize(id);
    };
    for (int id = 0; id < W.n_nodes; ++id)
      if (is_cut(id)) place(id);
    ctx->spc_ru_off = (size_t)off * 36;
    off += ru_blocks;
    ctx->spc_xchg = (size_t)off * 36;
    for (int id = 0; id < W.n_nodes; ++id)
      if (!is_cut(id)) place(id);
  }
  int rc;
  ctx->spc_nx = 0;
  if (ctx->spc_dist) {
    // exchange set of S: block (i, j) is assembled by the node that owns the earlier-eliminated of its two cameras
    std::vector<int32_t> node_of((size_t)n_cam, 0), gid((size_t)ctx->n_sblk_local + 1);
    for (int id = 0; id < S.n_nodes; ++id)
      for (int k = 0; k < S.node[(size_t)id * SPSYM_NODE_INTS + SPN_M]; ++k) node_of[S.node[(size_t)id * SPSYM_NODE_INTS + SPN_K0] + k] = id;
    if (ctx->n_sblk_local > 0) CK(cudaMemcpyAsync(gid.data(), ctx->sp_gid.p, (size_t)ctx->n_sblk_local * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<double> mask((size_t)n_blk + 1, 0.0);
    for (int l = 0; l < ctx->n_sblk_local; ++l) {
      const int g = gid[l];
      if (g < 0 || g >= n_blk) return fail(ctx, BA_ERR_STATE, "sparse Cholesky: local block without a global id");
      if (part.part[node_of[std::min(S.pos[bi[g]], S.pos[bj[g]])]] != ctx->rank) mask[g] = 1.0;
    }
    RES(spc_xbuf, ((size_t)n_blk + 1) * 8);
    CK(cudaMemcpyAsync(ctx->spc_xbuf.p, mask.data(), ((size_t)n_blk + 1) * 8, cudaMemcpyHostToDevice, s));
    if ((rc = nccl_allreduce(ctx, P<double>(ctx->spc_xbuf), (size_t)n_blk + 1, true))) return rc;
    CK(cudaMemcpyAsync(mask.data(), ctx->spc_xbuf.p, ((size_t)n_blk + 1) * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<int32_t> xs;
    for (int g = 0; g < n_blk; ++g)
      if (mask[g] != 0.0) xs.push_back(g);
    ctx->spc_nx = (int)xs.size();
    if ((rc = up(ctx->spc_xidx, xs))) return rc;
    RES(spc_xbuf, ((size_t)std::max<size_t>(xs.size(), ((size_t)n_blk + 1) / 36 + 1) + 1) * 288);
  }
  if ((rc = up(ctx->spn_node, S.node)) || (rc = up(ctx->spn_bord, S.bord)) || (rc = up(ctx->spn_children, S.children)) ||
      (rc = up(ctx->spn_rel, S.rel)) || (rc = up(ctx->spn_inv, S.inv)) || (rc = up(ctx->spn_aent, S.aent)) ||
      (rc = up(ctx->spn_perm, S.perm)) || (rc = up(ctx->spn_levels, S.level_nodes)))
    return rc;
  RES(spc_panel, ((size_t)S.panel_blocks + 1) * 288);
  RES(spc_U, ((size_t)S.u_blocks + (size_t)ru_blocks + 1) * 288);
  RES(spc_z, ((size_t)n_cam + 1) * 48);
  RES(spc_linv, ((size_t)n_cam + 1) * 288);
  RES(spc_ypos, ((size_t)n_cam + 1) * 48);
  RES(spc_prof, 128);
  CK(cudaMemsetAsync(ctx->spc_prof.p, 0, 128, s));
  RES(dsq, ((size_t)n_cam + 1) * 48);
  size_t sf = 0, ss = 0, su = 0;
  for (int id = 0; id < S.n_nodes; ++id) {
    const int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
    sf = std::max(sf, spc_factor_smem(N[SPN_M], N[SPN_NB], R));
    ss = std::max(ss, spc_solve_smem(N[SPN_M], N[SPN_NB]));
    su = std::max(su, spc_update_smem(N[SPN_M], N[SPN_NB], R));
  }
  // (at the front capacity, SPC_CAP_BLOCKS = 770 and SPC_MAX_OWN = 24, the five-row factor front needs 228,160 bytes)
  if (sf > 227 * 1024 || ss > 227 * 1024 || su > 227 * 1024)
    return fail(ctx, BA_ERR_STATE, "sparse Cholesky: front exceeds shared memory (%zu / %zu / %zu bytes)", sf, ss, su);
  ctx->spc_smem_factor = sf;
  ctx->spc_smem_solve = ss;
  ctx->spc_smem_update = su;
  if (R > 1) {
    CK(cudaFuncSetAttribute(k_spchol_factor<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sf));
    CK(cudaFuncSetAttribute(k_spchol_update<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)su));
  } else {
    CK(cudaFuncSetAttribute(k_spchol_factor<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sf));
    CK(cudaFuncSetAttribute(k_spchol_update<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)su));
  }
  CK(cudaFuncSetAttribute(k_spchol_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss));
  // work queues of the persistent tree kernel.  Phase A (one queue per part): per level (bottom-up) the factor items of the
  // part's nodes, then their update tiles -- more tiles per node where the part has few nodes on a level.  Phase B: the same
  // for the top part, then the backward substitution level by level top-down (top part first, then the subtrees this GPU
  // holds).  One part: phase A is the whole factorisation and the substitution follows in the same queue (one launch).
  {
    const int P_ = part.parts;
    // -2: this GPU holds every part.  BA_SPCHOL_ONLY_PART=p on one GPU: the queues rank p of a distributed run would execute
    // (the other parts' subtree roots count as done, their update matrices are whatever the buffer holds): timing experiments
    const int only = (ctx->n_ranks == 1 && P_ > 1 && getenv("BA_SPCHOL_ONLY_PART")) ? std::min(P_ - 1, std::max(0, atoi(getenv("BA_SPCHOL_ONLY_PART")))) : -1;
    const int me = ctx->spc_dist ? ctx->rank : (only >= 0 ? only : -2);
    auto N_ = [&](int id, int f) { return S.node[(size_t)id * SPSYM_NODE_INTS + f]; };
    std::vector<int32_t> tiles((size_t)S.n_nodes, 0), q, cnt_init((size_t)3 * S.n_nodes + 16, 0), topcams;
    auto push_factor_levels = [&](int which) {
      for (int l = 0; l < S.n_levels; ++l) {
        int nodes = 0;
        for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) nodes += part.part[S.level_nodes[e]] == which;
        if (!nodes) continue;
        const int t_lvl = std::max(1, std::min(8, ctx->n_sm / nodes));
        for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
          const int id = S.level_nodes[e];
          if (part.part[id] != which) continue;
          tiles[id] = N_(id, SPN_NB) > 0 ? t_lvl : 0;
          q.push_back(id);
          q.push_back(-1);
        }
        for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
          const int id = S.level_nodes[e];
          if (part.part[id] != which) continue;
          for (int t = 0; t < tiles[id]; ++t) {
            q.push_back(id);
            q.push_back(t);
          }
        }
      }
    };
    auto push_solve_levels = [&](bool top_part) {
      for (int l = S.n_levels - 1; l >= 0; --l)
        for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
          const int id = S.level_nodes[e], pr = part.part[id];
          if (top_part ? pr >= 0 : (pr < 0 || (me != -2 && pr != me))) continue;
          q.push_back(id);
          q.push_back(-2);
        }
    };
    for (int p = 0; p < P_; ++p) {
      ctx->spc_qA[p] = (int)(q.size() / 2);
      if (me == -2 || p == me) push_factor_levels(p);
      ctx->spc_qA[p + 1] = (int)(q.size() / 2);
    }
    ctx->spc_qB = (int)(q.size() / 2);
    if (P_ > 1) {
      push_factor_levels(-1);
      push_solve_levels(true);
    }
    push_solve_levels(false);
    ctx->spc_qB_n = (int)(q.size() / 2) - ctx->spc_qB;
    ctx->spc_n_items = (int)(q.size() / 2);
    // counters before a solve: zero, except "all update tiles done" for the subtree roots other ranks factorise (their
    // update matrices arrive with the exchange)
    for (int id = 0; id < S.n_nodes; ++id) {
      if (part.part[id] < 0)
        for (int k = 0; k < N_(id, SPN_M); ++k) topcams.push_back(S.perm[N_(id, SPN_K0) + k]);
      else if (me != -2 && part.part[id] != me)
        cnt_init[16 + (size_t)S.n_nodes + id] = 1 << 20;
    }
    ctx->spc_n_topcams = (int)topcams.size();
    if ((rc = up(ctx->spc_queue, q)) || (rc = up(ctx->spc_tiles, tiles)) || (rc = up(ctx->spc_cnt_init, cnt_init)) ||
        (rc = up(ctx->spc_topcams, topcams)))
      return rc;
    RES(spc_cnt, ((size_t)3 * S.n_nodes + 16) * 4);
    const size_t st_ = std::max(std::max(sf, ss), su);
    if (R > 1)
      CK(cudaFuncSetAttribute(k_spchol_tree<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_));
    else
      CK(cudaFuncSetAttribute(k_spchol_tree<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_));
    ctx->spc_tree = getenv("BA_SPCHOL_LEVELS") == nullptr;
    if (getenv("BA_SPCHOL_DEBUG"))
      fprintf(stderr, "[spchol] rank %d: %d parts%s, top %d nodes / %d cameras (%.1f %% of the work), heaviest part %.1f %%, "
              "exchange %.2f MB, items A %d B %d\n", ctx->rank, P_, ctx->spc_dist ? " (distributed)" : "",
              (int)std::count(part.part.begin(), part.part.end(), -1), ctx->spc_n_topcams, 100.0 * part.top / std::max(1.0, part.total),
              100.0 * part.heaviest / std::max(1.0, part.total), ctx->spc_xchg * 8e-6, ctx->spc_qB, ctx->spc_qB_n);
  }
  CK(cudaStreamSynchronize(s));  // host vectors of this call die here
  ctx->spchol = true;
  return 0;
}

// exchange buffers of the row-sharded PCG: one cudaMalloc per rank, handles all-gathered through NCCL,
// peers mapped with cudaIpcOpenMemHandle (NVLink peer access)
static int setup_dist_pcg(ba_gpu_ctx *ctx) {
  const int n_cam = ctx->n_cam, n_wb = cdiv(n_cam, 32), N = ctx->n_ranks;
  cudaStream_t s = ctx->stream;
  ctx->dist_pcg = false;
  if (N > BA_MAX_RANKS) return 0;
  // layout (16-byte slots): q[2][6n] pq[2][n] slice[2][n_slices] | epoch (u64) abort (int)
  const size_t n6 = (size_t)6 * n_cam, n_slices = (size_t)cdiv(n_cam, BA_PQ_SLICE);
  const size_t n_slots = 2 * n6 + 2 * (size_t)n_cam + 2 * n_slices;
  const size_t bytes = n_slots * sizeof(LLSlot) + 64;
  (void)n_wb;
  if (ctx->xch_ncam != n_cam || !ctx->xch) {
    CK(cudaStreamSynchronize(s));
    for (int k = 0; k < 8; ++k) {
      if (ctx->xch_peer[k] && k != ctx->rank) cudaIpcCloseMemHandle(ctx->xch_peer[k]);
      ctx->xch_peer[k] = nullptr;
    }
    {
      // every rank has closed its mappings of the peers' buffers (above) before any rank frees its exported one: the
      // camera count is the same on all ranks, so all of them pass through here in the same upload
      double tok = 1.0;
      int rcb = allreduce_host_scalar(ctx, &tok, false);
      if (rcb) return rcb;
    }
    if (ctx->xch) cudaFree(ctx->xch);
    ctx->xch = nullptr;
    CK(cudaMalloc(&ctx->xch, bytes));
    CK(cudaMemset(ctx->xch, 0, bytes));
    ctx->xch_cap = bytes;
    ctx->xch_ncam = n_cam;
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, ctx->xch));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    RES(ipc_stage, (size_t)64 * (N + 1));
    CK(cudaMemcpyAsync(P<char>(ctx->ipc_stage) + 64 * ctx->rank, &h, 64, cudaMemcpyHostToDevice, s));
    ncclResult_t nr = g_nccl.AllGather(P<char>(ctx->ipc_stage) + 64 * ctx->rank, ctx->ipc_stage.p, 8, ncclUint64_, ctx->comm, s);
    if (nr != 0) return fail(ctx, BA_ERR_COMM, "ncclAllGather(ipc handles): %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
    ctx->collectives++;
    std::vector<cudaIpcMemHandle_t> all(N);
    CK(cudaMemcpyAsync(all.data(), ctx->ipc_stage.p, (size_t)64 * N, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int k = 0; k < N; ++k) {
      if (k == ctx->rank) {
        ctx->xch_peer[k] = ctx->xch;
        continue;
      }
      cudaError_t e = cudaIpcOpenMemHandle(&ctx->xch_peer[k], all[k], cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        // no peer access between these GPUs: the replicated PCG is used instead (same on every rank? the
        // decision is all-reduced below)
        ctx->xch_peer[k] = nullptr;
        cudaGetLastError();
      }
    }
  }
  double ok = 1.0;
  for (int k = 0; k < N; ++k)
    if (!ctx->xch_peer[k]) ok = 0.0;
  ok = -ok;  // min over ranks through the max reduction
  int rc = allreduce_host_scalar(ctx, &ok, true);
  if (rc) return rc;
  if (ok != -1.0) return 0;
  PcgFan &f = ctx->fan;
  memset(&f, 0, sizeof(f));
  f.n_ranks = N;
  f.rank = ctx->rank;
  for (int k = 0; k < N; ++k) {
    LLSlot *base = reinterpret_cast<LLSlot *>(ctx->xch_peer[k]);
    f.q[k] = base;
    f.pq[k] = base + 2 * n6;
  }
  {
    LLSlot *base = reinterpret_cast<LLSlot *>(ctx->xch);
    f.slice = base + 2 * n6 + 2 * (size_t)n_cam;
    f.epoch = reinterpret_cast<unsigned long long *>(base + n_slots);
    f.abort_flag = reinterpret_cast<int *>(f.epoch + 1);
  }
  // own rows, in the global order of decreasing entry count
  RES(row_flag, ((size_t)n_cam + 2) * 4);
  RES(row_pos, ((size_t)n_cam + 2) * 4);
  RES(my_rows, ((size_t)n_cam + 2) * 4);
  CK(cudaMemsetAsync(ctx->row_flag.p, 0, ((size_t)n_cam + 2) * 4, s));
  LAUNCH(k_dist_flag_rows, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->row_order), ctx->rank, N, P<int32_t>(ctx->row_flag));
  CUBCALL(cub::DeviceScan::ExclusiveSum, P<int32_t>(ctx->row_flag), P<int32_t>(ctx->row_pos), n_cam + 1);
  LAUNCH(k_dist_pick_rows, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->row_order), P<int32_t>(ctx->row_flag),
         P<int32_t>(ctx->row_pos), P<int32_t>(ctx->my_rows));
  int32_t n_my = 0;
  CK(cudaMemcpyAsync(&n_my, P<int32_t>(ctx->row_pos) + n_cam, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  ctx->n_my_rows = n_my;
  {
    int per_sm = 0;
    CK(cudaFuncSetAttribute(k_pcg_sparse_dist, cudaFuncAttributeMaxDynamicSharedMemorySize, BA_WARPS * BA_PCG_SMEM_PER_WARP));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg_sparse_dist, BA_THREADS, (size_t)BA_WARPS * BA_PCG_SMEM_PER_WARP));
    ctx->dist_grid = per_sm > 0 ? ctx->n_sm : 0;
  }
  ctx->dist_pcg = ctx->dist_grid > 0;
  return 0;
}

// BA_UPLOAD_PROF=1: host wall-clock stamps of the upload phases on stderr (measurement aid)
struct UploadProf {
  bool on = getenv("BA_UPLOAD_PROF") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  char line[512];
  int len = 0;
  void stamp(const char *what) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    len += snprintf(line + len, sizeof(line) - len, " %s %.0f us |", what, std::chrono::duration<double, std::micro>(n - t).count());
    t = n;
  }
  void flush() {
    if (on) fprintf(stderr, "[BA_UPLOAD_PROF]%s\n", line);
  }
};

extern "C" int ba_gpu_upload(ba_gpu_ctx *ctx, int32_t n_cam, const double *pose7, int32_t fixed_cam, int32_t n_pt,
                             const double *pt3, int32_t n_obs, const int32_t *cam_idx, const int32_t *pt_idx,
                             const double *uv2, const double *depth, const double intr4[4], const double intr_prior4[4]) {
  if (!ctx) return BA_ERR_INVALID;
  ctx->pdl = false;
  UploadProf prof;
  ctx->uploaded = false;
  ctx->lm_graph_stale = true;
  ctx->linearized = false;
  ctx->cov_ready = false;
  const ba_gpu_options &o = ctx->opt;
  if (n_cam <= 0 || n_pt < 0 || n_obs < 0 || !pose7 || !intr4 || (n_pt > 0 && !pt3) ||
      (n_obs > 0 && (!cam_idx || !pt_idx || !uv2)))
    return fail(ctx, BA_ERR_INVALID, "bad sizes or null buffers");
  if (fixed_cam >= n_cam) return fail(ctx, BA_ERR_INVALID, "fixed_cam out of range");
  if (o.use_depth_prior && n_obs > 0 && !depth) return fail(ctx, BA_ERR_INVALID, "depth required when use_depth_prior");
  if (o.optimize_intrinsics && !intr_prior4) return fail(ctx, BA_ERR_INVALID, "intr_prior4 required when optimize_intrinsics");
  CK(cudaSetDevice(ctx->device));
  ctx->n_cam = n_cam;
  ctx->n_pt = n_pt;
  ctx->n_obs = n_obs;
  ctx->fixed_cam = fixed_cam < 0 ? -1 : fixed_cam;
  ctx->n_free = n_cam - (fixed_cam >= 0 ? 1 : 0);
  ctx->depth = o.use_depth_prior ? 1 : 0;
  ctx->nk = o.optimize_intrinsics ? 4 : 0;
  ctx->n_red = 6 * ctx->n_free + ctx->nk;
  int solver = o.solver;
  // the exact sparse Cholesky shares the block-sparse S machinery of the PCG variant; ctx->spchol switches the linear solve
  bool want_chol = solver == BA_SOLVER_SPARSE_SCHUR_CHOLESKY;
  if (want_chol) solver = BA_SOLVER_SPARSE_SCHUR_PCG;
  ctx->spchol = false;
  // depth prior and / or free intrinsics through the sparse Cholesky: when asked for, and under AUTO when free intrinsics
  // take the problem past the dense explicit limit.  It keeps the explicit solver's linearisation (planes store, W / WV) and
  // replaces the dense S by the block-sparse one; the four intrinsics columns become a border of the tree's solve.
  const bool sp_ref = (o.use_depth_prior || o.optimize_intrinsics) &&
                      (want_chol || (solver == BA_SOLVER_AUTO && ctx->nk && ctx->n_red > BA_EXPLICIT_MAX_DIM && ctx->n_ranks == 1));
  ctx->sp_ref = sp_ref;
  // right-hand-side rows of the tree, decided by THIS upload (a context reused after set_options must not keep the border of an
  // earlier REF problem: the NS path is the one-row tree)
  ctx->spc_nrhs = sp_ref && ctx->nk ? 5 : 1;
  if (sp_ref) {
    if (ctx->n_ranks > 1)
      return fail(ctx, BA_ERR_UNSUPPORTED, "the sparse Cholesky with depth prior / free intrinsics is single-GPU");
    if (o.jacobian_store == BA_JAC_FACTORED || o.jacobian_store == BA_JAC_TILED)
      return fail(ctx, BA_ERR_UNSUPPORTED, "the sparse Cholesky with depth prior / free intrinsics reads the planes Jacobian store");
    solver = BA_SOLVER_EXPLICIT_CHOLESKY;
    want_chol = false;
  }
  if (solver == BA_SOLVER_AUTO)
    solver = (ctx->n_red <= o.explicit_max_dim || ctx->nk) ? BA_SOLVER_EXPLICIT_CHOLESKY : BA_SOLVER_IMPLICIT_PCG;
  if ((solver == BA_SOLVER_IMPLICIT_PCG || solver == BA_SOLVER_SPARSE_SCHUR_PCG) && ctx->nk)
    return fail(ctx, BA_ERR_UNSUPPORTED, "optimize_intrinsics needs the explicit solver (as ITERATIVE_SCHUR needs points only)");
  if (solver == BA_SOLVER_SPARSE_SCHUR_PCG && o.use_depth_prior)
    return fail(ctx, BA_ERR_UNSUPPORTED, "the block-sparse Schur solver needs NS mode (no depth prior, fixed intrinsics)");
  if (solver == BA_SOLVER_EXPLICIT_CHOLESKY && !sp_ref && ctx->n_red > BA_EXPLICIT_MAX_DIM)
    return fail(ctx, BA_ERR_UNSUPPORTED, "dense explicit Cholesky supports reduced dimension <= %d (got %d)", BA_EXPLICIT_MAX_DIM,
                ctx->n_red);
  if (solver == BA_SOLVER_EXPLICIT_CHOLESKY && ctx->n_ranks > 1)
    return fail(ctx, BA_ERR_UNSUPPORTED, "the explicit solver is single-GPU (windowed problems stay on one GPU)");
  ctx->solver = solver;
  // AUTO on a large NS-mode problem, single GPU: block-sparse explicit S if the co-visibility
  // is sparse enough (decided after the index build, from the pair count), else implicit
  const bool auto_large = o.solver == BA_SOLVER_AUTO && solver == BA_SOLVER_IMPLICIT_PCG && !o.use_depth_prior &&
                          o.jacobian_store != BA_JAC_PLANES;
  bool sparse = solver == BA_SOLVER_SPARSE_SCHUR_PCG;
  const bool can_fact = ((solver == BA_SOLVER_IMPLICIT_PCG || sparse) && !o.use_depth_prior && !o.optimize_intrinsics);
  if (sparse && o.jacobian_store == BA_JAC_PLANES)
    return fail(ctx, BA_ERR_UNSUPPORTED, "the block-sparse Schur solver rebuilds its blocks from the factored store");
  if (o.jacobian_store == BA_JAC_FACTORED && !can_fact)
    return fail(ctx, BA_ERR_UNSUPPORTED, "the factored Jacobian store needs NS mode (no depth prior, fixed intrinsics) + implicit PCG");
  ctx->fact = can_fact && o.jacobian_store != BA_JAC_PLANES;
  ctx->planes_ready = false;

  const int64_t N = o.n_obs_total > 0 ? o.n_obs_total : (int64_t)n_obs;
  // src/OptimizationUtils.cpp:280, 290: weights 1/N and WEIGHT_UNPR/N; residual = sqrt(weight) * ...
  ctx->cp.sw_repr = sqrt(1.0 / (double)(N > 0 ? N : 1));
  ctx->cp.sw_unpr = sqrt(o.WEIGHT_UNPR / (double)(N > 0 ? N : 1));
  ctx->cp.hub_repr = o.HUB_P_REPR;
  ctx->cp.hub_unpr = o.HUB_P_UNPR;
  ctx->cp.sw_intr = sqrt(o.WEIGHT_INTRINSICS);
  ctx->cp.fixed_cam = ctx->fixed_cam;
  ctx->cp.pad = 0;
  LmOptions &lo = ctx->lo;
  lo.function_tolerance = o.function_tolerance;
  lo.gradient_tolerance = o.gradient_tolerance;
  lo.parameter_tolerance = o.parameter_tolerance;
  lo.max_radius = o.max_trust_region_radius;
  lo.min_radius = o.min_trust_region_radius;
  lo.min_relative_decrease = o.min_relative_decrease;
  lo.min_lm_diagonal = o.min_lm_diagonal;
  lo.max_lm_diagonal = o.max_lm_diagonal;
  lo.eta = o.eta;
  lo.max_num_iterations = o.max_num_iterations;
  lo.max_invalid = o.max_num_consecutive_invalid_steps;
  lo.max_pcg = o.max_linear_solver_iterations;
  lo.min_pcg = o.min_linear_solver_iterations;
  lo.reset_period = o.residual_reset_period;
  lo.trace_cap = o.max_num_iterations + 2;

  const size_t nc = (size_t)n_cam, np = (size_t)n_pt, no = (size_t)n_obs;
  const int n_ent = n_cam + n_pt + 1;
  ctx->nblk_obs = cdiv(n_obs, BA_THREADS);
  ctx->nblk_ent = cdiv(n_ent, BA_THREADS);
  ctx->nblk_cam = cdiv(n_cam, BA_THREADS);
  ctx->nblk_pt = cdiv(n_pt, BA_THREADS);
  ctx->n_tiles = cdiv(n_pt, BA_TILE_PTS);
  // planes-store point-major kernels: shorter tiles while the problem has fewer tiles than twice the SM count
  ctx->pl_tile_pts = BA_TILE_PTS;
  while (ctx->pl_tile_pts > 8 && cdiv(n_pt, ctx->pl_tile_pts) < 2 * ctx->n_sm) ctx->pl_tile_pts >>= 1;
  ctx->pl_tiles = cdiv(n_pt, ctx->pl_tile_pts);

  RES(pose, nc * 56);
  RES(pose_c, nc * 56);
  RES(pt, np * 24);
  RES(pt_c, np * 24);
  RES(intr, 32);
  RES(intr_c, 32);
  RES(intr_prior, 32);
  RES(cam_idx, no * 4);
  RES(pt_idx, no * 4);
  RES(uv, no * 16);
  RES(depthv, no * 8);
  RES(perm, no * 4);
  RES(pt_rowptr, (np + 1) * 4);
  RES(cam_rowptr, (nc + 1) * 4);
  RES(pt_cnt, (np + 1) * 4);
  RES(cam_cnt, (nc + 1) * 4);
  RES(cursor, (np + 1) * 4);
  RES(err_flag, 16);
  RES(pm_cam, no * 4);
  RES(pm_pt, no * 4);
  RES(pm_uv, no * 16);
  RES(pm_depth, no * 8);
  RES(item_ptr, (nc + 1) * 4);
  RES(item_cnt, (nc + 1) * 4);
  RES(cam_slot, nc * 4);
  const size_t n_pad = (no + 31) / 32 * 32 + 32;
  if (!ctx->fact) {
    int rcp = ensure_planes(ctx);
    if (rcp) return rcp;
  } else {
    RES(fcm, n_pad * 48);
    RES(fpm, n_pad * 48);
    auto setf = [&](FPlanes &F, double *base) {
      F.r = reinterpret_cast<double2 *>(base);
      F.g0 = reinterpret_cast<double2 *>(base + 2 * n_pad);
      F.g1 = reinterpret_cast<double2 *>(base + 4 * n_pad);
    };
    setf(ctx->Fc_, P<double>(ctx->fcm));
    setf(ctx->Fp_, P<double>(ctx->fpm));
    RES(geo, nc * BA_CAMREC * 8);
    RES(camx, nc * BA_CAMREC * 8);
    RES(Vs, np * 48);
    RES(ts, (np + 1) * 32);
    RES(tgs, (np + 1) * 32);
    RES(ys, (np + 1) * 32);
    RES(tile_lo, (size_t)(ctx->n_tiles + 1) * 4);
    RES(tile_span, (size_t)(ctx->n_tiles + 1) * 4);
  }
  RES(sc, nc * 48);
  RES(sp, np * 24);
  RES(sk, 32);
  RES(one_c, nc * 48);
  RES(one_p, np * 24);
  RES(one_k, 32);
  RES(dc, nc * 48);
  RES(dp, np * 24);
  RES(dk, 32);
  RES(gc, nc * 48);
  RES(gp, np * 24);
  RES(gk, 32);
  RES(U, nc * 288);
  RES(Uck, nc * 192);
  RES(Ukk, 128);
  RES(V, np * 48);
  RES(Vinv, np * 48);
  RES(Wk, ctx->nk ? np * 96 : 16);
  RES(tg, np * 24);
  RES(t, np * 24);
  RES(yc, nc * 48 + 16);  // (+ one slot: failure flag riding on the all-reduce of the distributed sparse Cholesky)
  RES(yp, np * 24);
  RES(yk, 32);
  RES(rk, 32);
  RES(Jkk, 32);
  RES(b, nc * 48);
  RES(x, nc * 48);
  RES(r, nc * 48);
  RES(z, nc * 48);
  RES(p, nc * 48);
  RES(q, nc * 48);
  RES(Minv, nc * 288);
  RES(pc_lin, (size_t)ctx->nblk_obs * 8);
  RES(pc_cand, (size_t)ctx->nblk_obs * 8);
  RES(pc_mcc, (size_t)ctx->nblk_obs * 8);
  RES(pe_gmax, (size_t)ctx->nblk_ent * 8);
  RES(pe_xn, (size_t)ctx->nblk_ent * 8);
  RES(pe_step, (size_t)ctx->nblk_ent * 8);
  RES(pcam_rho, (size_t)ctx->nblk_cam * 8);
  RES(pcam_bb, (size_t)ctx->nblk_cam * 8);
  RES(pcam_pq, (size_t)ctx->nblk_cam * 8);
  RES(pcam_Q, (size_t)ctx->nblk_cam * 8);
  RES(part_kk, (size_t)(ctx->nblk_pt + 1) * 14 * 8);
  RES(red_blk, nc * 27 * 8);
  RES(red6, nc * 48);
  RES(red21, nc * 21 * 8);
  RES(scal, 64 * 8);
  RES(ident, (nc + 1) * 4);
  RES(st, sizeof(LmState));
  RES(trace, (size_t)lo.trace_cap * sizeof(BaIterRec));

  prof.stamp("reserve");
  cudaStream_t s = ctx->stream;
  // (cudaMemcpyDefault: the arrays are host buffers for a C-ABI caller and device buffers when the device-resident store
  // assembled the window, ba_store_window_solve)
  CK(cudaMemcpyAsync(ctx->pose.p, pose7, nc * 56, cudaMemcpyDefault, s));
  if (np) CK(cudaMemcpyAsync(ctx->pt.p, pt3, np * 24, cudaMemcpyDefault, s));
  CK(cudaMemcpyAsync(ctx->intr.p, intr4, 32, cudaMemcpyDefault, s));
  CK(cudaMemcpyAsync(ctx->intr_prior.p, intr_prior4 ? intr_prior4 : intr4, 32, cudaMemcpyDefault, s));
  if (no) {
    CK(cudaMemcpyAsync(ctx->cam_idx.p, cam_idx, no * 4, cudaMemcpyDefault, s));
    CK(cudaMemcpyAsync(ctx->pt_idx.p, pt_idx, no * 4, cudaMemcpyDefault, s));
    CK(cudaMemcpyAsync(ctx->uv.p, uv2, no * 16, cudaMemcpyDefault, s));
    if (depth) CK(cudaMemcpyAsync(ctx->depthv.p, depth, no * 8, cudaMemcpyDefault, s));
  }
  prof.stamp("h2d");
  // ---- device-built indices
  CK(cudaMemsetAsync(ctx->pt_cnt.p, 0, (np + 1) * 4, s));
  CK(cudaMemsetAsync(ctx->cam_cnt.p, 0, (nc + 1) * 4, s));
  CK(cudaMemsetAsync(ctx->cursor.p, 0, (np + 1) * 4, s));
  CK(cudaMemsetAsync(ctx->err_flag.p, 0, 16, s));
  CK(cudaMemsetAsync(ctx->cam_rowptr.p, 0, (nc + 1) * 4, s));  // (no observations at all: every pointer is 0)
  LAUNCH(k_index_count, ctx->nblk_obs, BA_THREADS, 0, n_obs, n_cam, n_pt, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
         P<int32_t>(ctx->pt_cnt), P<int32_t>(ctx->cam_rowptr), P<int32_t>(ctx->err_flag));
  if (n_pt > 65536) {
    // (pt_cnt has n_pt + 1 entries, the last one zero: the scan's last output is the total; library scan, setup only --
    // the single-CTA scan below took 1.6 ms for 2 M points)
    CUBCALL(cub::DeviceScan::ExclusiveSum, P<int32_t>(ctx->pt_cnt), P<int32_t>(ctx->pt_rowptr), n_pt + 1);
  } else {
    LAUNCH(k_exclusive_scan, 1, 1024, 0, n_pt, P<int32_t>(ctx->pt_cnt), P<int32_t>(ctx->pt_rowptr));
  }
  LAUNCH(k_index_fill, ctx->nblk_obs, BA_THREADS, 0, n_obs, n_cam, n_pt, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
         P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->cursor), P<int32_t>(ctx->perm));
  LAUNCH(k_index_sort, ctx->nblk_pt, BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->perm));
  LAUNCH(k_index_gather, ctx->nblk_pt, BA_THREADS, 0, n_pt, n_obs, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->perm),
         P<int32_t>(ctx->cam_idx), P<double2>(ctx->uv), depth ? P<double>(ctx->depthv) : (double *)nullptr,
         P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->pm_pt), P<double2>(ctx->pm_uv), P<double>(ctx->pm_depth));
  // work-item length: 256 observations for streaming-sized problems, down to one observation per lane when the whole
  // problem has fewer items than twice the SM count (windows)
  int item_obs = BA_ITEM_OBS;
  while (item_obs > 32 && cdiv(n_obs, item_obs) < 2 * ctx->n_sm) item_obs >>= 1;
  LAUNCH(k_item_count, ctx->nblk_cam, BA_THREADS, 0, n_cam, item_obs, P<int32_t>(ctx->cam_rowptr), P<int32_t>(ctx->item_cnt));
  LAUNCH(k_exclusive_scan, 1, 1024, 0, n_cam, P<int32_t>(ctx->item_cnt), P<int32_t>(ctx->item_ptr));
  LAUNCH(k_slots, ctx->nblk_cam, BA_THREADS, 0, n_cam, ctx->fixed_cam, P<int32_t>(ctx->cam_slot));
  LAUNCH(k_iota, cdiv(n_cam + 1, 256), 256, 0, n_cam + 1, P<int32_t>(ctx->ident));
  int32_t h_items = 0, h_err = 0;
  CK(cudaMemcpyAsync(&h_items, P<int32_t>(ctx->item_ptr) + n_cam, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&h_err, ctx->err_flag.p, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (h_err) return fail(ctx, BA_ERR_INVALID, "observation indices out of range or cam_idx not non-decreasing");
  prof.stamp("index build + sync");
  ctx->n_items = h_items;
  ctx->nblk_item = cdiv(h_items * 32, BA_THREADS);
  RES(items, (size_t)(h_items + 1) * sizeof(BaItem));
  LAUNCH(k_item_fill, ctx->nblk_cam, BA_THREADS, 0, n_cam, item_obs, P<int32_t>(ctx->cam_rowptr), P<int32_t>(ctx->item_ptr),
         P<BaItem>(ctx->items));
  if (ctx->fact) {
    // camera span of every point tile -> shared-memory staging of pass 1
    CK(cudaMemsetAsync(ctx->err_flag.p, 0, 16, s));
    LAUNCH(k_tile_cam_range, ctx->n_tiles, BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
           P<int32_t>(ctx->tile_lo), P<int32_t>(ctx->tile_span), P<int32_t>(ctx->err_flag));
    int32_t h_span = 0;
    CK(cudaMemcpyAsync(&h_span, ctx->err_flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    ctx->staged = h_span <= BA_STAGE_CAMS;
  }
  ctx->tiled = false;
  if (auto_large) {
    long long n_pairs = 0;
    int rcs = sparse_count_pairs(ctx, &n_pairs);
    if (rcs) return rcs;
    double tot_pairs = (double)n_pairs, tot_obs = (double)n_obs, max_pairs = (double)n_pairs;  // same decision on every rank
    if ((rcs = allreduce_host_scalar(ctx, &tot_pairs, false)) || (rcs = allreduce_host_scalar(ctx, &tot_obs, false)) ||
        (rcs = allreduce_host_scalar(ctx, &max_pairs, true)))
      return rcs;
    if (tot_pairs <= (double)o.sparse_max_pairs_per_obs * tot_obs && max_pairs <= 2147483647.0) {
      sparse = true;
      want_chol = getenv("BA_AUTO_PCG") == nullptr;  // AUTO: exact factorisation (the reference's SPARSE_SCHUR) when its fronts fit
      ctx->solver = BA_SOLVER_SPARSE_SCHUR_PCG;
    }
  }
  if (sparse) {
    prof.stamp("to sparse");
    int rcs = build_sparse_structure(ctx);
    if (rcs) return rcs;
    prof.stamp("sparse structure");
    if (want_chol) {
      rcs = build_spchol(ctx);
      if (rcs == BA_ERR_UNSUPPORTED && o.solver == BA_SOLVER_AUTO) rcs = 0;  // falls back to PCG on the same S
      if (rcs) return rcs;
      prof.stamp("symbolic + tables");
    }
    ctx->dist_pcg = false;
    if (!ctx->spchol && ctx->n_ranks > 1 && o.persistent_pcg == 1 && (rcs = setup_dist_pcg(ctx))) return rcs;
  }
  if (sp_ref) {
    prof.stamp("to sparse");
    int rcs = build_sparse_structure(ctx);
    if (!rcs) rcs = build_spchol(ctx);
    if (rcs == BA_ERR_UNSUPPORTED && o.solver == BA_SOLVER_AUTO) {
      const std::string why = ctx->err;
      return fail(ctx, BA_ERR_UNSUPPORTED, "dense explicit Cholesky supports reduced dimension <= %d (got %d), and the sparse "
                  "Cholesky cannot take it: %s", BA_EXPLICIT_MAX_DIM, ctx->n_red, why.c_str());
    }
    if (rcs) return rcs;
    prof.stamp("sparse structure + symbolic");
  }
  if (ctx->fact && !sparse && o.jacobian_store != BA_JAC_FACTORED && ctx->n_tiles > 0) {
    // tile-fused product: tile metadata, then (if the locality bounds hold) the tile-camera-major store
    RES(tmeta, (size_t)ctx->n_tiles * sizeof(TileMeta));
    CK(cudaMemsetAsync(ctx->err_flag.p, 0, 16, s));
    LAUNCH(kt_tile_meta, ctx->n_tiles, BA_THREADS, 0, n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam), P<TileMeta>(ctx->tmeta),
           P<int32_t>(ctx->err_flag));
    int32_t h_max[2] = {0, 0};
    CK(cudaMemcpyAsync(h_max, ctx->err_flag.p, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const bool ok = h_max[0] <= BA_TILE_MAXSPAN && h_max[1] <= BA_TILE_MAXCAP;
    if (!ok && o.jacobian_store == BA_JAC_TILED)
      return fail(ctx, BA_ERR_UNSUPPORTED, "tiled store: a point tile spans %d cameras / holds %d observations (limits %d / %d)",
                  h_max[0], h_max[1], BA_TILE_MAXSPAN, BA_TILE_MAXCAP);
    if (ok) {
      const int need = std::max(1, cdiv(h_max[1], BA_THREADS));
      ctx->tile_npt = need <= 2 ? 2 : need <= 3 ? 3 : need <= 4 ? 4 : need <= 6 ? 6 : 8;
      RES(tseg, (size_t)ctx->n_tiles * (BA_TILE_MAXSPAN + 1) * 2);
      RES(tout, (size_t)ctx->n_tiles * BA_TILE_MAXSPAN * 4);
      RES(taux, no * 4);
      RES(tm_cam, no * 4);
      RES(tm_pt, no * 4);
      RES(tm_uv, no * 16);
      RES(ftm, n_pad * 32);
      ctx->Tg0 = P<double2>(ctx->ftm);
      ctx->Tg1 = P<double2>(ctx->ftm) + n_pad;
      RES(cam_tmin, nc * 4);
      RES(cam_tmax, nc * 4);
      RES(tcnt, (nc + 1) * 4);
      RES(tpart_ptr, (nc + 1) * 4);
      LAUNCH(k_fill_i32, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->cam_tmin), 0x7fffffff);
      LAUNCH(k_fill_i32, ctx->nblk_cam, BA_THREADS, 0, n_cam, P<int32_t>(ctx->cam_tmax), -1);
      LAUNCH(k_fill_i32, cdiv(ctx->n_tiles * BA_TILE_MAXSPAN, BA_THREADS), BA_THREADS, 0, ctx->n_tiles * BA_TILE_MAXSPAN,
             P<int32_t>(ctx->tout), -1);
      LAUNCH(kt_tile_build, ctx->n_tiles, BA_THREADS, (size_t)(h_max[1] + 1) * 4, P<TileMeta>(ctx->tmeta), P<int32_t>(ctx->pm_cam),
             P<int32_t>(ctx->pm_pt), P<double2>(ctx->pm_uv), P<int32_t>(ctx->tm_cam), P<int32_t>(ctx->tm_pt), P<double2>(ctx->tm_uv),
             P<uint32_t>(ctx->taux), P<uint16_t>(ctx->tseg), P<int32_t>(ctx->cam_tmin), P<int32_t>(ctx->cam_tmax));
      LAUNCH((kt_cam_tiles<0>), ctx->nblk_cam, BA_THREADS, 0, n_cam, P<TileMeta>(ctx->tmeta), P<uint16_t>(ctx->tseg),
             P<int32_t>(ctx->cam_tmin), P<int32_t>(ctx->cam_tmax), (const int32_t *)nullptr, P<int32_t>(ctx->tcnt),
             (int32_t *)nullptr);
      LAUNCH(k_exclusive_scan, 1, 1024, 0, n_cam, P<int32_t>(ctx->tcnt), P<int32_t>(ctx->tpart_ptr));
      LAUNCH((kt_cam_tiles<1>), ctx->nblk_cam, BA_THREADS, 0, n_cam, P<TileMeta>(ctx->tmeta), P<uint16_t>(ctx->tseg),
             P<int32_t>(ctx->cam_tmin), P<int32_t>(ctx->cam_tmax), P<int32_t>(ctx->tpart_ptr), (int32_t *)nullptr,
             P<int32_t>(ctx->tout));
      int32_t h_parts = 0;
      CK(cudaMemcpyAsync(&h_parts, P<int32_t>(ctx->tpart_ptr) + n_cam, 4, cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
      ctx->n_tparts = h_parts;
      RES(part6t, (size_t)(h_parts + 1) * 48);
      ctx->tiled = true;
    }
  }
  RES(part_blk, (size_t)(h_items + 1) * 61 * 8);
  RES(part6, (size_t)(h_items + 1) * 6 * 8);
  RES(part21, (size_t)(h_items + 1) * 21 * 8);
  RES(part_ex, (size_t)(h_items + 1) * 30 * 8);
  // unit scale vectors (jacobi_scaling off, and the un-scaled evaluation hook)
  LAUNCH(k_fill, cdiv(6 * n_cam, 256), 256, 0, P<double>(ctx->one_c), (size_t)6 * nc, 1.0);
  LAUNCH(k_fill, cdiv(3 * n_pt, 256), 256, 0, P<double>(ctx->one_p), (size_t)3 * np, 1.0);
  LAUNCH(k_fill, 1, 256, 0, P<double>(ctx->one_k), (size_t)4, 1.0);
  if (solver == BA_SOLVER_EXPLICIT_CHOLESKY && sp_ref) {
    // no dense S, no pair list: the block-sparse structure of build_sparse_structure() holds S
    RES(W, (no + 1) * 144);
    RES(WV, (no + 1) * 144);
    RES(spb_B, nc * 192 + 64);
    RES(spb_Z, nc * 192 + 64);
    RES(spb_kk, 20 * 8);
    RES(spb_part, (size_t)(ctx->nblk_cam + 1) * 14 * 8);
    CK(cudaMemsetAsync(ctx->yk.p, 0, 32, s));  // (no intrinsics: y_k stays 0)
    prof.stamp("rest");
  } else if (solver == BA_SOLVER_EXPLICIT_CHOLESKY) {
    RES(W, (no + 1) * 144);
    RES(WV, (no + 1) * 144);
    RES(S, (size_t)ctx->n_red * ctx->n_red * 8 + 64);
    RES(rhs, (size_t)ctx->n_red * 8 + 64);
    RES(chol_v, (size_t)(ctx->n_red + 64 + 8) * 8);
    // blocked Cholesky: L^-1 of every diagonal tile (kept for the substitution) and the flag-in-data slots of k_chol_solve2
    RES(chol_linv, (size_t)cdiv(ctx->n_red, CH_NB) * CH_NB * CH_NB * 8);
    RES(chol_lsub, (size_t)(cdiv(ctx->n_red, CH_NB) + 1) * CH_NB * CH_NB * 8);  // panel tiles right below the diagonal (look-ahead)
    RES(chol_slots, (size_t)2 * cdiv(ctx->n_red, CH_NB) * CH_NB * sizeof(ChSlot));
    prof.stamp("rest");
    // windows: device-built pair list; the global REF problem keeps the host-built list of NON-EMPTY blocks
    // (320 k mostly empty blocks at 800 keyframes)
    const bool dev_pairs = ctx->n_free <= 64 && (ctx->src_on_device || getenv("BA_HOST_PAIRS") == nullptr);
    if (!dev_pairs && ctx->src_on_device)
      return fail(ctx, BA_ERR_UNSUPPORTED, "device-resident windows are limited to 65 keyframes (the pair list of larger explicit problems is host-built)");
    int rc = dev_pairs ? build_pair_list_device(ctx) : build_pair_list(ctx, cam_idx, pt_idx);
    if (rc) return rc;
    prof.stamp("pair list");
  }
  prof.flush();
  CK(cudaGetLastError());
  ctx->forking = ctx->n_ranks == 1 && getenv("BA_NO_FORK") == nullptr;
  ctx->cur = ctx->stream;
  ctx->uploaded = true;
  return BA_OK;
}

// ------------------------------------------------------------------ multi-GPU reductions
static int nccl_allreduce(ba_gpu_ctx *ctx, double *buf, size_t n, bool is_max) {
  ncclResult_t r = g_nccl.AllReduce(buf, buf, n, ncclFloat64_, is_max ? ncclMax_ : ncclSum_, ctx->comm, ctx->stream);
  if (r != 0) return fail(ctx, BA_ERR_COMM, "ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  ctx->collectives++;
  return 0;
}
// scalar from per-CTA partials: single GPU -> the partial array itself (summed by
// the consumer in fixed order); sharded -> local sum, all-reduce, 1-entry array
struct PartRef {
  const double *p;
  int n;
};
static PartRef reduce_scalar(ba_gpu_ctx *ctx, const double *part, int nblk, int slot, bool is_max, int gate) {
  if (ctx->n_ranks == 1) return PartRef{part, nblk};
  double *out = P<double>(ctx->scal) + slot;
  k_reduce_partials<<<1, BA_THREADS, 0, ctx->stream>>>(nblk, part, out, is_max ? 1 : 0, P<LmState>(ctx->st), gate);
  ctx->launches++;
  if (nccl_allreduce(ctx, out, 1, is_max)) ctx->comm_error = true;
  return PartRef{out, 1};
}
// several sums at once: one collective for the group (a sharded LM iteration is latency-bound: every small all-reduce costs
// about as much as the kernels between two of them)
static void reduce_scalar_group(ba_gpu_ctx *ctx, int n, const double *const part[], const int nblk[], int slot0, int gate, PartRef out[]) {
  for (int k = 0; k < n; ++k) out[k] = PartRef{part[k], nblk[k]};
  if (ctx->n_ranks == 1) return;
  double *base = P<double>(ctx->scal) + slot0;
  for (int k = 0; k < n; ++k) {
    k_reduce_partials<<<1, BA_THREADS, 0, ctx->stream>>>(nblk[k], part[k], base + k, 0, P<LmState>(ctx->st), gate);
    ctx->launches++;
    out[k] = PartRef{base + k, 1};
  }
  if (nccl_allreduce(ctx, base, (size_t)n, false)) ctx->comm_error = true;
}
// per-camera sums of item partials: single GPU -> (item_ptr, part); sharded ->
// dense local sums, all-reduce, (identity, dense)
struct ItemRef {
  const int32_t *ptr;
  const double *part;
};
template <int NV>
static ItemRef reduce_items(ba_gpu_ctx *ctx, const double *part, Buf &dense, int gate, const int32_t *ptr = nullptr) {
  if (!ptr) ptr = P<int32_t>(ctx->item_ptr);
  if (ctx->n_ranks == 1) return ItemRef{ptr, part};
  k_sum_items<NV><<<cdiv(ctx->n_cam * NV, BA_THREADS), BA_THREADS, 0, ctx->stream>>>(
      ctx->n_cam, ptr, part, P<double>(dense), P<LmState>(ctx->st), gate);
  ctx->launches++;
  if (nccl_allreduce(ctx, P<double>(dense), (size_t)ctx->n_cam * NV, false)) ctx->comm_error = true;
  return ItemRef{P<int32_t>(ctx->ident), P<double>(dense)};
}
// failure flags must agree on every rank (they steer the control flow); a maximum over per-CTA partials (the gradient
// norm) can ride on the same collective
static PartRef sync_flags(ba_gpu_ctx *ctx, const double *max_part = nullptr, int max_nblk = 0, int gate = GATE_RUN) {
  if (ctx->n_ranks == 1) return PartRef{max_part, max_nblk};
  double *out = P<double>(ctx->scal) + 32;
  k_flags_pack<<<1, 1, 0, ctx->stream>>>(P<LmState>(ctx->st), out);
  if (max_part) {
    k_reduce_partials<<<1, BA_THREADS, 0, ctx->stream>>>(max_nblk, max_part, out + 2, 1, P<LmState>(ctx->st), gate);
    ctx->launches++;
  }
  if (nccl_allreduce(ctx, out, max_part ? 3 : 2, true)) ctx->comm_error = true;
  k_flags_unpack<<<1, 1, 0, ctx->stream>>>(P<LmState>(ctx->st), out);
  ctx->launches += 2;
  return PartRef{out + 2, 1};
}

// ------------------------------------------------------------------ fork / join of independent branches
// fork_side(): what follows runs on the side stream, after everything enqueued so far on the main one;
// fork_main(): back on the main stream (concurrently with the side branch); join(): the main stream waits
// for the side branch.  No-ops unless ctx->forking (single GPU, windowed explicit solver).
static void fork_side(ba_gpu_ctx *ctx) {
  if (!ctx->forking) return;
  cudaEventRecord(ctx->ev_fork, ctx->stream);
  cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0);
  ctx->cur = ctx->stream2;
}
static void fork_main(ba_gpu_ctx *ctx) { ctx->cur = ctx->stream; }
// inside a fork: the side branch continues after what the main branch has enqueued so far
static void side_after_main(ba_gpu_ctx *ctx) {
  if (ctx->forking) {
    cudaEventRecord(ctx->ev_mid, ctx->stream);
    cudaStreamWaitEvent(ctx->stream2, ctx->ev_mid, 0);
    ctx->cur = ctx->stream2;
  }
}
static void join(ba_gpu_ctx *ctx) {
  ctx->cur = ctx->stream;
  if (!ctx->forking) return;
  cudaEventRecord(ctx->ev_join, ctx->stream2);
  cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
}

// ------------------------------------------------------------------ phase timing (large-problem solvers)
static const char *const g_phase_names[BA_PHASE_COUNT] = {
    "start", "iteration_zero", "point_inverse", "reduced_rhs", "schur_complement", "linear_solve_factor_or_pcg",
    "linear_solve_substitution", "back_substitution_model_cost", "candidate_cost", "lm_control", "accept_relinearize"};
static void phase_mark(ba_gpu_ctx *ctx, int id) {
  if (!ctx->ph_on) return;
  if (ctx->ph_n >= (int)ctx->ph_ev.size()) {
    if (ctx->ph_ev.size() >= 8192) return;
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    ctx->ph_ev.push_back(e);
    ctx->ph_id.push_back(0);
  }
  ctx->ph_id[ctx->ph_n] = id;
  cudaEventRecord(ctx->ph_ev[ctx->ph_n], ctx->stream);
  ctx->ph_n++;
}
static void phase_collect(ba_gpu_ctx *ctx) {
  for (int k = 0; k < BA_PHASE_COUNT; ++k) ctx->ph_ms[k] = 0.0;
  for (int i = 1; i < ctx->ph_n; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ph_ev[i - 1], ctx->ph_ev[i]) == cudaSuccess) ctx->ph_ms[ctx->ph_id[i]] += ms;
  }
}

// ------------------------------------------------------------------ pipeline pieces
// linearise at the current point in both orders + normal-equation blocks
static void enqueue_linearize(ba_gpu_ctx *ctx, int gate, const double *sc, const double *sp, const double *sk,
                              bool force_planes = false, bool from_candidate = false) {
  const int D = ctx->depth, K = ctx->nk;
  LmState *st = P<LmState>(ctx->st);
  // from_candidate (planes path): read the accepted candidate x+ directly while k_accept copies it into x on the side stream
  const double *xpose = P<double>(from_candidate ? ctx->pose_c : ctx->pose), *xpt = P<double>(from_candidate ? ctx->pt_c : ctx->pt),
               *xintr = P<double>(from_candidate ? ctx->intr_c : ctx->intr);
  if (ctx->fact && !force_planes) {
    const double *intr = P<double>(ctx->intr);
    LAUNCH(k_cam_geo, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, ctx->fixed_cam, P<double>(ctx->pose), sc, P<double>(ctx->geo), st,
           gate);
    // point-major branch on the side stream, camera-major branch on the main one (both need geo)
    fork_side(ctx);
    LAUNCH((kf_linearize<0>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->pm_pt),
           P<double2>(ctx->pm_uv), P<double>(ctx->pose), P<double>(ctx->pt), intr, ctx->cp, ctx->Fp_, (double *)nullptr, st,
           gate);
    LAUNCH(kf_pt_blocks, ctx->n_tiles, BA_THREADS, 0, ctx->n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam), ctx->Fp_,
           P<double>(ctx->geo), intr, sp, P<double>(ctx->V), P<double>(ctx->gp), P<double>(ctx->dp), ctx->lo, st, gate);
    if (ctx->tiled)
      LAUNCH(kt_linearize, ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->tm_cam), P<int32_t>(ctx->tm_pt),
             P<double2>(ctx->tm_uv), P<double>(ctx->pose), P<double>(ctx->pt), intr, ctx->cp, ctx->Tg0, ctx->Tg1, st, gate);
    fork_main(ctx);
    LAUNCH((kf_linearize<1>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
           P<double2>(ctx->uv), P<double>(ctx->pose), P<double>(ctx->pt), intr, ctx->cp, ctx->Fc_, P<double>(ctx->pc_lin), st,
           gate);
    LAUNCH(kf_cam_blocks, ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), ctx->Fc_, P<double>(ctx->geo), intr,
           P<double>(ctx->part_blk), st, gate);
    ItemRef ir = reduce_items<27>(ctx, P<double>(ctx->part_blk), ctx->red_blk, gate);
    LAUNCH((k_cam_blocks_fin<0>), cdiv(ctx->n_cam * 27, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ir.ptr, ir.part, P<double>(ctx->U), P<double>(ctx->gc),
           P<double>(ctx->Uck), P<double>(ctx->dc), ctx->lo, st, gate);
    join(ctx);
    return;
  }
  DISPATCH_DK(D, K, {
    // point-major branch (side stream): linearise + point blocks
    fork_side(ctx);
    LAUNCH((k_linearize<DD, KK, 0>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->pm_pt),
           P<double2>(ctx->pm_uv), P<double>(ctx->pm_depth), xpose, xpt, xintr, sc,
           sp, sk, ctx->cp, ctx->Jp_, (double *)nullptr, st, gate);
    LAUNCH((k_pt_blocks<DD, KK>), ctx->pl_tiles, BA_THREADS, 0, ctx->n_pt, ctx->pl_tile_pts, P<int32_t>(ctx->pt_rowptr), ctx->Jp_, P<double>(ctx->V),
           P<double>(ctx->gp), P<double>(ctx->Wk), P<double>(ctx->dp), ctx->lo, st, gate);
    // camera-major branch (main stream): linearise + camera blocks
    fork_main(ctx);
    LAUNCH((k_linearize<DD, KK, 1>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
           P<double2>(ctx->uv), P<double>(ctx->depthv), xpose, xpt, xintr, sc, sp,
           sk, ctx->cp, ctx->Jc_, P<double>(ctx->pc_lin), st, gate);
    LAUNCH((k_cam_blocks<DD, KK>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), ctx->Jc_,
           P<double>(ctx->part_blk), st, gate);
    ItemRef ir = ItemRef{P<int32_t>(ctx->item_ptr), P<double>(ctx->part_blk)};
    if (KK == 0) ir = reduce_items<27>(ctx, P<double>(ctx->part_blk), ctx->red_blk, gate);
    if (KK) {
      // camera blocks and the intrinsics block finish in one launch
      const int nb = cdiv(ctx->n_cam * 51, BA_THREADS);
      LAUNCH(k_cam_kk_fin, nb + 1, BA_THREADS, 0, nb, ctx->n_cam, ir.ptr, ir.part, P<double>(ctx->U), P<double>(ctx->gc),
             P<double>(ctx->Uck), P<double>(ctx->dc), ctx->n_items, xintr, P<double>(ctx->intr_prior), sk, ctx->cp,
             ctx->lo, P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->rk), P<double>(ctx->Jkk), st, gate);
    } else {
      LAUNCH((k_cam_blocks_fin<0>), cdiv(ctx->n_cam * 27, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ir.ptr, ir.part,
             P<double>(ctx->U), P<double>(ctx->gc), P<double>(ctx->Uck), P<double>(ctx->dc), ctx->lo, st, gate);
    }
  });
  join(ctx);
}
static void enqueue_state_norms(ba_gpu_ctx *ctx, int gate, const double *sc, const double *sp, const double *sk) {
  LAUNCH(k_state_norms, ctx->nblk_ent, BA_THREADS, 0, ctx->n_cam, ctx->n_pt, ctx->nk, ctx->fixed_cam, P<double>(ctx->pose),
         P<double>(ctx->pt), P<double>(ctx->intr), P<double>(ctx->gc), P<double>(ctx->gp), P<double>(ctx->gk), sc, sp, sk,
         P<double>(ctx->pe_gmax), P<double>(ctx->pe_xn), P<LmState>(ctx->st), gate, ctx->rank == 0 ? 1.0 : 0.0);
}

// IterationZero of the trust-region minimizer
static void enqueue_iteration_zero(ba_gpu_ctx *ctx, bool begin_loop = true) {
  LmState *st = P<LmState>(ctx->st);
  LAUNCH(k_lm_init, 1, 1, 0, st, ctx->opt.initial_trust_region_radius);
  const bool js = ctx->opt.jacobi_scaling != 0;
  // first pass un-scaled: cost, gradient norm, column norms
  enqueue_linearize(ctx, GATE_RUN, P<double>(ctx->one_c), P<double>(ctx->one_p), P<double>(ctx->one_k));
  enqueue_state_norms(ctx, GATE_RUN, P<double>(ctx->one_c), P<double>(ctx->one_p), P<double>(ctx->one_k));
  if (js) {
    LAUNCH(k_make_scale, ctx->nblk_ent, BA_THREADS, 0, ctx->n_cam, ctx->n_pt, ctx->nk, P<double>(ctx->U), P<double>(ctx->V),
           P<double>(ctx->Ukk), P<double>(ctx->sc), P<double>(ctx->sp), P<double>(ctx->sk), st, GATE_RUN);
    enqueue_linearize(ctx, GATE_RUN, P<double>(ctx->sc), P<double>(ctx->sp), P<double>(ctx->sk));
  } else {
    cudaMemcpyAsync(ctx->sc.p, ctx->one_c.p, (size_t)ctx->n_cam * 48, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaMemcpyAsync(ctx->sp.p, ctx->one_p.p, (size_t)ctx->n_pt * 24, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaMemcpyAsync(ctx->sk.p, ctx->one_k.p, 32, cudaMemcpyDeviceToDevice, ctx->stream);
  }
  LAUNCH(k_set_have_scale, 1, 1, 0, st);
  sync_flags(ctx);
  const PartRef rc_ = reduce_scalar(ctx, P<double>(ctx->pc_lin), ctx->nblk_obs, 0, false, GATE_RUN);
  const PartRef rg_ = reduce_scalar(ctx, P<double>(ctx->pe_gmax), ctx->nblk_ent, 1, true, GATE_RUN);
  const PartRef rx_ = reduce_scalar(ctx, P<double>(ctx->pe_xn), ctx->nblk_ent, 2, false, GATE_RUN);
  LAUNCH(k_lm_iter0, 1, BA_THREADS, 0, rc_.n, rg_.n, ctx->nk, rc_.p, rg_.p, rx_.p, P<double>(ctx->rk), ctx->lo, st,
         P<BaIterRec>(ctx->trace));
  if (begin_loop) LAUNCH(k_lm_begin, 1, 1, 0, ctx->lo, st);  // top-of-loop checks of iteration 1; later ones ride on k_lm_control / k_lm_post
  ctx->linearized = true;
}

// one implicit-Schur product: part6 <- sum Jc^T (alpha Jc v - Jp t), t <- pass 1 of v
static void enqueue_point_inverse(ba_gpu_ctx *ctx, int gate) {
  LmState *st = P<LmState>(ctx->st);
  if (ctx->fact)
    LAUNCH(kf_point_inverse, ctx->nblk_pt, BA_THREADS, 0, ctx->n_pt, P<double>(ctx->V), P<double>(ctx->dp), P<double>(ctx->gp),
           P<double>(ctx->sp), P<double>(ctx->Vinv), P<double>(ctx->Vs), P<double>(ctx->tgs), st, gate);
  else
    LAUNCH(k_point_inverse, ctx->nblk_pt, BA_THREADS, 0, ctx->n_pt, P<double>(ctx->V), P<double>(ctx->dp), P<double>(ctx->gp),
           P<double>(ctx->Vinv), P<double>(ctx->tg), st, gate);
}

template <int NPT>
static void launch_fused(ba_gpu_ctx *ctx, const double *v, int gate) {
  LAUNCH((kt_schur_fused<NPT>), ctx->n_tiles, BA_THREADS, tile_smem_bytes(NPT), ctx->n_pt, P<int32_t>(ctx->pt_rowptr),
         P<TileMeta>(ctx->tmeta), P<uint16_t>(ctx->tseg), P<int32_t>(ctx->tout), P<uint32_t>(ctx->taux), ctx->Tg0, ctx->Tg1,
         P<double>(ctx->geo), P<double>(ctx->pose), v, P<double>(ctx->intr), P<double>(ctx->Vs), P<double>(ctx->part6t),
         P<LmState>(ctx->st), gate);
}

// One implicit-Schur product of v (without the LM damping term): enqueues the
// kernels and returns the per-camera partial list that k_pcg_q / k_pcg_reset add up.
// passes: 3 = product (fused kernel if the store is tiled), 1 / 2 = one pass of the
// two-pass form, 7 = force the two-pass form.
static ItemRef enqueue_matvec(ba_gpu_ctx *ctx, const double *v, int gate, int passes = 3) {
  LmState *st = P<LmState>(ctx->st);
  const int rp = ctx->lo.reset_period;
  if (ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG && passes == 3) {
    if (ctx->spmv6)
      LAUNCH(k_bsr_spmv6, cdiv(ctx->n_cam * 32, BA_THREADS), BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->ent_ptr),
             P<int2>(ctx->ent), P<double>(ctx->Sblk), v, P<double>(ctx->ysp), st, gate);
    else
      LAUNCH(k_bsr_spmv, cdiv(ctx->n_cam * 32, BA_THREADS), BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->ent_ptr),
             P<int2>(ctx->ent), P<double>(ctx->Sblk), v, P<double>(ctx->ysp), st, gate);
    return ItemRef{P<int32_t>(ctx->ident), P<double>(ctx->ysp)};
  }
  if (ctx->tiled && passes == 3) {
    switch (ctx->tile_npt) {
      case 2: launch_fused<2>(ctx, v, gate); break;
      case 3: launch_fused<3>(ctx, v, gate); break;
      case 4: launch_fused<4>(ctx, v, gate); break;
      case 6: launch_fused<6>(ctx, v, gate); break;
      default: launch_fused<8>(ctx, v, gate); break;
    }
    return ItemRef{P<int32_t>(ctx->tpart_ptr), P<double>(ctx->part6t)};
  }
  const ItemRef items_ref{P<int32_t>(ctx->item_ptr), P<double>(ctx->part6)};
  if (ctx->fact) {
    const double *intr = P<double>(ctx->intr);
    if (passes & 1) {
      if (ctx->staged) {
        LAUNCH((kf_schur_pass1<0, 1>), ctx->n_tiles, BA_THREADS, 0, ctx->n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
               ctx->Fp_, P<double>(ctx->geo), v, P<double>(ctx->camx), P<int32_t>(ctx->tile_lo), P<int32_t>(ctx->tile_span), intr,
               P<double>(ctx->Vinv), P<double>(ctx->sp), (const double *)nullptr, (double *)nullptr, P<double>(ctx->ts), st, gate);
      } else {
        LAUNCH(k_pack_camx, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, v, P<double>(ctx->geo), P<double>(ctx->camx), st, gate);
        LAUNCH((kf_schur_pass1<0, 0>), ctx->n_tiles, BA_THREADS, 0, ctx->n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
               ctx->Fp_, P<double>(ctx->geo), v, P<double>(ctx->camx), P<int32_t>(ctx->tile_lo), P<int32_t>(ctx->tile_span), intr,
               P<double>(ctx->Vinv), P<double>(ctx->sp), (const double *)nullptr, (double *)nullptr, P<double>(ctx->ts), st, gate);
      }
    }
    if (passes & 2)
      LAUNCH(kf_schur_pass2, ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx), ctx->Fc_,
             P<double>(ctx->geo), intr, v, P<double>(ctx->ts), 1.0, P<double>(ctx->part6), st, gate);
    return items_ref;
  }
  DISPATCH_D(ctx->depth, {
    if (passes & 1)
    LAUNCH((k_schur_pass1<DD, 0, 0>), ctx->pl_tiles, BA_THREADS, 0, ctx->n_pt, ctx->pl_tile_pts, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
           ctx->Jp_, v, (const double *)nullptr, P<double>(ctx->Vinv), (const double *)nullptr, P<double>(ctx->t), st, gate, rp);
    if (passes & 2)
    LAUNCH((k_schur_pass2<DD>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx),
           ctx->Jc_, v, P<double>(ctx->t), 1.0, P<double>(ctx->part6), st, gate, rp);
  });
  return items_ref;
}

// values of the explicit block-sparse Schur complement (needs V^-1 of this radius).  Point-sharded:
// every rank fills the blocks of its own points into the common structure, the values are all-reduced,
// then the (already reduced) camera blocks U go onto the diagonal.
static void enqueue_sparse_values(ba_gpu_ctx *ctx, int gate) {
  if (ctx->solver != BA_SOLVER_SPARSE_SCHUR_PCG) return;
  LmState *st = P<LmState>(ctx->st);
  if (ctx->n_ranks > 1) cudaMemsetAsync(ctx->Sblk.p, 0, (size_t)ctx->n_sblk * 288, ctx->stream);
  int *ticket = reinterpret_cast<int *>(P<char>(ctx->pcg_bar) + 16);
  cudaMemsetAsync(ticket, 0, 4, ctx->stream);
  // (pair records hold canonical observation indices: the kernel reads the CAMERA-major factored planes)
  const int sps_grid = std::min(cdiv(ctx->n_sblk_local, BA_SPS_CHUNK), ctx->n_sm * ctx->sp_ctas_per_sm);
  if (ctx->sps_simt)
    LAUNCH(k_sp_schur_simt, sps_grid, BA_THREADS, 0, ctx->n_sblk_local, ctx->n_cam, P<int32_t>(ctx->sb_ptr),
           P<unsigned long long>(ctx->sp_lkeys), P<int32_t>(ctx->sp_gid), P<unsigned long long>(ctx->sp_pairs),
           P<int32_t>(ctx->sp_pair_pt), ctx->Fc_, P<double>(ctx->geo), P<double>(ctx->intr), P<double>(ctx->Vs),
           P<double>(ctx->Sblk), ticket, st, gate);
  else
    LAUNCH(k_sp_schur, sps_grid, BA_THREADS, BA_SPS_SMEM, ctx->n_sblk_local, ctx->n_cam, P<int32_t>(ctx->sb_ptr),
           P<unsigned long long>(ctx->sp_lkeys), P<int32_t>(ctx->sp_gid), P<unsigned long long>(ctx->sp_pairs),
           P<int32_t>(ctx->sp_pair_pt), ctx->Fc_, P<double>(ctx->geo), P<double>(ctx->intr), P<double>(ctx->Vs),
           P<double>(ctx->Sblk), ticket, st, gate);
  if (ctx->n_ranks > 1) {
    if (ctx->spchol && ctx->spc_dist && !ctx->sp_full_next) {
      // distributed factorisation: only the blocks another rank needs from this one (and the top part's) are summed
      if (ctx->spc_nx > 0) {
        LAUNCH(k_sp_xpack, cdiv(ctx->spc_nx * 36, BA_THREADS), BA_THREADS, 0, ctx->spc_nx, P<int32_t>(ctx->spc_xidx), P<double>(ctx->Sblk),
               P<double>(ctx->spc_xbuf), 0, st, gate);
        if (nccl_allreduce(ctx, P<double>(ctx->spc_xbuf), (size_t)ctx->spc_nx * 36, false)) ctx->comm_error = true;
        LAUNCH(k_sp_xpack, cdiv(ctx->spc_nx * 36, BA_THREADS), BA_THREADS, 0, ctx->spc_nx, P<int32_t>(ctx->spc_xidx), P<double>(ctx->Sblk),
               P<double>(ctx->spc_xbuf), 1, st, gate);
      }
    } else if (nccl_allreduce(ctx, P<double>(ctx->Sblk), (size_t)ctx->n_sblk * 36, false)) {
      ctx->comm_error = true;
    }
    ctx->sp_full_next = false;
  }
  LAUNCH(k_sp_add_diag, cdiv(ctx->n_cam * 36, BA_THREADS), BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->sp_diag), P<double>(ctx->U),
         P<double>(ctx->Sblk), st, gate);
}

// exact solve of the reduced camera system by the sparse Cholesky: factorisation bottom-up (one launch per tree level, forward
// substitution fused), backward substitution top-down.  b / dsq are complete (all-reduced) on every rank: the solve is replicated.
static SpChol spchol_args(ba_gpu_ctx *ctx) {
  SpChol a;
  a.node = P<int32_t>(ctx->spn_node);
  a.bord = P<int32_t>(ctx->spn_bord);
  a.children = P<int32_t>(ctx->spn_children);
  a.rel = P<int32_t>(ctx->spn_rel);
  a.inv = P<int32_t>(ctx->spn_inv);
  a.aent = P<int32_t>(ctx->spn_aent);
  a.perm = P<int32_t>(ctx->spn_perm);
  a.level_nodes = P<int32_t>(ctx->spn_levels);
  a.S = P<double>(ctx->Sblk);
  a.dsq = P<double>(ctx->dsq);
  a.b = P<double>(ctx->b);
  a.panel = P<double>(ctx->spc_panel);
  a.U = P<double>(ctx->spc_U);
  a.ru = P<double>(ctx->spc_U) + ctx->spc_ru_off;
  a.z = P<double>(ctx->spc_z);
  a.linv = P<double>(ctx->spc_linv);
  a.ypos = P<double>(ctx->spc_ypos);
  a.yc = P<double>(ctx->yc);
  a.prof = getenv("BA_SPCHOL_PROF") ? P<unsigned long long>(ctx->spc_prof) : nullptr;
  const bool border = ctx->spc_nrhs > 1;
  a.Bc = border ? P<double>(ctx->spb_B) : nullptr;
  a.Zb = border ? P<double>(ctx->spb_Z) : nullptr;
  a.yk = border ? P<double>(ctx->yk) : nullptr;
  return a;
}
// intrinsics border between the forward and the backward substitution: T = C - Z^T Z, t = b_k - Z^T z, y_k = T^-1 t
static void enqueue_spchol_border(ba_gpu_ctx *ctx, int gate) {
  LmState *st = P<LmState>(ctx->st);
  const int nblk = ctx->nblk_cam;
  LAUNCH(k_spb_reduce, nblk, BA_THREADS, 0, ctx->n_cam, P<double>(ctx->spb_Z), P<double>(ctx->spc_z), P<double>(ctx->spb_part), st,
         gate);
  LAUNCH(k_spb_solve, 1, 32, 0, nblk, P<double>(ctx->spb_part), P<double>(ctx->spb_kk), P<double>(ctx->yk), st, gate);
}
static void enqueue_spchol(ba_gpu_ctx *ctx, int gate) {
  LmState *st = P<LmState>(ctx->st);
  const SpSymbolic &S = ctx->sym;
  const SpChol a = spchol_args(ctx);
  // every kernel of the chain starts with griddepcontrol.wait (gate_open): programmatic dependent launches let the blocks of
  // the next launch become resident on idle SMs (the upper tree levels have few nodes) while the previous one still runs
  if (ctx->spc_tree) {
    // the whole linear solve in one persistent launch (k_spchol_tree): dependency counters instead of level barriers.
    // Partitioned tree: one launch for the subtrees (phase A), one for the top part and the backward substitution (phase B).
    SpTree t;
    int *cnt = P<int>(ctx->spc_cnt);
    t.tiles = P<int32_t>(ctx->spc_tiles);
    t.fdone = cnt + 16;
    t.udone = t.fdone + S.n_nodes;
    t.sdone = t.udone + S.n_nodes;
    cudaMemcpyAsync(cnt, ctx->spc_cnt_init.p, ((size_t)3 * S.n_nodes + 16) * 4, cudaMemcpyDeviceToDevice, ctx->cur);
    const size_t smem = std::max(std::max(ctx->spc_smem_factor, ctx->spc_smem_solve), ctx->spc_smem_update);
    auto launch = [&](int first, int n, int slot) {
      if (n <= 0) return;
      t.queue = P<int2>(ctx->spc_queue) + first;
      t.n_items = n;
      t.ticket = cnt + slot;
      if (ctx->spc_nrhs > 1)
        LAUNCH((k_spchol_tree<5>), std::min(ctx->n_sm, n), SPC_THREADS, smem, a, t, st, gate);
      else
        LAUNCH((k_spchol_tree<1>), std::min(ctx->n_sm, n), SPC_THREADS, smem, a, t, st, gate);
    };
    if (ctx->spc_parts == 1 && ctx->spc_nrhs > 1) {
      // intrinsics border: the queue's factor / update prefix, the 4 x 4 border system, then the backward substitution
      launch(0, ctx->spc_qB, 0);
      enqueue_spchol_border(ctx, gate);
      phase_mark(ctx, BA_PHASE_FACTOR);
      launch(ctx->spc_qB, ctx->spc_qB_n, 1);
      return;
    }
    if (ctx->spc_parts == 1) {
      launch(0, ctx->spc_n_items, 0);
      phase_mark(ctx, BA_PHASE_FACTOR);
      return;
    }
    if (ctx->spc_dist) cudaMemsetAsync(ctx->spc_U.p, 0, ctx->spc_xchg * 8, ctx->cur);
    for (int p = 0; p < ctx->spc_parts; ++p) launch(ctx->spc_qA[p], ctx->spc_qA[p + 1] - ctx->spc_qA[p], p);
    if (ctx->spc_dist && nccl_allreduce(ctx, P<double>(ctx->spc_U), ctx->spc_xchg, false)) ctx->comm_error = true;
    if (ctx->spc_dist) cudaMemsetAsync(ctx->yc.p, 0, ((size_t)6 * ctx->n_cam + 1) * 8, ctx->cur);
    launch(ctx->spc_qB, ctx->spc_qB_n, ctx->spc_parts);
    if (ctx->spc_dist) {
      // the step: every rank holds the top part's and its own subtrees' cameras; summed over ranks (zeros elsewhere, the top
      // part kept by rank 0 only) with the failure flag in the extra slot
      LAUNCH(k_spchol_dist_pre, cdiv(std::max(1, ctx->spc_n_topcams) * 6, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->spc_n_topcams,
             P<int32_t>(ctx->spc_topcams), ctx->rank, P<double>(ctx->yc), st, gate);
      if (nccl_allreduce(ctx, P<double>(ctx->yc), (size_t)6 * ctx->n_cam + 1, false)) ctx->comm_error = true;
      LAUNCH(k_spchol_dist_post, 1, 32, 0, ctx->n_cam, P<double>(ctx->yc), st, gate);
    }
    phase_mark(ctx, BA_PHASE_FACTOR);
    return;
  }
  const bool pdl0 = ctx->pdl;
  ctx->pdl = !ctx->pdl_off;
  for (int l = 0; l < S.n_levels; ++l) {
    const int nodes = S.level_ptr[l + 1] - S.level_ptr[l];
    if (ctx->spc_nrhs > 1)
      LAUNCH((k_spchol_factor<5>), nodes, SPC_THREADS, ctx->spc_smem_factor, a, S.level_ptr[l], st, gate);
    else
      LAUNCH((k_spchol_factor<1>), nodes, SPC_THREADS, ctx->spc_smem_factor, a, S.level_ptr[l], st, gate);
    if (l + 1 < S.n_levels) {  // (roots have no border)
      const int tiles = std::max(1, std::min(8, ctx->n_sm / std::max(1, nodes)));
      if (ctx->spc_nrhs > 1)
        LAUNCH((k_spchol_update<5>), nodes * tiles, SPU_THREADS, ctx->spc_smem_update, a, S.level_ptr[l], tiles, st, gate);
      else
        LAUNCH((k_spchol_update<1>), nodes * tiles, SPU_THREADS, ctx->spc_smem_update, a, S.level_ptr[l], tiles, st, gate);
    }
  }
  if (ctx->spc_nrhs > 1) enqueue_spchol_border(ctx, gate);
  phase_mark(ctx, BA_PHASE_FACTOR);
  for (int l = S.n_levels - 1; l >= 0; --l)
    LAUNCH(k_spchol_solve, S.level_ptr[l + 1] - S.level_ptr[l], SPC_THREADS, ctx->spc_smem_solve, a, S.level_ptr[l], st, gate);
  ctx->pdl = pdl0;
}

static int poll_state(ba_gpu_ctx *ctx) {
  CK(cudaMemcpyAsync(ctx->h_st, ctx->st.p, sizeof(LmState), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// one PCG iteration; `it` mirrors the device-side iteration counter (they agree
// while the controller has not finished; afterwards every kernel is gated off)
static void enqueue_pcg_iteration(ba_gpu_ctx *ctx, int it) {
  LmState *st = P<LmState>(ctx->st);
  const int rp = ctx->lo.reset_period;
  const int reset = (rp > 0 && (it % rp) == 0) ? 1 : 0;
  LAUNCH(k_pcg_dir, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<double>(ctx->z), P<double>(ctx->p), st, GATE_PCG);
  const bool replicated = ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG;  // S is complete on every rank: no exchange in PCG
  ItemRef ir = enqueue_matvec(ctx, P<double>(ctx->p), GATE_PCG);
  if (!replicated) ir = reduce_items<6>(ctx, ir.part, ctx->red6, GATE_PCG, ir.ptr);
  LAUNCH(k_pcg_q, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, ir.ptr, ir.part, P<double>(ctx->dc), P<double>(ctx->p),
         P<double>(ctx->q), P<double>(ctx->pcam_pq), st, GATE_PCG);
  LAUNCH(k_pcg_step, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, ctx->nblk_cam, P<double>(ctx->pcam_pq), P<double>(ctx->p),
         P<double>(ctx->q), P<double>(ctx->b), P<double>(ctx->Minv), P<double>(ctx->x), P<double>(ctx->r), P<double>(ctx->z),
         P<double>(ctx->pcam_rho), P<double>(ctx->pcam_Q), ctx->lo, st, GATE_PCG, reset);
  if (reset) {
    ir = enqueue_matvec(ctx, P<double>(ctx->x), GATE_PCG);
    if (!replicated) ir = reduce_items<6>(ctx, ir.part, ctx->red6, GATE_PCG, ir.ptr);
    LAUNCH(k_pcg_reset, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, ctx->nblk_cam, ir.ptr, ir.part, P<double>(ctx->dc),
           P<double>(ctx->x), P<double>(ctx->b), P<double>(ctx->Minv), P<double>(ctx->r), P<double>(ctx->z),
           P<double>(ctx->pcam_rho), P<double>(ctx->pcam_Q), ctx->lo, st, GATE_PCG);
  }
}

// reduced system solve by implicit Schur + block-Jacobi PCG; host polls the
// device-side PCG controller every poll_interval iterations
static int solve_implicit(ba_gpu_ctx *ctx) {
  LmState *st = P<LmState>(ctx->st);
  if (ctx->fact) {
    const double *intr = P<double>(ctx->intr);
    LAUNCH(kf_schur_pass2, ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx), ctx->Fc_,
           P<double>(ctx->geo), intr, P<double>(ctx->gc), P<double>(ctx->tgs), 0.0, P<double>(ctx->part6), st, GATE_RUN);
    if (ctx->solver != BA_SOLVER_SPARSE_SCHUR_PCG)  // the block-sparse solver reads the diagonal blocks of S itself
    LAUNCH(kf_schur_diag, ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx), ctx->Fc_,
           P<double>(ctx->geo), intr, P<double>(ctx->Vs), P<double>(ctx->part21), st, GATE_RUN);
  } else
  DISPATCH_D(ctx->depth, {
    // rhs = -g_c + sum Jc^T Jp V^-1 g_p
    LAUNCH((k_schur_pass2<DD>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx),
           ctx->Jc_, P<double>(ctx->gc), P<double>(ctx->tg), 0.0, P<double>(ctx->part6), st, GATE_RUN, 0);
    LAUNCH((k_schur_diag<DD>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx), ctx->Jc_,
           P<double>(ctx->Vinv), P<double>(ctx->part21), st, GATE_RUN);
  });
  phase_mark(ctx, BA_PHASE_RHS);
  enqueue_sparse_values(ctx, GATE_RUN);
  // (the exact solve does not branch on the failure flags; the ranks agree on them after it, before the step is judged)
  if (!ctx->spchol) sync_flags(ctx);
  phase_mark(ctx, BA_PHASE_SCHUR);
  if (ctx->spchol) {
    // exact step: b and the damping, then the factorisation and the two substitutions (yc written by the last kernels)
    ItemRef i6c = reduce_items<6>(ctx, P<double>(ctx->part6), ctx->red6, GATE_RUN);
    LAUNCH(k_spchol_rhs, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, i6c.ptr, i6c.part, P<double>(ctx->gc), P<double>(ctx->dc),
           P<double>(ctx->b), P<double>(ctx->dsq), st, GATE_RUN, 0);
    enqueue_spchol(ctx, GATE_RUN);
    return 0;
  }
  if (ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG) {
    LAUNCH(k_sp_minv, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->sp_diag), P<double>(ctx->Sblk), P<double>(ctx->dc),
           P<double>(ctx->Minv), P<double>(ctx->dsq), st, GATE_RUN);
  } else {
    ItemRef i21 = reduce_items<21>(ctx, P<double>(ctx->part21), ctx->red21, GATE_RUN);
    LAUNCH(k_schur_diag_fin, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, i21.ptr, i21.part, P<double>(ctx->U), P<double>(ctx->dc),
           P<double>(ctx->Minv), (double *)nullptr, st, GATE_RUN);
  }
  ItemRef i6 = reduce_items<6>(ctx, P<double>(ctx->part6), ctx->red6, GATE_RUN);
  LAUNCH(k_pcg_init, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, i6.ptr, i6.part, P<double>(ctx->gc), P<double>(ctx->Minv),
         P<double>(ctx->b), P<double>(ctx->x), P<double>(ctx->r), P<double>(ctx->z), P<double>(ctx->pcam_rho),
         P<double>(ctx->pcam_bb), st, GATE_RUN);
  LAUNCH(k_pcg_start, 1, BA_THREADS, 0, ctx->nblk_cam, P<double>(ctx->pcam_bb), P<double>(ctx->pcam_rho), st, GATE_RUN);
  if (ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG && ctx->opt.persistent_pcg == 1 && ctx->dist_pcg) {
    // persistent PCG with the product row-sharded over the ranks, exchange through flag-in-data slots in
    // NVLink peer memory inside the kernel (ba_kernels_dist.cuh)
    cudaMemsetAsync(ctx->pcg_bar.p, 0, 16, ctx->stream);
    PcgFan fan = ctx->fan;
    int n_cam = ctx->n_cam, n_my = ctx->n_my_rows;
    const int32_t *my_rows = P<int32_t>(ctx->my_rows), *ent_ptr = P<int32_t>(ctx->ent_ptr);
    const int2 *ent = P<int2>(ctx->ent);
    const double *Sb = P<double>(ctx->Sblk), *dsq = P<double>(ctx->dsq), *bb = P<double>(ctx->b), *Minv = P<double>(ctx->Minv);
    double *x = P<double>(ctx->x), *r = P<double>(ctx->r), *z = P<double>(ctx->z), *p0 = P<double>(ctx->p), *p1 = P<double>(ctx->p2),
           *prho = P<double>(ctx->wb_rho), *pQ = P<double>(ctx->wb_Q);
    unsigned int *bar = P<unsigned int>(ctx->pcg_bar);
    LmOptions lo = ctx->lo;
    unsigned long long *prof = getenv("BA_PCG_PROF") ? P<unsigned long long>(ctx->pcg_bar) + 8 : nullptr;
    void *args[] = {&fan, &n_cam, &n_my, &my_rows, &ent_ptr, &ent, &Sb, &dsq, &bb, &Minv, &x, &r, &z, &p0, &p1, &prho, &pQ, &bar, &lo, &st,
                    &prof};
    CK(cudaLaunchCooperativeKernel((const void *)k_pcg_sparse_dist, dim3(ctx->dist_grid), dim3(BA_THREADS), args,
                                   (size_t)BA_WARPS * BA_PCG_SMEM_PER_WARP, ctx->stream));
    ctx->launches++;
    LAUNCH(k_pcg_finish, cdiv(6 * ctx->n_cam, BA_THREADS), BA_THREADS, 0, 6 * ctx->n_cam, P<double>(ctx->x), P<double>(ctx->yc), st,
           GATE_RUN);
    int32_t h_abort = 0;
    CK(cudaMemcpyAsync(&h_abort, ctx->fan.abort_flag, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (h_abort) return fail(ctx, BA_ERR_COMM, "row-sharded PCG: a peer GPU did not deliver its slots within 4 s");
    return 0;
  }
  if (ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG && ctx->opt.persistent_pcg && ctx->pcg_grid > 0) {
    // the whole PCG solve in one cooperative launch (ba_kernels_sparse.cuh)
    cudaMemsetAsync(ctx->pcg_bar.p, 0, 16, ctx->stream);  // (profile counters at +64 accumulate over the solve)
    int n_cam = ctx->n_cam;
    const int32_t *ent_ptr = P<int32_t>(ctx->ent_ptr), *row_order = P<int32_t>(ctx->row_order);
    const int2 *ent = P<int2>(ctx->ent);
    const double *Sb = P<double>(ctx->Sblk), *dsq = P<double>(ctx->dsq), *bb = P<double>(ctx->b), *Minv = P<double>(ctx->Minv);
    double *x = P<double>(ctx->x), *r = P<double>(ctx->r), *z = P<double>(ctx->z), *p0 = P<double>(ctx->p), *p1 = P<double>(ctx->p2),
           *q = P<double>(ctx->q), *rpq = P<double>(ctx->row_pq), *prho = P<double>(ctx->wb_rho), *pQ = P<double>(ctx->wb_Q);
    unsigned int *bar = P<unsigned int>(ctx->pcg_bar);
    LmOptions lo = ctx->lo;
    unsigned long long *prof = getenv("BA_PCG_PROF") ? P<unsigned long long>(ctx->pcg_bar) + 8 : nullptr;
    void *args[] = {&n_cam, &row_order, &ent_ptr, &ent, &Sb, &dsq, &bb, &Minv, &x, &r, &z, &p0, &p1, &q, &rpq, &prho, &pQ, &bar, &lo, &st, &prof};
    const int grid = std::max(1, std::min(ctx->pcg_grid, cdiv(ctx->n_cam, BA_WARPS)));
    CK(cudaLaunchCooperativeKernel((const void *)k_pcg_sparse_persistent, dim3(grid), dim3(BA_THREADS), args,
                                   (size_t)BA_WARPS * BA_PCG_SMEM_PER_WARP, ctx->stream));
    ctx->launches++;
    LAUNCH(k_pcg_finish, cdiv(6 * ctx->n_cam, BA_THREADS), BA_THREADS, 0, 6 * ctx->n_cam, P<double>(ctx->x), P<double>(ctx->yc), st,
           GATE_RUN);
    return 0;
  }
  const int batch = std::max(1, ctx->opt.poll_interval);
  int it = 1;
  for (;;) {
    for (int k = 0; k < batch; ++k, ++it) enqueue_pcg_iteration(ctx, it);
    int rc = poll_state(ctx);
    if (rc) return rc;
    if (ctx->comm_error) return BA_ERR_COMM;
    if (ctx->h_st->pcg_done || ctx->h_st->done) break;
    if (it > ctx->lo.max_pcg + batch + 1) return fail(ctx, BA_ERR_STATE, "PCG controller did not terminate");
  }
  LAUNCH(k_pcg_finish, cdiv(6 * ctx->n_cam, BA_THREADS), BA_THREADS, 0, 6 * ctx->n_cam, P<double>(ctx->x), P<double>(ctx->yc), st,
         GATE_RUN);
  return 0;
}

// reduced system by explicit Schur complement + dense Cholesky (windowed problems)
// Blocked Cholesky, look-ahead schedule 2 (in force): three streams.
//   main  (high priority): k_chol_potrf2 with the fused prologue -- diagonal tile k brought up to date inside the kernel, so the
//         critical chain is one kernel per tile column
//   side  (high priority): k_chol_trsm2 (panel k; the tile right below the diagonal goes to the side buffer), then the update
//         of the tiles (i, k + 1), i >= k + 2
//   bulk  (low priority) : the rest of the trailing update with panel k
// Dependencies (events; [k & 1] ping-pong where a wait refers to two steps back):
//   potrf2(k) <- potrf2(k-1) [stream order], column(k-2) = the next-column update of step k - 2, bulk(k-2)
//   trsm2(k)  <- potrf2(k), column(k-1) [stream order]
//   column(k) <- trsm2(k) [stream order], bulk(k-1)
//   bulk(k)   <- trsm2(k), bulk(k-1) [stream order]
// tile rows below the diagonal of tile column k that can be non-zero: n_band rows right below, then the border rows from bord0
struct ChActive {
  int n_band, bord0, n_act;
};
static ChActive chol_active(const ba_gpu_ctx *ctx, int n, int nt, int k) {
  ChActive a;
  const int below = nt - k - 1;
  if (ctx->ex_band_cams < 0 || getenv("BA_CHOL_DENSE")) {
    a.n_band = below;
    a.bord0 = nt;
    a.n_act = below;
    return a;
  }
  const int bt = (6 * ctx->ex_band_cams + 5 + CH_NB - 1) / CH_NB;  // tile distance of the furthest camera-camera entry
  a.n_band = std::min(below, std::max(1, bt));
  const int kb = k + a.n_band;                                     // last band row
  int nb0 = nt;                                                    // first tile row that holds intrinsics columns
  if (ctx->nk) nb0 = (6 * ctx->n_free) / CH_NB;
  a.bord0 = std::max(nb0, kb + 1);
  a.n_act = a.n_band + std::max(0, nt - a.bord0);
  (void)n;
  return a;
}
static int factor_blocked_lookahead2(ba_gpu_ctx *ctx, int n, int nt, double *S, double *Linv, double *Lsub, LmState *st) {
  const size_t tile = (size_t)CH_NB * CH_NB, sm2 = (size_t)2 * CH_NB * CH_LD * 8;
  cudaStream_t A = ctx->stream, B = ctx->stream2, C = ctx->stream3;
  bool col_rec[2] = {false, false}, bulk_rec[2] = {false, false};
  ctx->pdl = !ctx->pdl_off;
  for (int k = 0; k < nt; ++k) {
    const int below = nt - k - 1, e = k & 1;
    const ChActive act = chol_active(ctx, n, nt, k);  // band-aware: only the tile rows that can be non-zero (ba_kernels_chol.cuh)
    if (col_rec[e]) CK(cudaStreamWaitEvent(A, ctx->ev_col[e], 0));    // column(k - 2)
    if (bulk_rec[e]) CK(cudaStreamWaitEvent(A, ctx->ev_bulk2[e], 0));  // bulk(k - 2)
    ctx->cur = A;
    LAUNCH(k_chol_potrf2, 1, 1024, chol_potrf2_smem_bytes(), n, S, Linv + k * tile, k, 1, st, GATE_RUN);
    if (below == 0) break;
    CK(cudaEventRecord(ctx->ev_panel, A));
    CK(cudaStreamWaitEvent(B, ctx->ev_panel, 0));
    ctx->cur = B;
    LAUNCH(k_chol_trsm2, act.n_act, 256, sm2, n, S, Linv + k * tile, Lsub + (size_t)(k + 1) * tile, k, act.n_band, act.bord0, st, GATE_RUN);
    if (act.n_act > 1) {
      CK(cudaEventRecord(ctx->ev_trsm, B));
      if (bulk_rec[e ^ 1]) CK(cudaStreamWaitEvent(B, ctx->ev_bulk2[e ^ 1], 0));  // bulk(k - 1)
      LAUNCH(k_chol_update, act.n_act - 1, 256, CH_UPD_SMEM, n, S, (const double *)(Lsub + (size_t)(k + 1) * tile), k, k, 1, act.n_band,
             act.bord0, st, GATE_RUN);
      CK(cudaEventRecord(ctx->ev_col[e], B));
      col_rec[e] = true;
      CK(cudaStreamWaitEvent(C, ctx->ev_trsm, 0));
      ctx->cur = C;
      // the rest of the trailing update: active rows without the first one (tile row k + 1), as rows from k + 2
      LAUNCH(k_chol_update, (act.n_act - 1) * act.n_act / 2, 256, CH_UPD_SMEM, n, S, (const double *)nullptr, k, k + 1, 0, act.n_band - 1,
             act.bord0, st, GATE_RUN);
      CK(cudaEventRecord(ctx->ev_bulk2[e], C));
      bulk_rec[e] = true;
    } else {
      CK(cudaEventRecord(ctx->ev_col[e], B));  // the last panel: nothing left to update, the main stream waits for the panel
      col_rec[e] = true;
    }
  }
  ctx->cur = A;
  for (int e = 0; e < 2; ++e) {
    if (col_rec[e]) CK(cudaStreamWaitEvent(A, ctx->ev_col[e], 0));
    if (bulk_rec[e]) CK(cudaStreamWaitEvent(A, ctx->ev_bulk2[e], 0));
  }
  LAUNCH(k_chol_fixup, nt - 1, 256, 0, n, S, Lsub, st, GATE_RUN);
  ctx->pdl = false;
  return 0;
}

static int solve_explicit(ba_gpu_ctx *ctx) {
  LmState *st = P<LmState>(ctx->st);
  const int n = ctx->n_red;
  if (n == 0) return 0;
  if (!ctx->sp_ref) cudaMemsetAsync(ctx->S.p, 0, (size_t)n * n * 8, ctx->stream);
  // side stream: point-block inverses (k_obs_W re-derives the inverse it needs), then -- once W is there -- borders +
  // right-hand side; main stream: W, then the camera-camera blocks (disjoint parts of S)
  fork_side(ctx);
  enqueue_point_inverse(ctx, GATE_RUN);
  fork_main(ctx);
  const int obs_w_threads = ctx->n_obs <= 64 * 2 * ctx->n_sm ? 64 : BA_THREADS;  // latency-bound on windows: spread over the SMs
  DISPATCH_D(ctx->depth, {
    LAUNCH((k_obs_W<DD>), cdiv(ctx->n_obs, obs_w_threads), obs_w_threads, 0, ctx->n_obs, P<int32_t>(ctx->pt_idx), ctx->Jc_, P<double>(ctx->V),
           P<double>(ctx->dp), P<double>(ctx->W), P<double>(ctx->WV), st, GATE_RUN);
  });
  side_after_main(ctx);
  if (ctx->sp_ref) {
    // sparse Cholesky: side stream -- camera-side vectors, then b_c, B, C and b_k by camera; main stream -- the blocks of S
    if (ctx->nk) {
      LAUNCH(k_explicit_cam_kk, ctx->nblk_item + ctx->nblk_pt, BA_THREADS, 0, ctx->nblk_item, ctx->n_items, P<BaItem>(ctx->items),
             P<int32_t>(ctx->pt_idx), P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->tg), P<double>(ctx->Wk),
             P<double>(ctx->part_ex), ctx->n_pt, P<double>(ctx->Vinv), P<double>(ctx->part_kk), st, GATE_RUN);
      LAUNCH((k_spb_assemble<4>), cdiv(ctx->n_cam * 30 + 14, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->fixed_cam,
             P<int32_t>(ctx->item_ptr), P<double>(ctx->part_ex), ctx->nblk_pt, P<double>(ctx->part_kk), P<double>(ctx->gc),
             P<double>(ctx->Uck), P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->b),
             P<double>(ctx->spb_B), P<double>(ctx->spb_kk), st, GATE_RUN);
    } else {
      LAUNCH((k_explicit_cam<0>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx),
             P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->tg), P<double>(ctx->Wk), P<double>(ctx->part_ex), st, GATE_RUN);
      LAUNCH((k_spb_assemble<0>), cdiv(ctx->n_cam * 6, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->fixed_cam,
             P<int32_t>(ctx->item_ptr), P<double>(ctx->part_ex), ctx->nblk_pt, P<double>(ctx->part_kk), P<double>(ctx->gc),
             P<double>(ctx->Uck), P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->b),
             P<double>(ctx->spb_B), P<double>(ctx->spb_kk), st, GATE_RUN);
    }
    fork_main(ctx);
    LAUNCH(k_sp_schur_planes, cdiv(ctx->n_sblk * 32, BA_THREADS), BA_THREADS, 0, ctx->n_sblk, P<int32_t>(ctx->sb_ptr),
           P<unsigned long long>(ctx->sp_pairs), P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->Sblk), st, GATE_RUN);
    LAUNCH(k_sp_add_diag, cdiv(ctx->n_cam * 36, BA_THREADS), BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->sp_diag), P<double>(ctx->U),
           P<double>(ctx->Sblk), st, GATE_RUN);
    join(ctx);
    phase_mark(ctx, BA_PHASE_SCHUR);
    // LM damping of the camera columns (b is already assembled), then factorisation, border and substitutions
    LAUNCH(k_spchol_rhs, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->item_ptr), P<double>(ctx->part6), P<double>(ctx->gc),
           P<double>(ctx->dc), P<double>(ctx->b), P<double>(ctx->dsq), st, GATE_RUN, 1);
    enqueue_spchol(ctx, GATE_RUN);
    return 0;
  }
  if (ctx->nk) {
    LAUNCH(k_explicit_cam_kk, ctx->nblk_item + ctx->nblk_pt, BA_THREADS, 0, ctx->nblk_item, ctx->n_items, P<BaItem>(ctx->items),
           P<int32_t>(ctx->pt_idx), P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->tg), P<double>(ctx->Wk),
           P<double>(ctx->part_ex), ctx->n_pt, P<double>(ctx->Vinv), P<double>(ctx->part_kk), st, GATE_RUN);
    LAUNCH((k_explicit_assemble<4>), cdiv(ctx->n_cam * 30 + 14, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->n_free, n,
           P<int32_t>(ctx->cam_slot), P<int32_t>(ctx->item_ptr), P<double>(ctx->part_ex), ctx->nblk_pt, P<double>(ctx->part_kk),
           P<double>(ctx->gc), P<double>(ctx->Uck), P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->S),
           P<double>(ctx->rhs), st, GATE_RUN);
  } else {
    LAUNCH((k_explicit_cam<0>), ctx->nblk_item, BA_THREADS, 0, ctx->n_items, P<BaItem>(ctx->items), P<int32_t>(ctx->pt_idx),
           P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->tg), P<double>(ctx->Wk), P<double>(ctx->part_ex), st, GATE_RUN);
    LAUNCH((k_explicit_assemble<0>), cdiv(ctx->n_cam * 6, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->n_free, n,
           P<int32_t>(ctx->cam_slot), P<int32_t>(ctx->item_ptr), P<double>(ctx->part_ex), ctx->nblk_pt, P<double>(ctx->part_kk),
           P<double>(ctx->gc), P<double>(ctx->Uck), P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->S),
           P<double>(ctx->rhs), st, GATE_RUN);
  }
  fork_main(ctx);
  if (ctx->n_blk <= 4 * ctx->n_sm)
    LAUNCH(k_schur_pairs<28>, ctx->n_blk, 28 * 36, 0, n, P<int32_t>(ctx->blk_i), P<int32_t>(ctx->blk_j), P<int32_t>(ctx->blk_cam),
         P<int32_t>(ctx->pair_ptr), P<int32_t>(ctx->pair_a), P<int32_t>(ctx->pair_b), P<double>(ctx->W), P<double>(ctx->WV),
         P<double>(ctx->U), P<double>(ctx->dc), P<double>(ctx->S), st, GATE_RUN);
  else
    LAUNCH(k_schur_pairs<7>, ctx->n_blk, 7 * 36, 0, n, P<int32_t>(ctx->blk_i), P<int32_t>(ctx->blk_j), P<int32_t>(ctx->blk_cam),
         P<int32_t>(ctx->pair_ptr), P<int32_t>(ctx->pair_a), P<int32_t>(ctx->pair_b), P<double>(ctx->W), P<double>(ctx->WV),
         P<double>(ctx->U), P<double>(ctx->dc), P<double>(ctx->S), st, GATE_RUN);
  join(ctx);
  if (n <= BA_LDLT2_MAX_N && !ctx->legacy_chol) {
    // single CTA, L D L^T with the trailing matrix in registers and the right-hand side as an extra row (ba_kernels_chol.cuh)
#define LDLT2_LAUNCH(NT)                                                                                                  \
  LAUNCH(k_ldlt2_solve<NT>, 1, 1024, ldlt2_smem_bytes(n), n, P<double>(ctx->S), P<double>(ctx->rhs), ctx->n_cam, ctx->n_free, \
         P<int32_t>(ctx->cam_slot), ctx->nk, P<double>(ctx->yc), P<double>(ctx->yk), st, GATE_RUN)
    switch (ldlt2_tiles(n)) {
      case 1: LDLT2_LAUNCH(1); break;
      case 2: LDLT2_LAUNCH(2); break;
      case 3: LDLT2_LAUNCH(3); break;
      case 4: LDLT2_LAUNCH(4); break;
      default: LDLT2_LAUNCH(5); break;
    }
#undef LDLT2_LAUNCH
  } else if (n <= BA_LDLT_MAX_N && ctx->legacy_chol != 1) {
    // single CTA, matrix in shared memory, L D L^T with the right-hand side as an extra row (ba_kernels_chol.cuh)
    LAUNCH(k_ldlt_solve, 1, 1024, ldlt_smem_bytes(n), n, P<double>(ctx->S), P<double>(ctx->rhs), ctx->n_cam, ctx->n_free,
           P<int32_t>(ctx->cam_slot), ctx->nk, P<double>(ctx->yc), P<double>(ctx->yk), st, GATE_RUN);
  } else if (n <= 160) {
    const size_t smem = ((size_t)n * n + n + 8) * 8;
    LAUNCH((k_cholesky_solve<1>), 1, 256, smem, n, P<double>(ctx->S), P<double>(ctx->rhs), ctx->n_cam, ctx->n_free,
           P<int32_t>(ctx->cam_slot), ctx->nk, P<double>(ctx->yc), P<double>(ctx->yk), st, GATE_RUN);
  } else {
    // blocked right-looking Cholesky (ba_kernels_chol.cuh): the reference's global BA with free intrinsics
    const int nt = cdiv(n, CH_NB);
    double *S = P<double>(ctx->S);
    double *Linv = P<double>(ctx->chol_linv);
    // one GPU: three-stream look-ahead schedule (factor_blocked_lookahead2); otherwise (sharded run, BA_NO_LOOKAHEAD=1, legacy
    // kernels) the plain right-looking sequence on the solver stream
    const bool lookahead = ctx->forking && ctx->stream2 && ctx->cur == ctx->stream && ctx->legacy_chol == 0 &&
                           getenv("BA_NO_LOOKAHEAD") == nullptr;
    if (lookahead) {
      int rcf = factor_blocked_lookahead2(ctx, n, nt, S, Linv, P<double>(ctx->chol_lsub), st);
      ctx->cur = ctx->stream;
      ctx->pdl = false;
      if (rcf) return rcf;
    }
    for (int k = 0; k < nt && !lookahead; ++k) {
      const int below = nt - k - 1;
      if (ctx->legacy_chol == 1) {
        LAUNCH(k_chol_potrf, 1, CH_NB, 0, n, S, k, st, GATE_RUN);
        LAUNCH(k_chol_trsm, below, CH_NB, (size_t)2 * CH_NB * CH_LD * 8, n, S, k, st, GATE_RUN);
      } else {
        // diagonal tile: register-resident L D L^T that also yields L^-1; panel: product with L^-1
        LAUNCH(k_chol_potrf2, 1, 1024, chol_potrf2_smem_bytes(), n, S, Linv + (size_t)k * CH_NB * CH_NB, k, 0, st, GATE_RUN);
        const ChActive act = chol_active(ctx, n, nt, k);
        LAUNCH(k_chol_trsm2, act.n_act, 256, (size_t)2 * CH_NB * CH_LD * 8, n, S, Linv + (size_t)k * CH_NB * CH_NB, (double *)nullptr, k,
               act.n_band, act.bord0, st, GATE_RUN);
        LAUNCH(k_chol_update, act.n_act * (act.n_act + 1) / 2, 256, CH_UPD_SMEM, n, S, (const double *)nullptr, k, k, 0, act.n_band,
               act.bord0, st, GATE_RUN);
        continue;
      }
      LAUNCH(k_chol_update, below * (below + 1) / 2, 256, CH_UPD_SMEM, n, S, (const double *)nullptr, k, k, 0, below, nt, st,
             GATE_RUN);
    }
    int nn = n, n_cam = ctx->n_cam, n_free = ctx->n_free, nk = ctx->nk, gate = GATE_RUN;
    const double *Sc = S, *rhs = P<double>(ctx->rhs);
    double *yc = P<double>(ctx->yc), *yk = P<double>(ctx->yk);
    const int32_t *cam_slot = P<int32_t>(ctx->cam_slot);
    if (ctx->legacy_chol == 0 && nt <= CH_S2_OWN * ctx->n_sm) {
      // substitution through the stored L_kk^-1 tiles, solved values exchanged as flag-in-data slots (k_chol_solve2)
      ChSlot *fwd = P<ChSlot>(ctx->chol_slots), *bwd = fwd + (size_t)nt * CH_NB;
      CK(cudaMemsetAsync(fwd, 0, (size_t)2 * nt * CH_NB * sizeof(ChSlot), ctx->stream));
      const double *Li = Linv;
      void *args[] = {&nn, &Sc, &Li, &rhs, &fwd, &bwd, &n_cam, &n_free, &cam_slot, &nk, &yc, &yk, &st, &gate};
      CK(cudaLaunchCooperativeKernel((const void *)k_chol_solve2, dim3(ctx->n_sm), dim3(256), args, 0, ctx->stream));
      ctx->launches++;
    } else {
      CK(cudaMemsetAsync(P<char>(ctx->chol_v) + (size_t)(n + 64) * 8, 0, 16, ctx->stream));
      double *v = P<double>(ctx->chol_v), *ztg = v + n;
      unsigned int *bar = reinterpret_cast<unsigned int *>(v + n + 64);
      void *args[] = {&nn, &Sc, &rhs, &v, &ztg, &bar, &n_cam, &n_free, &cam_slot, &nk, &yc, &yk, &st, &gate};
      CK(cudaLaunchCooperativeKernel((const void *)k_chol_solve, dim3(ctx->n_sm), dim3(256), args, 0, ctx->stream));
      ctx->launches++;
    }
  }
  return 0;
}

static int enqueue_lm_iteration(ba_gpu_ctx *ctx) {
  LmState *st = P<LmState>(ctx->st);
  const int D = ctx->depth, K = ctx->nk;
  if (ctx->solver != BA_SOLVER_EXPLICIT_CHOLESKY) enqueue_point_inverse(ctx, GATE_RUN);  // (explicit: inside solve_explicit)
  phase_mark(ctx, BA_PHASE_POINT_INVERSE);
  int rc = ctx->solver != BA_SOLVER_EXPLICIT_CHOLESKY ? solve_implicit(ctx) : solve_explicit(ctx);
  if (rc) return rc;
  phase_mark(ctx, BA_PHASE_SUBSTITUTION);
  if (ctx->fact) {
    const double *intr = P<double>(ctx->intr);
    LAUNCH(k_pack_camx, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<double>(ctx->yc), P<double>(ctx->geo), P<double>(ctx->camx), st,
           GATE_RUN);
    LAUNCH((kf_schur_pass1<1, 0>), ctx->n_tiles, BA_THREADS, 0, ctx->n_pt, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
           ctx->Fp_, P<double>(ctx->geo), P<double>(ctx->yc), P<double>(ctx->camx), P<int32_t>(ctx->tile_lo),
           P<int32_t>(ctx->tile_span), intr, P<double>(ctx->Vinv), P<double>(ctx->sp), P<double>(ctx->gp), P<double>(ctx->yp),
           P<double>(ctx->ys), st, GATE_RUN);
    LAUNCH(kf_model_cost, ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx), ctx->Fc_,
           P<double>(ctx->camx), intr, P<double>(ctx->ys), P<double>(ctx->pc_mcc), st, GATE_RUN);
  } else
  DISPATCH_DK(D, K, {
    // back-substitution y_p = V^-1 (-g_p - W^T y_c)
    LAUNCH((k_schur_pass1<DD, KK, 1>), ctx->pl_tiles, BA_THREADS, 0, ctx->n_pt, ctx->pl_tile_pts, P<int32_t>(ctx->pt_rowptr), P<int32_t>(ctx->pm_cam),
           ctx->Jp_, P<double>(ctx->yc), P<double>(ctx->yk), P<double>(ctx->Vinv), P<double>(ctx->gp), P<double>(ctx->yp), st,
           GATE_RUN, 0);
    fork_side(ctx);  // the model cost change does not depend on the candidate point
    LAUNCH((k_model_cost<DD, KK>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
           ctx->Jc_, P<double>(ctx->yc), P<double>(ctx->yp), P<double>(ctx->yk), P<double>(ctx->pc_mcc), st, GATE_RUN);
    fork_main(ctx);
  });
  if (!ctx->forking) phase_mark(ctx, BA_PHASE_BACKSUB);
  LAUNCH(k_candidate, ctx->nblk_ent, BA_THREADS, 0, ctx->n_cam, ctx->n_pt, K, ctx->fixed_cam, P<double>(ctx->pose), P<double>(ctx->pt),
         P<double>(ctx->intr), P<double>(ctx->yc), P<double>(ctx->yp), P<double>(ctx->yk), P<double>(ctx->sc), P<double>(ctx->sp),
         P<double>(ctx->sk), P<double>(ctx->pose_c), P<double>(ctx->pt_c), P<double>(ctx->intr_c), P<double>(ctx->pe_step), st,
         GATE_RUN, ctx->rank == 0 ? 1.0 : 0.0);
  DISPATCH_D(D, {
    LAUNCH((k_cost<DD>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
           P<double2>(ctx->uv), P<double>(ctx->depthv), P<double>(ctx->pose_c), P<double>(ctx->pt_c), P<double>(ctx->intr_c),
           ctx->cp, P<double>(ctx->pc_cand), st, GATE_RUN);
  });
  join(ctx);
  phase_mark(ctx, ctx->forking ? BA_PHASE_BACKSUB : BA_PHASE_CANDIDATE);
  sync_flags(ctx);
  {
    const double *const parts[3] = {P<double>(ctx->pc_mcc), P<double>(ctx->pe_step), P<double>(ctx->pc_cand)};
    const int nblks[3] = {ctx->nblk_obs, ctx->nblk_ent, ctx->nblk_obs};
    PartRef grp[3];
    reduce_scalar_group(ctx, 3, parts, nblks, 3, GATE_RUN, grp);
    const PartRef rm = grp[0], rs = grp[1], rc2 = grp[2];
    LAUNCH(k_lm_control, 1, BA_THREADS, 0, rm.n, rs.n, K, rm.p, rs.p, rc2.p, P<double>(ctx->rk), P<double>(ctx->Jkk),
           P<double>(ctx->yk), P<double>(ctx->intr_c), P<double>(ctx->intr_prior), ctx->cp.sw_intr, ctx->lo, st,
           P<BaIterRec>(ctx->trace));
  }
  phase_mark(ctx, BA_PHASE_CONTROL);
  // accepted: x <- x+, relinearise (all gated on the device-side decision)
  const bool overlap_accept = ctx->forking && !ctx->fact;  // windowed explicit path
  if (overlap_accept) fork_side(ctx);
  LAUNCH(k_accept, ctx->nblk_ent, BA_THREADS, 0, ctx->n_cam, ctx->n_pt, P<double>(ctx->pose), P<double>(ctx->pt), P<double>(ctx->intr),
         P<double>(ctx->pose_c), P<double>(ctx->pt_c), P<double>(ctx->intr_c), st, GATE_ACCEPTED);
  if (overlap_accept) fork_main(ctx);
  // (the side stream runs k_accept, then the point-major branch of the relinearisation; enqueue_linearize joins both)
  enqueue_linearize(ctx, GATE_ACCEPTED, P<double>(ctx->sc), P<double>(ctx->sp), P<double>(ctx->sk), false, overlap_accept);
  enqueue_state_norms(ctx, GATE_ACCEPTED, P<double>(ctx->sc), P<double>(ctx->sp), P<double>(ctx->sk));
  const PartRef rg = sync_flags(ctx, P<double>(ctx->pe_gmax), ctx->nblk_ent, GATE_ACCEPTED);  // flags + gradient norm: one max
  {
    const double *const parts[2] = {P<double>(ctx->pc_lin), P<double>(ctx->pe_xn)};
    const int nblks[2] = {ctx->nblk_obs, ctx->nblk_ent};
    PartRef grp[2];
    reduce_scalar_group(ctx, 2, parts, nblks, 6, GATE_ACCEPTED, grp);
    const PartRef rc3 = grp[0], rx = grp[1];
    LAUNCH(k_lm_post, 1, BA_THREADS, 0, rc3.n, rg.n, K, rc3.p, rg.p, rx.p, P<double>(ctx->rk), ctx->lo, st,
           P<BaIterRec>(ctx->trace), GATE_ACCEPTED);
  }
  phase_mark(ctx, BA_PHASE_RELINEARIZE);
  return 0;
}

extern "C" int ba_gpu_solve(ba_gpu_ctx *ctx, ba_gpu_summary *summary) {
  if (!ctx) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_solve before ba_gpu_upload");
  CK(cudaSetDevice(ctx->device));
  ctx->pdl = false;  // (an error return may have left the LM-iteration launch mode on)
  ctx->cur = ctx->stream;
  const int64_t l0 = ctx->launches;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  // windowed explicit solver on one GPU (single-CTA solve: every kernel is a small gated kernel): programmatic dependent launches
  const bool pdl = !ctx->pdl_off && ctx->solver == BA_SOLVER_EXPLICIT_CHOLESKY && !ctx->sp_ref && ctx->n_ranks == 1 && ctx->n_red > 0 &&
                   ctx->n_red <= BA_LDLT_MAX_N;
  ctx->pdl = pdl;
  ctx->ph_on = (ctx->solver != BA_SOLVER_EXPLICIT_CHOLESKY || ctx->sp_ref) && getenv("BA_NO_PHASE_TIMES") == nullptr;
  ctx->ph_n = 0;
  phase_mark(ctx, BA_PHASE_START);
  enqueue_iteration_zero(ctx);
  phase_mark(ctx, BA_PHASE_ITER0);
  ctx->pdl = false;
  const int poll = std::max(1, ctx->opt.poll_interval);
  int rc = 0;
  // windowed explicit solver on one GPU: the ~26 small kernels of an LM iteration (two streams, fork / join) are
  // captured once per upload and replayed
  const bool graphed = !ctx->lm_graph_off && ctx->solver == BA_SOLVER_EXPLICIT_CHOLESKY && !ctx->sp_ref && ctx->n_ranks == 1 &&
                       ctx->n_red > 0 && ctx->n_red <= BA_LDLT_MAX_N;
  for (int it = 1;; ++it) {
    if (graphed) {
      if (!ctx->lm_graph || ctx->lm_graph_stale) {
        const int64_t lb = ctx->launches;
        cudaGraph_t g = nullptr;
        CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        ctx->pdl = pdl;
        rc = enqueue_lm_iteration(ctx);
        ctx->pdl = false;
        const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
        ctx->lm_graph_launches = ctx->launches - lb;
        ctx->launches = lb;
        if (rc) {
          if (g) cudaGraphDestroy(g);
          return rc;
        }
        if (ce != cudaSuccess || !g) {
          if (g) cudaGraphDestroy(g);
          return fail(ctx, BA_ERR_CUDA, "LM iteration graph capture: %s", cudaGetErrorString(ce));
        }
        if (ctx->lm_graph) {  // same topology, new sizes / pointers: update in place
          cudaGraphExecUpdateResultInfo info;
          if (cudaGraphExecUpdate(ctx->lm_graph, g, &info) != cudaSuccess) {
            cudaGetLastError();  // topology changed (e.g. another cost model): rebuild
            drop_lm_graph(ctx);
          }
        }
        cudaError_t ie = cudaSuccess;
        if (!ctx->lm_graph) ie = cudaGraphInstantiate(&ctx->lm_graph, g, 0);
        cudaGraphDestroy(g);
        if (ie != cudaSuccess) return fail(ctx, BA_ERR_CUDA, "LM iteration graph instantiate: %s", cudaGetErrorString(ie));
        ctx->lm_graph_stale = false;
      }
      CK(cudaGraphLaunch(ctx->lm_graph, ctx->stream));
      ctx->launches += ctx->lm_graph_launches;
    } else {
      ctx->pdl = pdl;
      rc = enqueue_lm_iteration(ctx);
      ctx->pdl = false;
      if (rc) return rc;
    }
    // The launch-per-step PCG loops on the host (it polls the PCG controller itself) and the row-sharded PCG reads its abort
    // flag after every solve; every other path takes all decisions on the device, so the host only looks at the controller
    // state every poll_interval iterations and keeps the launch queue full in between (a host synchronisation per LM
    // iteration left the GPU idle while the ~60 launches of the next iteration were being enqueued).
    const bool host_in_loop = ctx->solver == BA_SOLVER_IMPLICIT_PCG ||
                              (ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG && !ctx->spchol &&
                               (ctx->dist_pcg || !(ctx->opt.persistent_pcg && ctx->pcg_grid > 0)));
    if (!host_in_loop && (it % poll) != 0 && it <= ctx->lo.max_num_iterations) continue;
    rc = poll_state(ctx);
    if (rc) return rc;
    if (ctx->h_st->done) break;
    if (it > ctx->lo.max_num_iterations + 2) return fail(ctx, BA_ERR_STATE, "LM controller did not terminate");
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  CK(cudaGetLastError());
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  phase_collect(ctx);
  ctx->ph_on = false;
  const LmState &h = *ctx->h_st;
  ba_gpu_summary s;
  memset(&s, 0, sizeof(s));
  s.termination = h.termination;
  s.num_iterations = h.iter > 0 ? (h.termination == BA_TERM_NO_CONVERGENCE || h.termination == BA_TERM_GRADIENT ||
                                           h.termination == BA_TERM_MIN_RADIUS
                                       ? h.iter - 1
                                       : h.iter)
                                : 0;
  s.num_successful = h.num_successful;
  s.num_unsuccessful = h.num_unsuccessful;
  s.initial_cost = h.initial_cost;
  s.final_cost = h.x_cost;
  s.total_linear_iters = h.total_lin_iters;
  s.solver_used = ctx->spchol ? BA_SOLVER_SPARSE_SCHUR_CHOLESKY : ctx->solver;
  s.reduced_dim = ctx->n_red;
  s.solve_ms = ms;
  s.kernel_launches = ctx->launches - l0;
  const int nt = std::min(h.n_trace, ctx->lo.trace_cap);
  ctx->h_trace.resize(nt);
  if (nt) CK(cudaMemcpy(ctx->h_trace.data(), ctx->trace.p, (size_t)nt * sizeof(BaIterRec), cudaMemcpyDeviceToHost));
  ctx->last_summary = s;
  if (summary) *summary = s;
  if (getenv("BA_SPCHOL_PROF") && ctx->spchol) {
    unsigned long long pr[8];
    cudaMemcpy(pr, ctx->spc_prof.p, 64, cudaMemcpyDeviceToHost);
    cudaMemset(ctx->spc_prof.p, 0, 64);
    const double n = (double)std::max<unsigned long long>(1, pr[4]);
    fprintf(stderr, "[BA_SPCHOL_PROF] us per factor launch (thread block 0, %llu launches): assemble S %.2f | extend-add %.2f | factor loop %.2f | "
                    "write panel %.2f\n", pr[4], pr[0] / n / 1e3, pr[1] / n / 1e3, pr[2] / n / 1e3, pr[3] / n / 1e3);
  }
  if (getenv("BA_PCG_PROF") && ctx->pcg_bar.p && ctx->solver == BA_SOLVER_SPARSE_SCHUR_PCG) {
    unsigned long long pr[6];
    cudaMemcpy(pr, P<unsigned long long>(ctx->pcg_bar) + 8, 48, cudaMemcpyDeviceToHost);
    cudaMemset(P<unsigned long long>(ctx->pcg_bar) + 8, 0, 48);
    const double n = (double)std::max<int64_t>(1, s.total_linear_iters);
    fprintf(stderr, "[BA_PCG_PROF] us/iteration (CTA 0): product %.2f | barrier %.2f | sum+alpha %.2f | update %.2f | barrier %.2f | reset+controller %.2f\n",
            pr[0] / n / 1e3, pr[1] / n / 1e3, pr[2] / n / 1e3, pr[3] / n / 1e3, pr[4] / n / 1e3, pr[5] / n / 1e3);
  }
  if (h.termination == BA_TERM_FAILURE && h.n_trace <= 1 && h.eval_fail)
    return fail(ctx, BA_ERR_NUMERIC, "non-finite cost or Jacobian at the initial point");
  return BA_OK;
}

extern "C" int ba_gpu_phase_times(const ba_gpu_ctx *ctx, double ms[BA_PHASE_COUNT]) {
  if (!ctx || !ms) return BA_ERR_INVALID;
  for (int k = 0; k < BA_PHASE_COUNT; ++k) ms[k] = ctx->ph_ms[k];
  return BA_OK;
}
extern "C" const char *ba_gpu_phase_name(int32_t phase) { return phase >= 0 && phase < BA_PHASE_COUNT ? g_phase_names[phase] : ""; }

extern "C" int ba_gpu_get_trace(ba_gpu_ctx *ctx, ba_gpu_iter *out, int32_t cap) {
  if (!ctx || (!out && cap > 0)) return BA_ERR_INVALID;
  const int n = std::min<int>(cap, (int)ctx->h_trace.size());
  static_assert(sizeof(ba_gpu_iter) == sizeof(BaIterRec), "trace record layout");
  if (n > 0) memcpy(out, ctx->h_trace.data(), (size_t)n * sizeof(BaIterRec));
  return n;
}

extern "C" int ba_gpu_download(ba_gpu_ctx *ctx, double *pose7, double *pt3, double intr4[4]) {
  if (!ctx) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_download before ba_gpu_upload");
  CK(cudaSetDevice(ctx->device));
  if (pose7) CK(cudaMemcpyAsync(pose7, ctx->pose.p, (size_t)ctx->n_cam * 56, cudaMemcpyDeviceToHost, ctx->stream));
  if (pt3 && ctx->n_pt) CK(cudaMemcpyAsync(pt3, ctx->pt.p, (size_t)ctx->n_pt * 24, cudaMemcpyDeviceToHost, ctx->stream));
  if (intr4) CK(cudaMemcpyAsync(intr4, ctx->intr.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BA_OK;
}

// ------------------------------------------------------------------ test hooks
extern "C" int ba_gpu_eval(ba_gpu_ctx *ctx, double *r, double *Jc, double *Jp, double *Jk, double *cost, double *g_c,
                           double *g_p, double *g_k) {
  if (!ctx) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_eval before ba_gpu_upload");
  CK(cudaSetDevice(ctx->device));
  LmState *st = P<LmState>(ctx->st);
  {
    int rcp = ensure_planes(ctx);
    if (rcp) return rcp;
  }
  LAUNCH(k_lm_init, 1, 1, 0, st, ctx->opt.initial_trust_region_radius);
  enqueue_linearize(ctx, GATE_RUN, P<double>(ctx->one_c), P<double>(ctx->one_p), P<double>(ctx->one_k), /*force_planes=*/true);
  ctx->linearized = false;
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  const size_t n = ctx->n_obs;
  const int R = 2 + ctx->depth;
  std::vector<double> h(n * 2 + 1);
  auto get2 = [&](const double2 *src) -> int {
    if (n) CK(cudaMemcpy(h.data(), src, n * 16, cudaMemcpyDeviceToHost));
    return 0;
  };
  auto get1 = [&](const double *src) -> int {
    if (n) CK(cudaMemcpy(h.data(), src, n * 8, cudaMemcpyDeviceToHost));
    return 0;
  };
  int rc;
  const JPlanes &J = ctx->Jc_;
  if (r) {
    if ((rc = get2(J.r))) return rc;
    for (size_t i = 0; i < n; ++i) {
      r[i * R] = h[2 * i];
      r[i * R + 1] = h[2 * i + 1];
    }
    if (ctx->depth) {
      if ((rc = get1(J.r3))) return rc;
      for (size_t i = 0; i < n; ++i) r[i * R + 2] = h[i];
    }
  }
  if (Jc)
    for (int k = 0; k < 6; ++k) {
      if ((rc = get2(J.Jc[k]))) return rc;
      for (size_t i = 0; i < n; ++i) {
        Jc[(i * R + 0) * 6 + k] = h[2 * i];
        Jc[(i * R + 1) * 6 + k] = h[2 * i + 1];
      }
      if (ctx->depth) {
        if ((rc = get1(J.Jc3[k]))) return rc;
        for (size_t i = 0; i < n; ++i) Jc[(i * R + 2) * 6 + k] = h[i];
      }
    }
  if (Jp)
    for (int k = 0; k < 3; ++k) {
      if ((rc = get2(J.Jp[k]))) return rc;
      for (size_t i = 0; i < n; ++i) {
        Jp[(i * R + 0) * 3 + k] = h[2 * i];
        Jp[(i * R + 1) * 3 + k] = h[2 * i + 1];
      }
      if (ctx->depth) {
        if ((rc = get1(J.Jp3[k]))) return rc;
        for (size_t i = 0; i < n; ++i) Jp[(i * R + 2) * 3 + k] = h[i];
      }
    }
  if (Jk) {
    memset(Jk, 0, n * 8 * sizeof(double));
    if (ctx->nk)
      for (int k = 0; k < 2; ++k) {
        if ((rc = get2(J.Jk[k]))) return rc;
        for (size_t i = 0; i < n; ++i) {
          Jk[(i * 2 + 0) * 4 + 2 * k] = h[2 * i];          // row0: fx (k=0) / cx (k=1) column
          Jk[(i * 2 + 1) * 4 + 2 * k + 1] = h[2 * i + 1];  // row1: fy / cy column
        }
      }
  }
  if (cost) {
    std::vector<double> pc(ctx->nblk_obs + 1);
    if (ctx->nblk_obs) CK(cudaMemcpy(pc.data(), ctx->pc_lin.p, (size_t)ctx->nblk_obs * 8, cudaMemcpyDeviceToHost));
    double c = 0.0;
    for (int i = 0; i < ctx->nblk_obs; ++i) c += pc[i];
    if (ctx->nk) {
      double rk[4];
      CK(cudaMemcpy(rk, ctx->rk.p, 32, cudaMemcpyDeviceToHost));
      double s = 0.0;
      for (int k = 0; k < 4; ++k) s += rk[k] * rk[k];
      c = 0.5 * s + c;
    }
    *cost = c;
  }
  if (g_c) CK(cudaMemcpy(g_c, ctx->gc.p, (size_t)ctx->n_cam * 48, cudaMemcpyDeviceToHost));
  if (g_p && ctx->n_pt) CK(cudaMemcpy(g_p, ctx->gp.p, (size_t)ctx->n_pt * 24, cudaMemcpyDeviceToHost));
  if (g_k) {
    memset(g_k, 0, 32);
    if (ctx->nk) CK(cudaMemcpy(g_k, ctx->gk.p, 32, cudaMemcpyDeviceToHost));
  }
  if ((rc = poll_state(ctx))) return rc;
  if (ctx->h_st->eval_fail) return fail(ctx, BA_ERR_NUMERIC, "non-finite residual or Jacobian");
  return BA_OK;
}

extern "C" int ba_gpu_get_indices(ba_gpu_ctx *ctx, int32_t *perm_pt_major, int32_t *pt_rowptr, int32_t *cam_rowptr) {
  if (!ctx) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_get_indices before ba_gpu_upload");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  if (perm_pt_major && ctx->n_obs) CK(cudaMemcpy(perm_pt_major, ctx->perm.p, (size_t)ctx->n_obs * 4, cudaMemcpyDeviceToHost));
  if (pt_rowptr) CK(cudaMemcpy(pt_rowptr, ctx->pt_rowptr.p, ((size_t)ctx->n_pt + 1) * 4, cudaMemcpyDeviceToHost));
  if (cam_rowptr) CK(cudaMemcpy(cam_rowptr, ctx->cam_rowptr.p, ((size_t)ctx->n_cam + 1) * 4, cudaMemcpyDeviceToHost));
  return BA_OK;
}

__global__ void k_set_radius(LmState *st, double radius) { st->radius = radius; }

// brings the device to "linearised at the current point" with a given radius:
// iteration zero (scaling included) + damped point-block inverses
static int prepare_linear_system(ba_gpu_ctx *ctx, double radius) {
  enqueue_iteration_zero(ctx, false);
  LmState *st = P<LmState>(ctx->st);
  LAUNCH(k_set_radius, 1, 1, 0, st, radius);
  enqueue_point_inverse(ctx, GATE_RUN);
  enqueue_sparse_values(ctx, GATE_RUN);
  int rc = poll_state(ctx);
  if (rc) return rc;
  if (ctx->h_st->eval_fail) return fail(ctx, BA_ERR_NUMERIC, "non-finite residual or Jacobian");
  if (ctx->h_st->lin_fail) return fail(ctx, BA_ERR_NUMERIC, "singular point block");
  return 0;
}
__global__ void k_clear_done(LmState *st) {
  st->done = 0;
  st->pcg_done = 0;
  st->pcg_it = 1;
}

extern "C" int ba_gpu_schur_matvec(ba_gpu_ctx *ctx, double radius, const double *x, double *y) {
  if (!ctx || !x || !y) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_schur_matvec before ba_gpu_upload");
  if (ctx->nk) return fail(ctx, BA_ERR_UNSUPPORTED, "implicit Schur product needs optimize_intrinsics = 0");
  if (ctx->sp_ref) return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_schur_matvec with the sparse Cholesky needs NS mode");
  CK(cudaSetDevice(ctx->device));
  ctx->sp_full_next = true;  // (the product needs every block of S on every rank)
  int rc = prepare_linear_system(ctx, radius);
  if (rc) return rc;
  LmState *st = P<LmState>(ctx->st);
  LAUNCH(k_clear_done, 1, 1, 0, st);
  const size_t n = (size_t)6 * ctx->n_cam;
  std::vector<double> sc(n), xs(n);
  CK(cudaMemcpy(sc.data(), ctx->sc.p, n * 8, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) xs[i] = x[i] / sc[i];
  CK(cudaMemcpyAsync(ctx->p.p, xs.data(), n * 8, cudaMemcpyHostToDevice, ctx->stream));
  const ItemRef mv = enqueue_matvec(ctx, P<double>(ctx->p), GATE_RUN);
  LAUNCH(k_pcg_q, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, mv.ptr, mv.part, P<double>(ctx->dc),
         P<double>(ctx->p), P<double>(ctx->q), P<double>(ctx->pcam_pq), st, GATE_RUN);
  CK(cudaMemcpyAsync(xs.data(), ctx->q.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  for (size_t i = 0; i < n; ++i) y[i] = xs[i] / sc[i];
  return BA_OK;
}

// y = (S + D^2)^-1 rhs by the sparse Cholesky of the last upload (test hook; un-scaled coordinates like ba_gpu_schur_matvec)
extern "C" int ba_gpu_schur_solve(ba_gpu_ctx *ctx, double radius, const double *rhs, double *y) {
  if (!ctx || !rhs || !y) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_schur_solve before ba_gpu_upload");
  if (!ctx->spchol) return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_schur_solve needs the sparse Cholesky solver");
  if (ctx->sp_ref) return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_schur_solve needs NS mode (no depth prior, fixed intrinsics)");
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_linear_system(ctx, radius);
  if (rc) return rc;
  LmState *st = P<LmState>(ctx->st);
  LAUNCH(k_clear_done, 1, 1, 0, st);
  const size_t n = (size_t)6 * ctx->n_cam;
  std::vector<double> sc(n), bs(n);
  CK(cudaMemcpy(sc.data(), ctx->sc.p, n * 8, cudaMemcpyDeviceToHost));
  // S_unscaled = diag(1/sc) S_scaled diag(1/sc):  S_scaled (y / sc) = sc .* rhs
  for (size_t i = 0; i < n; ++i) bs[i] = rhs[i] * sc[i];
  CK(cudaMemcpyAsync(ctx->b.p, bs.data(), n * 8, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(k_spchol_rhs, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->ident), P<double>(ctx->part6), P<double>(ctx->gc),
         P<double>(ctx->dc), P<double>(ctx->b), P<double>(ctx->dsq), st, GATE_RUN, 1);
  enqueue_spchol(ctx, GATE_RUN);
  CK(cudaMemcpyAsync(bs.data(), ctx->yc.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if ((rc = poll_state(ctx))) return rc;
  CK(cudaGetLastError());
  if (ctx->h_st->lin_fail) return fail(ctx, BA_ERR_NUMERIC, "sparse Cholesky: non-positive pivot");
  for (size_t i = 0; i < n; ++i) y[i] = bs[i] * sc[i];
  return BA_OK;
}

// ------------------------------------------------------------------ covariance
// structure of ba_gpu_covariance, once per upload: under another solver (dense explicit, matrix-free PCG) the block structure and the symbolic tree
// that solver = 4 builds (the sp_ref branch of the upload); then the selected-inversion queue, the block -> front records and
// the scratch buffers.  Growing buffers a captured LM-iteration graph may point at marks that graph stale.
static int cov_prepare(ba_gpu_ctx *ctx) {
  if (ctx->cov_ready) return 0;
  cudaStream_t s = ctx->stream;
  int rc;
  if (!ctx->sp_ref) {
    ctx->lm_graph_stale = true;
    if ((rc = build_sparse_structure(ctx))) return rc;
    ctx->spc_nrhs = ctx->nk ? 5 : 1;
    rc = build_spchol(ctx);
    ctx->spchol = false;  // (the LM solve of this context stays the dense explicit one)
    if (rc == BA_ERR_UNSUPPORTED) {
      const std::string why = ctx->err;
      return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_covariance: %s", why.c_str());
    }
    if (rc) return rc;
    const size_t nc = (size_t)ctx->n_cam;
    RES(W, ((size_t)ctx->n_obs + 1) * 144);  // (the matrix-free PCG, AUTO on a large DEPTH problem, has no per-observation W)
    RES(WV, ((size_t)ctx->n_obs + 1) * 144);
    RES(spb_B, nc * 192 + 64);
    RES(spb_Z, nc * 192 + 64);
    RES(spb_kk, 20 * 8);
    RES(spb_part, (size_t)(ctx->nblk_cam + 1) * 14 * 8);
  }
  const SpSymbolic &S = ctx->sym;
  auto N_ = [&](int id, int f) { return S.node[(size_t)id * SPSYM_NODE_INTS + f]; };
  // queue: levels top-down; per level the prepare items, the product tiles (more per node where the level has few nodes), the
  // finish items
  std::vector<int32_t> q, tiles((size_t)S.n_nodes, 0);
  size_t smem = 0;
  for (int l = S.n_levels - 1; l >= 0; --l) {
    const int nodes = S.level_ptr[l + 1] - S.level_ptr[l];
    const int t_lvl = std::max(1, std::min(8, ctx->n_sm / std::max(1, nodes)));
    for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
      const int id = S.level_nodes[e];
      tiles[id] = N_(id, SPN_NB) > 0 ? t_lvl : 0;
      smem = std::max(smem, si_smem(N_(id, SPN_M), N_(id, SPN_NB)));
      q.push_back(id);
      q.push_back(-1);
    }
    for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
      const int id = S.level_nodes[e];
      for (int t = 0; t < tiles[id]; ++t) {
        q.push_back(id);
        q.push_back(t);
      }
    }
    for (int e = S.level_ptr[l]; e < S.level_ptr[l + 1]; ++e) {
      q.push_back(S.level_nodes[e]);
      q.push_back(-3);
    }
  }
  if (smem > 227 * 1024) return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_covariance: a front does not fit shared memory (%zu bytes)", smem);
  // stored block of S -> (node, local row, local column, flags: 1 transposed, 2 diagonal) from the entry table
  std::vector<int32_t> brec((size_t)ctx->n_sblk * 4 + 4, 0);
  for (int id = 0; id < S.n_nodes; ++id)
    for (int e = N_(id, SPN_AENT); e < N_(id, SPN_AENT) + N_(id, SPN_NAENT); ++e) {
      const uint32_t code = (uint32_t)S.aent[4 * (size_t)e];
      const uint32_t blk = code & 0x3fffffffu;
      if (blk == 0x3fffffffu) continue;
      if ((int)blk >= ctx->n_sblk) return fail(ctx, BA_ERR_STATE, "ba_gpu_covariance: inconsistent entry table");
      int32_t *r = brec.data() + 4 * (size_t)blk;
      r[0] = id;
      r[1] = S.aent[4 * (size_t)e + 1];
      r[2] = S.aent[4 * (size_t)e + 2];
      r[3] = (code & 0x80000000u ? 1 : 0) | (code & 0x40000000u ? 2 : 0);
    }
  auto up = [&](Buf &b, const std::vector<int32_t> &v) -> int {
    int rc2 = buf_reserve(ctx, b, (v.size() + 1) * 4);
    if (rc2) return rc2;
    if (!v.empty()) CK(cudaMemcpyAsync(b.p, v.data(), v.size() * 4, cudaMemcpyHostToDevice, s));
    return 0;
  };
  if ((rc = up(ctx->cov_queue, q)) || (rc = up(ctx->cov_tiles, tiles)) || (rc = up(ctx->cov_brec, brec)) || (rc = up(ctx->cov_pos, S.pos)))
    return rc;
  ctx->cov_n_items = (int)(q.size() / 2);
  ctx->cov_smem = smem;
  CK(cudaFuncSetAttribute(k_selinv_tree, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const size_t nc = (size_t)ctx->n_cam;
  RES(cov_Y, ((size_t)S.panel_blocks + 1) * 288);
  RES(cov_X, (4 * nc + 1) * 48);
  RES(cov_zq, (nc + 1) * 48);
  RES(cov_yscr, (nc + 1) * 48);
  RES(cov_Tinv, 16 * 8);
  RES(cov_S, ((size_t)ctx->n_sblk + 1) * 288);
  RES(cov_ck, (nc + 1) * 192);
  RES(cov_cnt, ((size_t)3 * S.n_nodes + 16) * 4);
  RES(cov_cam, nc * 288);
  RES(cov_ci, nc * 192);
  RES(cov_pt, ((size_t)ctx->n_pt + 1) * 72);
  RES(cov_bad, 16);
  RES(cov_piv, sizeof(CovPivots));
  CK(cudaStreamSynchronize(s));  // (host vectors die here)
  ctx->cov_ready = true;
  return 0;
}

extern "C" int ba_gpu_covariance(ba_gpu_ctx *ctx, double *cov_cam, double *cov_cam_intr, double cov_intr[4 * 4], double *cov_pt,
                                 int32_t n_pairs, const int32_t *cam_a, const int32_t *cam_b, double *cov_pairs) {
  if (!ctx) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_covariance before ba_gpu_upload");
  if (ctx->n_ranks > 1) return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_covariance is single-GPU");
  if (!ctx->depth)
    return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_covariance needs the depth prior: without it (%s cost) the scale is free and the "
                "Gauss-Newton Hessian is singular", ctx->nk ? "INTR" : "NS");
  if (ctx->fixed_cam < 0)
    return fail(ctx, BA_ERR_UNSUPPORTED, "ba_gpu_covariance needs a fixed camera: with fixed_cam < 0 the gauge is free and the "
                "Gauss-Newton Hessian is singular");
  if (n_pairs < 0 || (n_pairs > 0 && (!cam_a || !cam_b || !cov_pairs))) return fail(ctx, BA_ERR_INVALID, "bad camera pair list");
  for (int i = 0; i < n_pairs; ++i)
    if (cam_a[i] < 0 || cam_a[i] >= ctx->n_cam || cam_b[i] < 0 || cam_b[i] >= ctx->n_cam)
      return fail(ctx, BA_ERR_INVALID, "camera pair %d (%d, %d) out of range", i, cam_a[i], cam_b[i]);
  CK(cudaSetDevice(ctx->device));
  ctx->pdl = false;
  ctx->cur = ctx->stream;
  int rc = cov_prepare(ctx);
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  LmState *st = P<LmState>(ctx->st);
  const SpSymbolic &S = ctx->sym;
  const size_t nc = (size_t)ctx->n_cam;
  // linearisation at the current point, radius +inf: every LM damping D = sqrt(diag / radius) is exactly 0 (the next
  // ba_gpu_solve starts from k_lm_init)
  enqueue_iteration_zero(ctx, false);
  LAUNCH(k_clear_done, 1, 1, 0, st);
  LAUNCH(k_set_radius, 1, 1, 0, st, INFINITY);
  enqueue_point_inverse(ctx, GATE_RUN);
  CovPivots *cp = P<CovPivots>(ctx->cov_piv);
  LAUNCH(k_cov_pivots_init, 1, 1, 0, cp, st);
  DISPATCH_D(ctx->depth, {
    LAUNCH((k_obs_W<DD>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->pt_idx), ctx->Jc_, P<double>(ctx->V),
           P<double>(ctx->dp), P<double>(ctx->W), P<double>(ctx->WV), st, GATE_RUN);
  });
  if (ctx->nk) {
    LAUNCH(k_explicit_cam_kk, ctx->nblk_item + ctx->nblk_pt, BA_THREADS, 0, ctx->nblk_item, ctx->n_items, P<BaItem>(ctx->items),
           P<int32_t>(ctx->pt_idx), P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->tg), P<double>(ctx->Wk),
           P<double>(ctx->part_ex), ctx->n_pt, P<double>(ctx->Vinv), P<double>(ctx->part_kk), st, GATE_RUN);
    LAUNCH((k_spb_assemble<4>), cdiv(ctx->n_cam * 30 + 14, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->fixed_cam,
           P<int32_t>(ctx->item_ptr), P<double>(ctx->part_ex), ctx->nblk_pt, P<double>(ctx->part_kk), P<double>(ctx->gc),
           P<double>(ctx->Uck), P<double>(ctx->Ukk), P<double>(ctx->gk), P<double>(ctx->dk), P<double>(ctx->b),
           P<double>(ctx->spb_B), P<double>(ctx->spb_kk), st, GATE_RUN);
  }
  LAUNCH(k_sp_schur_planes, cdiv(ctx->n_sblk * 32, BA_THREADS), BA_THREADS, 0, ctx->n_sblk, P<int32_t>(ctx->sb_ptr),
         P<unsigned long long>(ctx->sp_pairs), P<double>(ctx->W), P<double>(ctx->WV), P<double>(ctx->Sblk), st, GATE_RUN);
  LAUNCH(k_sp_add_diag, cdiv(ctx->n_cam * 36, BA_THREADS), BA_THREADS, 0, ctx->n_cam, P<int32_t>(ctx->sp_diag), P<double>(ctx->U),
         P<double>(ctx->Sblk), st, GATE_RUN);
  // no damping; the fixed camera (no block of S, no border row) gets a unit pivot so that the tree can eliminate it
  CK(cudaMemsetAsync(ctx->dsq.p, 0, nc * 48, s));
  LAUNCH(k_fill, 1, 32, 0, P<double>(ctx->dsq) + 6 * (size_t)ctx->fixed_cam, (size_t)6, 1.0);
  // factorisation (forward substitution: Z = L^-1 B with the border)
  SpChol a = spchol_args(ctx);
  if (ctx->spc_tree && ctx->spc_parts == 1) {
    SpTree t;
    int *cnt = P<int>(ctx->spc_cnt);
    t.tiles = P<int32_t>(ctx->spc_tiles);
    t.fdone = cnt + 16;
    t.udone = t.fdone + S.n_nodes;
    t.sdone = t.udone + S.n_nodes;
    CK(cudaMemcpyAsync(cnt, ctx->spc_cnt_init.p, ((size_t)3 * S.n_nodes + 16) * 4, cudaMemcpyDeviceToDevice, s));
    const size_t smem = std::max(std::max(ctx->spc_smem_factor, ctx->spc_smem_solve), ctx->spc_smem_update);
    t.queue = P<int2>(ctx->spc_queue);
    t.n_items = ctx->spc_qB;
    t.ticket = cnt;
    if (ctx->spc_nrhs > 1)
      LAUNCH((k_spchol_tree<5>), std::min(ctx->n_sm, t.n_items), SPC_THREADS, smem, a, t, st, GATE_RUN);
    else
      LAUNCH((k_spchol_tree<1>), std::min(ctx->n_sm, t.n_items), SPC_THREADS, smem, a, t, st, GATE_RUN);
  } else {
    for (int l = 0; l < S.n_levels; ++l) {
      const int nodes = S.level_ptr[l + 1] - S.level_ptr[l];
      if (ctx->spc_nrhs > 1)
        LAUNCH((k_spchol_factor<5>), nodes, SPC_THREADS, ctx->spc_smem_factor, a, S.level_ptr[l], st, GATE_RUN);
      else
        LAUNCH((k_spchol_factor<1>), nodes, SPC_THREADS, ctx->spc_smem_factor, a, S.level_ptr[l], st, GATE_RUN);
      if (l + 1 < S.n_levels) {
        const int tiles = std::max(1, std::min(8, ctx->n_sm / std::max(1, nodes)));
        if (ctx->spc_nrhs > 1)
          LAUNCH((k_spchol_update<5>), nodes * tiles, SPU_THREADS, ctx->spc_smem_update, a, S.level_ptr[l], tiles, st, GATE_RUN);
        else
          LAUNCH((k_spchol_update<1>), nodes * tiles, SPU_THREADS, ctx->spc_smem_update, a, S.level_ptr[l], tiles, st, GATE_RUN);
      }
    }
  }
  LAUNCH(k_cov_pivots, cdiv(6 * ctx->n_cam, BA_THREADS), BA_THREADS, 0, ctx->n_cam, a.perm, P<int32_t>(ctx->sp_diag), a.S, a.dsq,
         a.linv, BA_COV_MIN_PIVOT_RATIO, cp);
  // intrinsics border: T^-1, then X = L^-T Z one column at a time (the backward substitution of the LM step, levels top-down)
  const double *X = nullptr;
  if (ctx->nk) {
    LAUNCH(k_spb_reduce, ctx->nblk_cam, BA_THREADS, 0, ctx->n_cam, P<double>(ctx->spb_Z), P<double>(ctx->spc_z),
           P<double>(ctx->spb_part), st, GATE_RUN);
    LAUNCH(k_cov_border, 1, 32, 0, ctx->nblk_cam, P<double>(ctx->spb_part), P<double>(ctx->spb_kk), P<double>(ctx->cov_Tinv),
           BA_COV_MIN_PIVOT_RATIO, cp, st);
    SpChol ax = a;
    ax.Zb = nullptr;
    ax.yk = nullptr;
    ax.z = P<double>(ctx->cov_zq);
    ax.yc = P<double>(ctx->cov_yscr);
    for (int qc = 0; qc < 4; ++qc) {
      LAUNCH(k_cov_zcol, cdiv(6 * ctx->n_cam, BA_THREADS), BA_THREADS, 0, 6 * ctx->n_cam, qc, P<double>(ctx->spb_Z), P<double>(ctx->cov_zq));
      ax.ypos = P<double>(ctx->cov_X) + (size_t)qc * 6 * nc;
      for (int l = S.n_levels - 1; l >= 0; --l)
        LAUNCH(k_spchol_solve, S.level_ptr[l + 1] - S.level_ptr[l], SPC_THREADS, ctx->spc_smem_solve, ax, S.level_ptr[l], st, GATE_RUN);
    }
    X = P<double>(ctx->cov_X);
  }
  // selected inversion of A on the pattern of L (overwrites the panels and the update-matrix slots)
  {
    SelInv si;
    si.node = a.node;
    si.rel = a.rel;
    si.linv = a.linv;
    si.panel = a.panel;
    si.U = a.U;
    si.Y = P<double>(ctx->cov_Y);
    si.queue = P<int2>(ctx->cov_queue);
    si.n_items = ctx->cov_n_items;
    si.tiles = P<int32_t>(ctx->cov_tiles);
    int *cnt = P<int>(ctx->cov_cnt);
    si.ticket = cnt;
    si.pdone = cnt + 16;
    si.tdone = si.pdone + S.n_nodes;
    si.sdone = si.tdone + S.n_nodes;
    CK(cudaMemsetAsync(cnt, 0, ((size_t)3 * S.n_nodes + 16) * 4, s));
    LAUNCH(k_selinv_tree, std::min(ctx->n_sm, si.n_items), SPC_THREADS, ctx->cov_smem, si);
  }
  // Sigma on the stored blocks of S (+ border correction), per camera, pairs, points
  LAUNCH(k_cov_blocks, cdiv(ctx->n_sblk * 36, BA_THREADS), BA_THREADS, 0, ctx->n_sblk, P<int4>(ctx->cov_brec), P<int32_t>(ctx->sb_i),
         P<int32_t>(ctx->sb_j), a.node, a.panel, P<int32_t>(ctx->cov_pos), ctx->n_cam, X, P<double>(ctx->cov_Tinv), P<double>(ctx->cov_S));
  LAUNCH(k_cov_cam, cdiv(ctx->n_cam * 60, BA_THREADS), BA_THREADS, 0, ctx->n_cam, ctx->fixed_cam, ctx->nk, P<int32_t>(ctx->sp_diag),
         P<double>(ctx->cov_S), P<int32_t>(ctx->cov_pos), X, P<double>(ctx->cov_Tinv), P<double>(ctx->sc), P<double>(ctx->sk),
         P<double>(ctx->cov_ck), P<double>(ctx->cov_cam), P<double>(ctx->cov_ci));
  CK(cudaMemsetAsync(ctx->cov_bad.p, 0, 16, s));
  if (n_pairs > 0) {
    RES(cov_pin, (size_t)n_pairs * 8 + 16);
    RES(cov_pout, (size_t)n_pairs * 288 + 16);
    CK(cudaMemcpyAsync(ctx->cov_pin.p, cam_a, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(P<int32_t>(ctx->cov_pin) + n_pairs, cam_b, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
    LAUNCH(k_cov_pairs, cdiv(n_pairs * 36, BA_THREADS), BA_THREADS, 0, n_pairs, P<int32_t>(ctx->cov_pin),
           P<int32_t>(ctx->cov_pin) + n_pairs, ctx->fixed_cam, P<int32_t>(ctx->ent_ptr), P<int2>(ctx->ent), P<double>(ctx->cov_S),
           P<double>(ctx->sc), P<double>(ctx->cov_pout), P<int>(ctx->cov_bad));
  }
  if (cov_pt && ctx->n_pt > 0)
    LAUNCH(k_cov_points, ctx->nblk_pt, BA_THREADS, 0, ctx->n_pt, ctx->fixed_cam, ctx->nk, P<int32_t>(ctx->pt_rowptr),
           P<int32_t>(ctx->pm_cam), P<int32_t>(ctx->perm), P<double>(ctx->W), P<double>(ctx->Wk), P<double>(ctx->Vinv),
           P<int32_t>(ctx->ent_ptr), P<int2>(ctx->ent), P<double>(ctx->cov_S), P<double>(ctx->cov_ck), P<double>(ctx->cov_Tinv),
           P<double>(ctx->sp), P<double>(ctx->cov_pt));
  if ((rc = poll_state(ctx))) return rc;
  CK(cudaGetLastError());
  if (ctx->h_st->eval_fail) return fail(ctx, BA_ERR_NUMERIC, "ba_gpu_covariance: non-finite residual or Jacobian");
  CovPivots piv;
  CK(cudaMemcpy(&piv, cp, sizeof(piv), cudaMemcpyDeviceToHost));
  memcpy(&ctx->cov_ratio[0], &piv.min_cam, 8);
  memcpy(&ctx->cov_ratio[1], &piv.min_border, 8);
  if (!ctx->nk) ctx->cov_ratio[1] = 0.0;
  if (piv.bad_point)
    return fail(ctx, BA_ERR_NUMERIC, "ba_gpu_covariance: the Hessian is singular: the 3x3 block of a point is singular (a point "
                "without observations, or one its observations do not fix)");
  if (piv.first_bad) {
    const int k = ctx->n_cam - piv.first_bad;
    return fail(ctx, BA_ERR_NUMERIC, "ba_gpu_covariance: the Hessian is rank-deficient: a pivot of camera %d (elimination position "
                "%d) is below %g times its diagonal (a camera its observations do not fix, or cameras not connected to the fixed one)",
                S.perm[k], k, BA_COV_MIN_PIVOT_RATIO);
  }
  if (piv.bad_border)
    return fail(ctx, BA_ERR_NUMERIC, "ba_gpu_covariance: the Hessian is rank-deficient: intrinsics pivot %d is below %g times its "
                "diagonal (the observations do not fix the intrinsics)", piv.bad_border - 1, BA_COV_MIN_PIVOT_RATIO);
  if (ctx->h_st->lin_fail) return fail(ctx, BA_ERR_NUMERIC, "ba_gpu_covariance: non-positive pivot (the Hessian is not positive definite)");
  int bad = 0;
  CK(cudaMemcpy(&bad, ctx->cov_bad.p, 4, cudaMemcpyDeviceToHost));
  if (bad) return fail(ctx, BA_ERR_INVALID, "ba_gpu_covariance: a requested camera pair shares no point (outside the pattern of S)");
  if (cov_cam) CK(cudaMemcpy(cov_cam, ctx->cov_cam.p, nc * 288, cudaMemcpyDeviceToHost));
  if (cov_cam_intr) CK(cudaMemcpy(cov_cam_intr, ctx->cov_ci.p, nc * 192, cudaMemcpyDeviceToHost));
  if (cov_pt && ctx->n_pt > 0) CK(cudaMemcpy(cov_pt, ctx->cov_pt.p, (size_t)ctx->n_pt * 72, cudaMemcpyDeviceToHost));
  if (n_pairs > 0) CK(cudaMemcpy(cov_pairs, ctx->cov_pout.p, (size_t)n_pairs * 288, cudaMemcpyDeviceToHost));
  if (cov_intr) {
    double ti[16] = {0.0}, sk[4] = {0.0};
    if (ctx->nk) {
      CK(cudaMemcpy(ti, ctx->cov_Tinv.p, 128, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(sk, ctx->sk.p, 32, cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) cov_intr[4 * i + j] = ti[4 * i + j] * (sk[i] * sk[j]);
  }
  return BA_OK;
}

extern "C" int ba_gpu_covariance_pivots(const ba_gpu_ctx *ctx, double ratio[2]) {
  if (!ctx || !ratio) return BA_ERR_INVALID;
  ratio[0] = ctx->cov_ratio[0];
  ratio[1] = ctx->cov_ratio[1];
  return BA_OK;
}

extern "C" int ba_gpu_spchol_info(const ba_gpu_ctx *ctx, int64_t info[24]) {
  if (!ctx || !info) return BA_ERR_INVALID;
  memset(info, 0, 24 * sizeof(int64_t));
  if (!ctx->uploaded || !ctx->spchol) return BA_OK;
  const SpSymbolic &s = ctx->sym;
  info[0] = s.n_cam; info[1] = s.n_nodes; info[2] = s.n_levels; info[3] = s.panel_blocks; info[4] = s.u_blocks;
  info[5] = s.max_front_blocks; info[6] = s.max_m; info[7] = s.max_nb; info[8] = s.max_children;
  info[9] = (int64_t)s.flops; info[10] = (int64_t)s.crit_blocks; info[11] = (int64_t)(ctx->sym_ms * 1e3);
  info[12] = ctx->spc_parts; info[13] = ctx->spc_dist ? 1 : 0; info[14] = ctx->spc_n_topcams; info[15] = (int64_t)(ctx->spc_xchg * 8); info[16] = ctx->spc_dist ? ctx->spc_nx : 0;
  return BA_OK;
}

__global__ void k_se3_plus(int n, const double *__restrict__ pose, const double *__restrict__ delta, double *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double T[7], d[6], o[7];
  for (int k = 0; k < 7; ++k) T[k] = pose[7 * (size_t)i + k];
  for (int k = 0; k < 6; ++k) d[k] = delta[6 * (size_t)i + k];
  se3_plus(T, d, o);
  for (int k = 0; k < 7; ++k) out[7 * (size_t)i + k] = o[k];
}

extern "C" int ba_gpu_se3_plus(ba_gpu_ctx *ctx, int32_t n, const double *pose7, const double *delta6, double *out7) {
  if (!ctx || n < 0 || (n > 0 && (!pose7 || !delta6 || !out7))) return BA_ERR_INVALID;
  if (n == 0) return BA_OK;
  CK(cudaSetDevice(ctx->device));
  double *d = nullptr;
  CK(cudaMalloc(&d, (size_t)n * 20 * 8));
  double *dp = d, *dd = d + (size_t)7 * n, *dout = dd + (size_t)6 * n;
  cudaMemcpyAsync(dp, pose7, (size_t)n * 56, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(dd, delta6, (size_t)n * 48, cudaMemcpyHostToDevice, ctx->stream);
  LAUNCH(k_se3_plus, cdiv(n, 256), 256, 0, n, dp, dd, dout);
  cudaMemcpyAsync(out7, dout, (size_t)n * 56, cudaMemcpyDeviceToHost, ctx->stream);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  cudaFree(d);
  if (e != cudaSuccess) return fail(ctx, BA_ERR_CUDA, "se3_plus: %s", cudaGetErrorString(e));
  return BA_OK;
}

// ------------------------------------------------------------------ back-projection (SURVEY.md 8f, row N3)
// The step right before BA in the reference: getLocalPoints3D (src/Map3D.cpp:76-97) turns every key
// point into a camera-frame point from the depth image, addNewLandmark (:44) moves it to the world
// frame with the key frame's pose.  One thread per key point; explicit _rn intrinsics so that no FMA
// contraction changes a bit relative to the reference's plain C++ (Eigen _transformVector order).
__device__ __forceinline__ void cross_rn(const double a[3], const double b[3], double o[3]) {
  o[0] = __dsub_rn(__dmul_rn(a[1], b[2]), __dmul_rn(a[2], b[1]));
  o[1] = __dsub_rn(__dmul_rn(a[2], b[0]), __dmul_rn(a[0], b[2]));
  o[2] = __dsub_rn(__dmul_rn(a[0], b[1]), __dmul_rn(a[1], b[0]));
}
__global__ void __launch_bounds__(BA_THREADS)
k_backproject(int n, const float2 *__restrict__ uv, const float *__restrict__ depth, int width, int height, double fx, double fy,
              double cx, double cy, const double *__restrict__ pose7, double *__restrict__ local3, double *__restrict__ world3,
              int32_t *err) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i >= n) return;
  const float2 p = uv[i];
  const double u = (double)p.x, v = (double)p.y;
  const int col = (int)truncf(p.x), row = (int)truncf(p.y);  // depth_frame.at<float>(trunc(v), trunc(u))
  if (col < 0 || col >= width || row < 0 || row >= height) {
    atomicOr(err, 1);
    return;
  }
  const double z = (double)depth[(size_t)row * width + col];
  const double l[3] = {__ddiv_rn(__dmul_rn(z, __dsub_rn(u, cx)), fx), __ddiv_rn(__dmul_rn(z, __dsub_rn(v, cy)), fy), z};
  if (local3) {
    local3[3 * (size_t)i] = l[0];
    local3[3 * (size_t)i + 1] = l[1];
    local3[3 * (size_t)i + 2] = l[2];
  }
  if (world3) {
    // T * p = q._transformVector(p) + t: uv = 2 (q.vec x p); p + w uv + q.vec x uv
    const double q[3] = {pose7[0], pose7[1], pose7[2]}, w = pose7[3];
    double t2[3], c3[3];
    cross_rn(q, l, t2);
#pragma unroll
    for (int k = 0; k < 3; ++k) t2[k] = __dadd_rn(t2[k], t2[k]);
    cross_rn(q, t2, c3);
#pragma unroll
    for (int k = 0; k < 3; ++k)
      world3[3 * (size_t)i + k] = __dadd_rn(__dadd_rn(__dadd_rn(l[k], __dmul_rn(w, t2[k])), c3[k]), pose7[4 + k]);
  }
}

extern "C" int ba_gpu_backproject(ba_gpu_ctx *ctx, int32_t n, const float *uv2f, const float *depth_img, int32_t width, int32_t height,
                                  const double intr4[4], const double *pose7, double *local3, double *world3) {
  if (!ctx || n < 0 || width <= 0 || height <= 0 || !intr4 || (n > 0 && (!uv2f || !depth_img)) || (world3 && !pose7))
    return fail(ctx, BA_ERR_INVALID, "backproject: bad arguments");
  if (n == 0) return BA_OK;
  CK(cudaSetDevice(ctx->device));
  const size_t img = (size_t)width * height;
  RES(bp_buf, (size_t)n * 8 + img * 4 + 64 + (size_t)n * 48 + 64);
  char *base = P<char>(ctx->bp_buf);
  float2 *d_uv = reinterpret_cast<float2 *>(base);
  float *d_img = reinterpret_cast<float *>(base + (size_t)n * 8);
  size_t off = ((size_t)n * 8 + img * 4 + 63) / 64 * 64;
  double *d_pose = reinterpret_cast<double *>(base + off);
  double *d_local = d_pose + 8, *d_world = d_local + 3 * (size_t)n;
  cudaStream_t s = ctx->stream;
  RES(err_flag_bp, 16);
  CK(cudaMemsetAsync(ctx->err_flag_bp.p, 0, 16, s));
  CK(cudaMemcpyAsync(d_uv, uv2f, (size_t)n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_img, depth_img, img * 4, cudaMemcpyHostToDevice, s));
  if (pose7) CK(cudaMemcpyAsync(d_pose, pose7, 56, cudaMemcpyHostToDevice, s));
  LAUNCH(k_backproject, cdiv(n, BA_THREADS), BA_THREADS, 0, n, d_uv, d_img, width, height, intr4[0], intr4[1], intr4[2], intr4[3],
         d_pose, local3 ? d_local : (double *)nullptr, world3 ? d_world : (double *)nullptr, P<int32_t>(ctx->err_flag_bp));
  int32_t h_err = 0;
  if (local3) CK(cudaMemcpyAsync(local3, d_local, (size_t)n * 24, cudaMemcpyDeviceToHost, s));
  if (world3) CK(cudaMemcpyAsync(world3, d_world, (size_t)n * 24, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&h_err, ctx->err_flag_bp.p, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  if (h_err) return fail(ctx, BA_ERR_INVALID, "backproject: a key point lies outside the %d x %d depth image", width, height);
  return BA_OK;
}

// ------------------------------------------------------------------ measurement hooks
__global__ void k_flush(double *p, size_t n, double v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

extern "C" int ba_gpu_time_kernel(ba_gpu_ctx *ctx, int32_t which, int32_t warmup, int32_t iters, int32_t flush_l2,
                                  float *ms_avg) {
  if (!ctx || !ms_avg || iters <= 0 || warmup < 0) return BA_ERR_INVALID;
  if (!ctx->uploaded) return fail(ctx, BA_ERR_STATE, "ba_gpu_time_kernel before ba_gpu_upload");
  if (which < BA_KERNEL_LINEARIZE || which > BA_KERNEL_SCHUR_PASS2) return fail(ctx, BA_ERR_INVALID, "unknown kernel id");
  if (which != BA_KERNEL_LINEARIZE && ctx->nk) return fail(ctx, BA_ERR_UNSUPPORTED, "matvec needs optimize_intrinsics = 0");
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_linear_system(ctx, ctx->opt.initial_trust_region_radius);
  if (rc) return rc;
  LmState *st = P<LmState>(ctx->st);
  LAUNCH(k_clear_done, 1, 1, 0, st);
  if (which != BA_KERNEL_LINEARIZE) {
    // t must hold a finite pass-1 result before a pass-2-only timing
    CK(cudaMemcpyAsync(ctx->p.p, ctx->gc.p, (size_t)ctx->n_cam * 48, cudaMemcpyDeviceToDevice, ctx->stream));
    enqueue_matvec(ctx, P<double>(ctx->p), GATE_RUN, 7);
  }
  const size_t flush_n = (size_t)512 * 1024 * 1024 / 8;  // 512 MiB > 126 MB L2
  if (flush_l2) RES(flush, flush_n * 8);
  auto one = [&]() {
    if (which == BA_KERNEL_LINEARIZE && ctx->fact) {
      LAUNCH((kf_linearize<1>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx), P<int32_t>(ctx->pt_idx),
             P<double2>(ctx->uv), P<double>(ctx->pose), P<double>(ctx->pt), P<double>(ctx->intr), ctx->cp, ctx->Fc_,
             P<double>(ctx->pc_lin), st, GATE_RUN);
    } else if (which == BA_KERNEL_LINEARIZE) {
      DISPATCH_DK(ctx->depth, ctx->nk, {
        LAUNCH((k_linearize<DD, KK, 1>), ctx->nblk_obs, BA_THREADS, 0, ctx->n_obs, P<int32_t>(ctx->cam_idx),
               P<int32_t>(ctx->pt_idx), P<double2>(ctx->uv), P<double>(ctx->depthv), P<double>(ctx->pose), P<double>(ctx->pt),
               P<double>(ctx->intr), P<double>(ctx->sc), P<double>(ctx->sp), P<double>(ctx->sk), ctx->cp, ctx->Jc_,
               P<double>(ctx->pc_lin), st, GATE_RUN);
      });
    } else {
      enqueue_matvec(ctx, P<double>(ctx->p), GATE_RUN,
                     which == BA_KERNEL_SCHUR_PASS1 ? 1 : (which == BA_KERNEL_SCHUR_PASS2 ? 2 : 3));
    }
  };
  for (int i = 0; i < warmup; ++i) one();
  double total = 0.0;
  if (flush_l2) {
    for (int i = 0; i < iters; ++i) {
      k_flush<<<1184, 256, 0, ctx->stream>>>(P<double>(ctx->flush), flush_n, (double)i);
      CK(cudaEventRecord(ctx->ev0, ctx->stream));
      one();
      CK(cudaEventRecord(ctx->ev1, ctx->stream));
      CK(cudaEventSynchronize(ctx->ev1));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
      total += ms;
    }
  } else {
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    for (int i = 0; i < iters; ++i) one();
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    total = ms;
  }
  CK(cudaGetLastError());
  *ms_avg = (float)(total / iters);
  return BA_OK;
}

// ------------------------------------------------------------------ multi-GPU
extern "C" int ba_gpu_comm_unique_id(char id128[128]) {
  std::string err;
  if (!id128) return BA_ERR_INVALID;
  if (!nccl_load(&err)) return fail(nullptr, BA_ERR_COMM, "%s", err.c_str());
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != 0) return fail(nullptr, BA_ERR_COMM, "ncclGetUniqueId: %d", r);
  memcpy(id128, id.internal, 128);
  return BA_OK;
}

extern "C" int ba_gpu_comm_init(ba_gpu_ctx *ctx, const char id128[128], int32_t rank, int32_t n_ranks) {
  if (!ctx || !id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return BA_ERR_INVALID;
  std::string err;
  if (!nccl_load(&err)) return fail(ctx, BA_ERR_COMM, "%s", err.c_str());
  CK(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(id.internal, id128, 128);
  if (ctx->comm && g_nccl.CommDestroy) {  // re-initialisation: release the previous communicator
    cudaStreamSynchronize(ctx->stream);
    g_nccl.CommDestroy(ctx->comm);
    ctx->comm = nullptr;
  }
  ncclResult_t r = g_nccl.CommInitRank(&ctx->comm, n_ranks, id, rank);
  if (r != 0) return fail(ctx, BA_ERR_COMM, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  ctx->rank = rank;
  ctx->n_ranks = n_ranks;
  return BA_OK;
}

// ------------------------------------------------------------------ device-resident keyframe / landmark store (SURVEY 8f, N1)
// Host bookkeeping of ba_kernels_store.cuh: one observation pool (keyframe segments in container order), world poses by
// keyframe, world points by landmark id.  Not thread-safe; lives on the stream of its solver context.
struct ba_store {
  ba_gpu_ctx *ctx = nullptr;
  struct DBuf {
    void *p = nullptr;
    size_t cap = 0;
  };
  DBuf lm, uvf, depth;              // observation pool
  size_t pool_used = 0;
  std::vector<long long> seg_off;   // per keyframe: first slot in the pool, -1 = never set
  std::vector<int32_t> seg_n, seg_cap;
  DBuf pose_w, pt_w, first;         // [kf * 7], [id * 3], [id]
  size_t n_kf_cap = 0, n_lm_cap = 0;
  DBuf stage, win_off, win_seg, flag, pos, isfirst, rank, w_cam, w_pt, w_uv, w_depth, w_pose, w_pt3, w_lm, T0, out_pose, out_pt, cub, cnt;
  std::vector<DBuf *> all;
  double ms[3] = {0, 0, 0};         // last window: enumeration + index build, solve, write-back + copies
  int max_id = -1;                  // largest landmark id any keyframe list refers to
  unsigned long long epoch = 0;     // window counter (stamps the first-appearance table)
  // pinned staging of the host -> device copies (a pageable source costs ~40 us per copy at these sizes); a slice is reused
  // only after the stream has been synchronised (window_solve ends with one)
  char *pin = nullptr;
  size_t pin_cap = 0, pin_used = 0;
};
// copies `bytes` from the caller's array to device memory through the pinned staging area (asynchronous; the caller's
// array is free on return)
static int store_h2d(ba_gpu_ctx *ctx, ba_store *st, void *dst, const void *src, size_t bytes) {
  if (bytes == 0) return 0;
  const size_t need = st->pin_used + ((bytes + 63) / 64) * 64;
  if (need > st->pin_cap) {
    // no room: drain the copies in flight, then start over (and grow if one request alone does not fit)
    CK(cudaStreamSynchronize(ctx->stream));
    st->pin_used = 0;
    if (((bytes + 63) / 64) * 64 > st->pin_cap) {
      if (st->pin) cudaFreeHost(st->pin);
      st->pin = nullptr;
      st->pin_cap = std::max(((bytes + 63) / 64) * 64 * 4, (size_t)1 << 20);
      CK(cudaMallocHost((void **)&st->pin, st->pin_cap));
    }
  }
  char *stage = st->pin + st->pin_used;
  st->pin_used += ((bytes + 63) / 64) * 64;
  memcpy(stage, src, bytes);
  CK(cudaMemcpyAsync(dst, stage, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}
static int sgrow(ba_gpu_ctx *ctx, ba_store *st, ba_store::DBuf &b, size_t bytes, bool keep) {
  if (b.cap >= bytes) return 0;
  // growing tables (keep = true: observation pool, pose / landmark tables) start at 32 MiB and double: a reallocation
  // (cudaMalloc + copy + cudaFree) was measured at up to 200 ms on this driver, so it must stay a rare event; the scratch
  // buffers of a window settle at the window size
  const size_t want = keep ? std::max(bytes * 2, (size_t)32 << 20) : std::max(bytes + bytes / 2, (size_t)65536);
  void *np = nullptr;
  cudaError_t e = cudaMalloc(&np, want);
  if (e != cudaSuccess) return fail(ctx, BA_ERR_CUDA, "store: cudaMalloc(%zu): %s", want, cudaGetErrorString(e));
  if (keep && b.p && b.cap) {
    cudaMemcpyAsync(np, b.p, b.cap, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
  }
  if (b.p) cudaFree(b.p);
  b.p = np;
  b.cap = want;
  if (std::find(st->all.begin(), st->all.end(), &b) == st->all.end()) st->all.push_back(&b);
  return 0;
}
#define SGROW(buf, bytes, keep)                              \
  do {                                                       \
    int rc_ = sgrow(ctx, st, st->buf, (size_t)(bytes), keep); \
    if (rc_) return rc_;                                     \
  } while (0)
#define BA_STORE_MAX_ID (1 << 24)

extern "C" int ba_store_create(ba_gpu_ctx *ctx, ba_store **out) {
  if (!ctx || !out) return BA_ERR_INVALID;
  ba_store *st = new ba_store();
  st->ctx = ctx;
  *out = st;
  return BA_OK;
}
extern "C" void ba_store_destroy(ba_store *st) {
  if (!st) return;
  if (st->ctx) {
    cudaSetDevice(st->ctx->device);
    if (st->ctx->stream) cudaStreamSynchronize(st->ctx->stream);
  }
  for (ba_store::DBuf *b : st->all)
    if (b->p) cudaFree(b->p);
  if (st->pin) cudaFreeHost(st->pin);
  delete st;
}
// forget every keyframe / landmark (the device buffers are kept: allocating them again costs far more than a window)
extern "C" int ba_store_clear(ba_store *st) {
  if (!st) return BA_ERR_INVALID;
  ba_gpu_ctx *ctx = st->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  std::fill(st->seg_off.begin(), st->seg_off.end(), -1);
  std::fill(st->seg_n.begin(), st->seg_n.end(), 0);
  st->pool_used = 0;
  st->pin_used = 0;
  st->max_id = -1;
  return BA_OK;
}
static int store_fit_kf(ba_gpu_ctx *ctx, ba_store *st, int kf) {
  if ((size_t)kf >= st->seg_off.size()) {
    const size_t n = (size_t)kf + 1 + st->seg_off.size() / 2;
    st->seg_off.resize(n, -1);
    st->seg_n.resize(n, 0);
    st->seg_cap.resize(n, 0);
  }
  if ((size_t)kf >= st->n_kf_cap) {
    const size_t n = (size_t)kf + 64 + st->n_kf_cap / 2;
    SGROW(pose_w, n * 56, true);
    st->n_kf_cap = n;
  }
  return 0;
}
// the observation lists of n_kf keyframes (kf[k] has cnt[k] entries, lists back to back) in the iteration order of their
// global_points_map; replaces any earlier list of these keyframes.  The lists of one call go to one contiguous piece at the
// end of the pool: three copies per call, whatever the number of keyframes.  Earlier segments of the same keyframes are
// abandoned, not reclaimed: a keyframe's map is re-sent once or twice in its life (it grows only while it is one of the two
// newest keyframes, src/Map3D.cpp:52-53), so the pool holds at most a small multiple of the live lists.
extern "C" int ba_store_set_keyframes(ba_store *st, int32_t n_kf, const int32_t *kf, const int32_t *cnt, const int32_t *landmark_id,
                                      const float *uv2f, const double *depth) {
  if (!st || n_kf < 0 || (n_kf > 0 && (!kf || !cnt))) return BA_ERR_INVALID;
  if (n_kf == 0) return BA_OK;
  ba_gpu_ctx *ctx = st->ctx;
  CK(cudaSetDevice(ctx->device));
  size_t total = 0;
  int kf_max = 0;
  for (int k = 0; k < n_kf; ++k) {
    if (kf[k] < 0 || cnt[k] < 0) return BA_ERR_INVALID;
    total += (size_t)cnt[k];
    kf_max = std::max(kf_max, kf[k]);
  }
  if (total > 0 && (!landmark_id || !uv2f || !depth)) return BA_ERR_INVALID;
  for (size_t i = 0; i < total; ++i) {
    if (landmark_id[i] < 0 || landmark_id[i] >= BA_STORE_MAX_ID)
      return fail(ctx, BA_ERR_UNSUPPORTED, "store: landmark id %d outside [0, 2^24)", landmark_id[i]);
    st->max_id = std::max(st->max_id, landmark_id[i]);
  }
  int rc = store_fit_kf(ctx, st, kf_max);
  if (rc) return rc;
  const size_t need = st->pool_used + total;
  SGROW(lm, need * 4, true);
  SGROW(uvf, need * 8, true);
  SGROW(depth, need * 8, true);
  size_t o = st->pool_used;
  for (int k = 0; k < n_kf; ++k) {
    st->seg_off[kf[k]] = (long long)o;
    st->seg_n[kf[k]] = cnt[k];
    o += (size_t)cnt[k];
  }
  if (total) {
    if ((rc = store_h2d(ctx, st, (int32_t *)st->lm.p + st->pool_used, landmark_id, total * 4)) ||
        (rc = store_h2d(ctx, st, (float2 *)st->uvf.p + st->pool_used, uv2f, total * 8)) ||
        (rc = store_h2d(ctx, st, (double *)st->depth.p + st->pool_used, depth, total * 8)))
      return rc;
  }
  st->pool_used = need;
  return BA_OK;
}
extern "C" int ba_store_set_keyframe(ba_store *st, int32_t kf, int32_t n, const int32_t *landmark_id, const float *uv2f,
                                     const double *depth) {
  return ba_store_set_keyframes(st, 1, &kf, &n, landmark_id, uv2f, depth);
}
extern "C" int ba_store_set_poses(ba_store *st, int32_t kf0, int32_t n, const double *pose7) {
  if (!st || kf0 < 0 || n <= 0 || !pose7) return BA_ERR_INVALID;
  ba_gpu_ctx *ctx = st->ctx;
  CK(cudaSetDevice(ctx->device));
  int rc = store_fit_kf(ctx, st, kf0 + n - 1);
  if (rc) return rc;
  return store_h2d(ctx, st, (double *)st->pose_w.p + 7 * (size_t)kf0, pose7, (size_t)n * 56);
}
extern "C" int ba_store_set_landmarks(ba_store *st, int32_t n, const int32_t *id, const double *xyz) {
  if (!st || n < 0 || (n > 0 && (!id || !xyz))) return BA_ERR_INVALID;
  if (n == 0) return BA_OK;
  ba_gpu_ctx *ctx = st->ctx;
  CK(cudaSetDevice(ctx->device));
  int mx = 0;
  for (int i = 0; i < n; ++i) {
    if (id[i] < 0 || id[i] >= BA_STORE_MAX_ID) return fail(ctx, BA_ERR_UNSUPPORTED, "store: landmark id %d outside [0, 2^24)", id[i]);
    mx = std::max(mx, id[i]);
  }
  if ((size_t)mx >= st->n_lm_cap) {
    const size_t cap = (size_t)mx + 1024 + st->n_lm_cap / 2;
    SGROW(pt_w, cap * 24, true);
    SGROW(first, cap * 8, false);  // (epoch << 32 | ~position) per landmark: zero = older than any window
    CK(cudaMemsetAsync(st->first.p, 0, st->first.cap, ctx->stream));
    st->n_lm_cap = cap;
  }
  const size_t id_bytes = (((size_t)n * 4 + 63) / 64) * 64;
  SGROW(stage, id_bytes + (size_t)n * 24, false);
  int32_t *d_id = (int32_t *)st->stage.p;
  double *d_xyz = (double *)((char *)st->stage.p + id_bytes);
  cudaStream_t s = ctx->stream;
  int rch;
  if ((rch = store_h2d(ctx, st, d_id, id, (size_t)n * 4)) || (rch = store_h2d(ctx, st, d_xyz, xyz, (size_t)n * 24))) return rch;
  ks_scatter_points<<<cdiv(n, BA_THREADS), BA_THREADS, 0, s>>>(n, d_id, d_xyz, (double *)st->pt_w.p);
  ctx->launches++;
  return BA_OK;
}

// windowOptimize on the resident data (src/OptimizationUtils.cpp:215-313): enumeration of the admissible observations of
// keyframes kf_i..kf_f in canonical order, change into the frame of keyframe kf_i, solve with the context's options (REF
// cost: depth prior + free intrinsics are the caller's choice through ba_gpu_set_options), write-back into the world frame.
//   intr4: in = current intrinsics, out = optimised;  pose7_out [n_cam * 7] world poses;  landmark_of_pt / pt3_out: the
//   window's landmarks in order of first appearance and their optimised world points (capacity lm_cap).
// The store's own poses / points are only touched after a successful solve.
extern "C" int ba_store_window_solve(ba_store *st, int32_t kf_i, int32_t kf_f, const double intr_prior4[4], double intr4[4],
                                     ba_gpu_summary *summary, double *pose7_out, int32_t lm_cap, int32_t *n_pt_out,
                                     int32_t *landmark_of_pt, double *pt3_out, int32_t *n_obs_out, double ms_out[3]) {
  if (!st || kf_i < 0 || kf_f < kf_i || !intr4 || !pose7_out || !n_pt_out || (lm_cap > 0 && (!landmark_of_pt || !pt3_out)))
    return BA_ERR_INVALID;
  ba_gpu_ctx *ctx = st->ctx;
  CK(cudaSetDevice(ctx->device));
  const int n_cam = kf_f - kf_i + 1;
  if ((size_t)kf_f >= st->seg_off.size()) return fail(ctx, BA_ERR_STATE, "store: keyframe %d was never set", kf_f);
  const auto t_begin = std::chrono::steady_clock::now();
  std::vector<int32_t> off((size_t)n_cam + 1, 0);
  std::vector<long long> seg((size_t)n_cam, 0);
  for (int k = 0; k < n_cam; ++k) {
    if (st->seg_off[kf_i + k] < 0) return fail(ctx, BA_ERR_STATE, "store: keyframe %d was never set", kf_i + k);
    seg[k] = st->seg_off[kf_i + k];
    off[k + 1] = off[k] + st->seg_n[kf_i + k];
  }
  const int total = off[n_cam];
  if (st->max_id >= 0 && (size_t)st->max_id >= st->n_lm_cap)  // (the reference would throw from map.at, :270)
    return fail(ctx, BA_ERR_STATE, "store: a keyframe refers to landmark %d, which was never set", st->max_id);
  cudaStream_t s = ctx->stream;
  SGROW(win_off, ((size_t)n_cam + 1) * 4, false);
  SGROW(win_seg, (size_t)n_cam * 8, false);
  SGROW(flag, ((size_t)total + 2) * 8, false);  // packed (admissible | first appearance << 32)
  SGROW(pos, ((size_t)total + 2) * 8, false);   // its exclusive scan
  SGROW(w_cam, ((size_t)total + 1) * 4, false);
  SGROW(w_pt, ((size_t)total + 1) * 4, false);
  SGROW(w_uv, ((size_t)total + 1) * 16, false);
  SGROW(w_depth, ((size_t)total + 1) * 8, false);
  SGROW(w_lm, ((size_t)total + 1) * 4, false);
  SGROW(w_pt3, ((size_t)total + 1) * 24, false);
  SGROW(w_pose, (size_t)n_cam * 56, false);
  SGROW(T0, 14 * 8, false);
  SGROW(out_pose, (size_t)n_cam * 56, false);
  SGROW(cnt, 64, false);
  {
    int rch;
    if ((rch = store_h2d(ctx, st, st->win_off.p, off.data(), ((size_t)n_cam + 1) * 4)) ||
        (rch = store_h2d(ctx, st, st->win_seg.p, seg.data(), (size_t)n_cam * 8)))
      return rch;
  }
  const int32_t *d_off = (const int32_t *)st->win_off.p;
  const long long *d_seg = (const long long *)st->win_seg.p;
  unsigned long long *d_packed = (unsigned long long *)st->flag.p, *d_prefix = (unsigned long long *)st->pos.p;
  const int nb = cdiv(total + 1, BA_THREADS);
  const unsigned long long epoch = ++st->epoch;
  double *d_T0 = (double *)st->T0.p, *d_T0inv = d_T0 + 7;
  ks_frame<<<cdiv(std::max(n_cam, 1), 64), 64, 0, s>>>(n_cam, (const double *)st->pose_w.p + 7 * (size_t)kf_i, d_T0, d_T0inv, (double *)st->w_pose.p);
  ks_mark<<<nb, BA_THREADS, 0, s>>>(total, n_cam, d_off, d_seg, (const double *)st->depth.p, (const int32_t *)st->lm.p, epoch,
                                    (unsigned long long *)st->first.p, d_packed);
  ks_isfirst<<<nb, BA_THREADS, 0, s>>>(total, n_cam, d_off, d_seg, (const int32_t *)st->lm.p, epoch, (const unsigned long long *)st->first.p,
                                       d_packed);
  {
    size_t tb = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_packed, d_prefix, total + 1, s));
    int rcs = sgrow(ctx, st, st->cub, tb + 16, false);
    if (rcs) return rcs;
    CK(cub::DeviceScan::ExclusiveSum(st->cub.p, tb, d_packed, d_prefix, total + 1, s));
  }
  unsigned long long h_counts = 0;
  CK(cudaMemcpyAsync(&h_counts, d_prefix + total, 8, cudaMemcpyDeviceToHost, s));
  ks_emit<<<nb, BA_THREADS, 0, s>>>(total, n_cam, d_off, d_seg, d_packed, d_prefix, (const int32_t *)st->lm.p, (const float2 *)st->uvf.p,
                                    (const double *)st->depth.p, (const unsigned long long *)st->first.p, (const double *)st->pt_w.p, d_T0inv,
                                    (int32_t *)st->w_cam.p, (int32_t *)st->w_pt.p, (double2 *)st->w_uv.p, (double *)st->w_depth.p,
                                    (int32_t *)st->w_lm.p, (double *)st->w_pt3.p);
  ctx->launches += 4;
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  st->pin_used = 0;  // every staged copy has landed
  int rc;
  const int32_t h_cnt[2] = {(int32_t)(h_counts & 0xffffffffull), (int32_t)(h_counts >> 32)};
  const int n_obs = h_cnt[0];
  const int n_pt = h_cnt[1];
  if (n_obs_out) *n_obs_out = n_obs;
  *n_pt_out = n_pt;
  if (n_pt > lm_cap) return fail(ctx, BA_ERR_INVALID, "store: %d landmarks in the window, caller's capacity %d", n_pt, lm_cap);
  ctx->src_on_device = true;
  rc = ba_gpu_upload(ctx, n_cam, (const double *)st->w_pose.p, 0, n_pt, (const double *)st->w_pt3.p, n_obs, (const int32_t *)st->w_cam.p,
                     (const int32_t *)st->w_pt.p, (const double *)st->w_uv.p, (const double *)st->w_depth.p, intr4, intr_prior4);
  ctx->src_on_device = false;
  if (rc) return rc;
  st->ms[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
  auto t_ph = std::chrono::steady_clock::now();
  rc = ba_gpu_solve(ctx, summary);
  if (rc) return rc;
  st->ms[1] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_ph).count();
  t_ph = std::chrono::steady_clock::now();
  SGROW(out_pt, ((size_t)n_pt + 1) * 24, false);
  ks_writeback<<<cdiv(n_cam + n_pt, BA_THREADS), BA_THREADS, 0, s>>>(n_cam, n_pt, d_T0, P<double>(ctx->pose), P<double>(ctx->pt),
                                                                    (const int32_t *)st->w_lm.p, (double *)st->pose_w.p + 7 * (size_t)kf_i,
                                                                    (double *)st->pt_w.p, (double *)st->out_pose.p, (double *)st->out_pt.p);
  ctx->launches++;
  CK(cudaMemcpyAsync(pose7_out, st->out_pose.p, (size_t)n_cam * 56, cudaMemcpyDeviceToHost, s));
  if (n_pt) {
    CK(cudaMemcpyAsync(pt3_out, st->out_pt.p, (size_t)n_pt * 24, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(landmark_of_pt, st->w_lm.p, (size_t)n_pt * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(intr4, ctx->intr.p, 32, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  st->ms[2] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_ph).count();
  if (ms_out)
    for (int k = 0; k < 3; ++k) ms_out[k] = st->ms[k];
  return BA_OK;
}

// ------------------------------------------------------------------ symbolic phase of the sparse Cholesky (host only; test hook)
struct ba_spsym {
  SpSymbolic s;
};
extern "C" int ba_sparse_symbolic_create(int32_t n_cam, int32_t n_blk, const int32_t *blk_i, const int32_t *blk_j, int32_t leaf_cams,
                                         int32_t cap_blocks, int32_t max_own, ba_spsym **out) {
  if (!out || n_cam <= 0 || n_blk < 0 || (n_blk > 0 && (!blk_i || !blk_j)) || cap_blocks < 2 || max_own < 1) return BA_ERR_INVALID;
  for (int b = 0; b < n_blk; ++b)
    if (blk_i[b] < 0 || blk_j[b] >= n_cam || blk_i[b] > blk_j[b]) return BA_ERR_INVALID;
  ba_spsym *h = new ba_spsym();
  h->s = spsym_build(n_cam, n_blk, blk_i, blk_j, leaf_cams, cap_blocks, max_own);
  if (h->s.error) {
    const int e = h->s.error;
    delete h;
    return e == 1 ? BA_ERR_UNSUPPORTED : BA_ERR_STATE;
  }
  *out = h;
  return BA_OK;
}
extern "C" void ba_sparse_symbolic_destroy(ba_spsym *h) { delete h; }
static const std::vector<int32_t> *spsym_array(const SpSymbolic &s, int which) {
  switch (which) {
    case 0: return &s.perm;
    case 1: return &s.pos;
    case 2: return &s.node;
    case 3: return &s.bord;
    case 4: return &s.children;
    case 5: return &s.rel;
    case 6: return &s.inv;
    case 7: return &s.aent;
    case 8: return &s.level_ptr;
    case 9: return &s.level_nodes;
    default: return nullptr;
  }
}
extern "C" int ba_sparse_symbolic_info(const ba_spsym *h, int64_t info[24]) {
  if (!h || !info) return BA_ERR_INVALID;
  const SpSymbolic &s = h->s;
  memset(info, 0, 24 * sizeof(int64_t));
  info[0] = s.n_cam;
  info[1] = s.n_nodes;
  info[2] = s.n_levels;
  info[3] = s.panel_blocks;
  info[4] = s.u_blocks;
  info[5] = s.max_front_blocks;
  info[6] = s.max_m;
  info[7] = s.max_nb;
  info[8] = s.max_children;
  info[9] = (int64_t)s.flops;
  info[10] = (int64_t)s.crit_blocks;
  for (int w = 0; w < 10; ++w) info[12 + w] = (int64_t)spsym_array(s, w)->size();
  return BA_OK;
}
extern "C" int ba_sparse_symbolic_partition(const ba_spsym *h, int32_t parts, int32_t *part, double work[3]) {
  if (!h || !part || parts < 1) return BA_ERR_INVALID;
  const SpPartition R = spsym_partition(h->s, parts);
  if (!R.part.empty()) memcpy(part, R.part.data(), R.part.size() * sizeof(int32_t));
  if (work) {
    work[0] = R.total;
    work[1] = R.top;
    work[2] = R.heaviest;
  }
  return R.parts;
}
extern "C" int ba_sparse_symbolic_get(const ba_spsym *h, int32_t which, int32_t *dst) {
  if (!h || !dst) return BA_ERR_INVALID;
  const std::vector<int32_t> *a = spsym_array(h->s, which);
  if (!a) return BA_ERR_INVALID;
  if (!a->empty()) memcpy(dst, a->data(), a->size() * sizeof(int32_t));
  return BA_OK;
}
