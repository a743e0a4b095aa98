// OptimizationUtils_gpu.cpp -- drop-in replacement for the Ceres-facing half of
// the reference's src/OptimizationUtils.cpp: countConstraints (:184-213) and
// windowOptimize (:215-313) keep their signatures (headers/OptimizationUtils.h:42,
// 55) and their observable behaviour -- enumeration order, in-place frame change
// and write-back -- while ceres::Problem / ceres::Solve (:218-300) are replaced by
// ba_gpu_upload / ba_gpu_solve / ba_gpu_download (include/ba_gpu.h).
//
// Inside the reference tree: compile with -DBA_USE_REFERENCE_HEADERS in place of
// the cost-functor / Ceres part of src/OptimizationUtils.cpp (INTEGRATION.md).
#ifdef BA_USE_REFERENCE_HEADERS
#include "OptimizationUtils.h"
#else
#include "compat/reference_types.h"
#endif

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../include/ba_gpu.h"
#include "ba_host_debug.h"
#include "se3_raw.h"

using std::vector;

namespace {
// one solver context per host thread, reused across windows (device buffers are
// kept; sliding windows repeat every frame_frequency keyframes, src/main.cpp:163-168)
struct Ctx {
  ba_gpu_ctx *ctx = nullptr;
  ~Ctx() {
    if (ctx) ba_gpu_destroy(ctx);
  }
};
thread_local Ctx g_ctx;
thread_local BaHostLastProblem g_last;
thread_local bool g_fixed_iterations = false;

// ---- device-resident store (SURVEY.md 8f row N1; ba_store_* in include/ba_gpu.h): what this thread has put on the device
struct StoreState {
  ba_store *st = nullptr;
  bool on = false;
  vector<long long> kf_size;      // global_points_map.size() of every keyframe at its last upload (-1: never)
  vector<Landmark *> lm_ptr;      // landmark id -> its node in the caller's Map3D (nodes of an unordered_map do not move)
  ~StoreState() {
    if (st) ba_store_destroy(st);
  }
  void reset() {  // forget what is on the device; the device buffers themselves are kept for the next sequence
    if (st && ba_store_clear(st) != BA_OK) {
      ba_store_destroy(st);
      st = nullptr;
    }
    kf_size.clear();
    lm_ptr.clear();
  }
};
thread_local StoreState g_store;
inline double ms_since(const std::chrono::steady_clock::time_point &t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}
}  // namespace

const BaHostLastProblem &ba_host_last_problem() { return g_last; }
void ba_host_fixed_iterations(bool on) { g_fixed_iterations = on; }
void ba_host_device_store(bool on) {
  // (the store is declared after the context in this file, so it is destroyed first at thread exit)
  g_store.reset();
  g_store.on = on;
}

namespace {
// windowOptimize through the device-resident store: only keyframes whose global_points_map is new or grew since the
// last call are walked and uploaded; enumeration, frame changes and write-back run on the device.  Returns 1 = done,
// 0 = failed (inputs untouched), -1 = not applicable (caller takes the full-upload path).
int window_optimize_store(const ba_gpu_options &opt, int kf_i, int kf_f, vector<KeyFrame> &keyframes, Map3D &map,
                          const Vector4d &intrinsics_initial, Vector4d &intrinsics_optimized) {
  const int n_cam = kf_f - kf_i + 1;
  const auto t_begin = std::chrono::steady_clock::now();
  int rc = g_ctx.ctx ? ba_gpu_set_options(g_ctx.ctx, &opt) : ba_gpu_create(&opt, &g_ctx.ctx);
  if (rc == BA_OK && !g_store.st) rc = ba_store_create(g_ctx.ctx, &g_store.st);
  if (rc != BA_OK) return -1;
  StoreState &S = g_store;
  if (S.kf_size.size() < keyframes.size()) S.kf_size.resize(keyframes.size(), -1);
  // (persistent scratch: no allocation per window)
  static thread_local vector<int32_t> ids, new_id, kf_list, kf_cnt;
  static thread_local vector<float> uvf;
  static thread_local vector<double> dep, new_xyz;
  ids.clear(); new_id.clear(); kf_list.clear(); kf_cnt.clear(); uvf.clear(); dep.clear(); new_xyz.clear();
  size_t lm_bound = 0;
  for (int kf_n = kf_i; kf_n <= kf_f; ++kf_n) {
    const KeyFrame &kf = keyframes[kf_n];
    lm_bound += kf.global_points_map.size();
    if (S.kf_size[kf_n] == (long long)kf.global_points_map.size()) continue;  // unchanged since its last upload
    const size_t before = ids.size();
    for (const auto &index_pair : kf.global_points_map) {  // container order == canonical order (:257)
      const int localId = index_pair.first, landmarkId = index_pair.second;
      if (landmarkId < 0 || landmarkId >= (1 << 24)) return -1;
      if ((size_t)landmarkId >= S.lm_ptr.size()) S.lm_ptr.resize((size_t)landmarkId + 1 + S.lm_ptr.size() / 2, nullptr);
      if (!S.lm_ptr[landmarkId]) {  // first time this landmark is referenced: its world point goes to the device
        auto found = map.find(landmarkId);
        if (found == map.end()) {
          std::fprintf(stderr, "windowOptimize: keyframe references a landmark that is not in the map\n");
          g_store.reset();
          return 0;
        }
        S.lm_ptr[landmarkId] = &found->second;
        new_id.push_back(landmarkId);
        for (int j = 0; j < 3; ++j) new_xyz.push_back(found->second.point(j));
      }
      ids.push_back(landmarkId);
      uvf.push_back(kf.keypoints[localId].pt.x);
      uvf.push_back(kf.keypoints[localId].pt.y);
      dep.push_back(kf.points3d_local[localId](2));
    }
    kf_list.push_back(kf_n);
    kf_cnt.push_back((int32_t)(ids.size() - before));
  }
  static thread_local double prof[5] = {0, 0, 0, 0, 0};
  const bool do_prof = std::getenv("BA_STORE_PROF") != nullptr;
  const double t_walk = ms_since(t_begin);
  rc = ba_store_set_keyframes(S.st, (int32_t)kf_list.size(), kf_list.data(), kf_cnt.data(), ids.data(), uvf.data(), dep.data());
  const double t_kf = ms_since(t_begin);
  if (rc == BA_ERR_UNSUPPORTED) {
    g_store.reset();
    return -1;
  }
  if (rc != BA_OK) return 0;
  for (int kf_n : kf_list) S.kf_size[kf_n] = (long long)keyframes[kf_n].global_points_map.size();
  if (!new_id.empty() && ba_store_set_landmarks(S.st, (int32_t)new_id.size(), new_id.data(), new_xyz.data()) != BA_OK) return 0;
  vector<double> pose7((size_t)n_cam * 7);
  for (int k = 0; k < n_cam; ++k)
    for (int j = 0; j < 7; ++j) pose7[(size_t)k * 7 + j] = keyframes[kf_i + k].T_w_c.data()[j];
  const double t_lm = ms_since(t_begin);
  if (ba_store_set_poses(S.st, kf_i, n_cam, pose7.data()) != BA_OK) return 0;
  g_last.ms_extract = ms_since(t_begin);
  if (do_prof) {
    prof[4] += 1;
    if ((int)prof[4] % 10 == 0 || g_last.ms_extract > 1.0)
      std::fprintf(stderr, "[BA_STORE_PROF] window %d ms: options+walk %.3f set_keyframes %.3f set_landmarks %.3f set_poses %.3f (%d kf, %zu obs, %zu new lm)\n",
                   (int)prof[4], t_walk, t_kf - t_walk, t_lm - t_kf, g_last.ms_extract - t_lm, (int)kf_list.size(), ids.size(), new_id.size());
  }

  double intr[4], prior[4], ms3[3] = {0, 0, 0};
  for (int j = 0; j < 4; ++j) {
    intr[j] = intrinsics_optimized(j);
    prior[j] = intrinsics_initial(j);
  }
  vector<int32_t> lm_of_pt(lm_bound + 1);
  vector<double> pt3((lm_bound + 1) * 3);
  int32_t n_pt = 0, n_obs = 0;
  ba_gpu_summary summary;
  rc = ba_store_window_solve(S.st, kf_i, kf_f, prior, intr, &summary, pose7.data(), (int32_t)lm_bound, &n_pt, lm_of_pt.data(), pt3.data(),
                             &n_obs, ms3);
  if (rc != BA_OK) {
    std::fprintf(stderr, "windowOptimize: GPU solve failed (%d): %s\n", rc, ba_gpu_last_error(g_ctx.ctx));
    // the device copy may no longer mirror the host state: start over at the next call
    g_store.reset();
    return 0;
  }
  g_last.ms_upload = ms3[0];
  g_last.ms_solve = ms3[1];
  g_last.ms_download = ms3[2];
  const auto t_wb = std::chrono::steady_clock::now();
  g_last.summary = summary;
  g_last.admissible_obs = n_obs;
  g_last.cam_idx.clear();
  g_last.pt_idx.clear();
  g_last.landmark_of_pt.assign(lm_of_pt.begin(), lm_of_pt.begin() + n_pt);
  for (int k = 0; k < n_cam; ++k) keyframes[kf_i + k].T_w_c = se3_from_raw(pose7.data() + (size_t)k * 7);
  for (int p = 0; p < n_pt; ++p) {
    Vector3d &x = S.lm_ptr[lm_of_pt[p]]->point;
    for (int j = 0; j < 3; ++j) x(j) = pt3[(size_t)p * 3 + j];
  }
  for (int j = 0; j < 4; ++j) intrinsics_optimized(j) = intr[j];
  g_last.ms_writeback = ms_since(t_wb);
  return 1;
}
}  // namespace

int countConstraints(const Map3D &map, const vector<KeyFrame> &keyframes, int kf_i, int kf_f) {
  (void)map;
  int admissible_obs = 0;
  for (int kf_n = kf_i; kf_n <= kf_f; kf_n++) {
    const KeyFrame &kf = keyframes[kf_n];
    for (const auto &index_pair : kf.global_points_map) {
      const double depth = kf.points3d_local[index_pair.first](2);
      if (depth <= 1e-15) {
        // the reference prints here (:202); kept quiet on purpose: same count
        continue;
      }
      admissible_obs++;
    }
  }
  return admissible_obs;
}

bool windowOptimize(ceresGlobalProblem &globalProblem, int kf_i, int kf_f, vector<KeyFrame> &keyframes, Map3D &map,
                    const Vector4d &intrinsics_initial, Vector4d &intrinsics_optimized) {
  const int n_cam = kf_f - kf_i + 1;
  if (n_cam <= 0) return true;

  // ---- options: ceresGlobalProblem knobs (:47-50, :64-65) -> ba_gpu_options
  ba_gpu_options opt;
  ba_gpu_default_options(&opt);
  opt.HUB_P_REPR = globalProblem.HUB_P_REPR;
  opt.HUB_P_UNPR = globalProblem.HUB_P_UNPR;
  opt.WEIGHT_UNPR = globalProblem.WEIGHT_UNPR;
  opt.WEIGHT_INTRINSICS = globalProblem.WEIGHT_INTRINSICS;
  opt.max_num_iterations = globalProblem.options.max_num_iterations;
  opt.eta = globalProblem.options.eta;
  // convergence tolerances travel in ceres::Solver::Options as they did for ceres::Solve (the reference leaves them at
  // Ceres' defaults, headers/BundleAdjustmentConfig.h:61-67; bench/ceres_baseline.cpp sets them to zero for fixed-count runs)
  opt.function_tolerance = globalProblem.options.function_tolerance;
  opt.gradient_tolerance = globalProblem.options.gradient_tolerance;
  opt.parameter_tolerance = globalProblem.options.parameter_tolerance;
  opt.use_depth_prior = 1;       // DepthPrior residual per observation (:288-294)
  opt.optimize_intrinsics = 1;   // intrinsics are a free block with a prior (:236-241)
  opt.solver = BA_SOLVER_AUTO;   // SPARSE_SCHUR == exact Schur step
  if (g_fixed_iterations)        // measurement only (ba_host_debug.h): exactly max_num_iterations LM iterations
    opt.function_tolerance = opt.parameter_tolerance = opt.gradient_tolerance = 0.0;
  if (g_store.on) {
    const int done = window_optimize_store(opt, kf_i, kf_f, keyframes, map, intrinsics_initial, intrinsics_optimized);
    if (done >= 0) return done == 1;
  }
  const auto t_begin = std::chrono::steady_clock::now();

  // ---- snapshot for the error path: inputs stay untouched on failure
  vector<Sophus::SE3d> pose_backup(n_cam);
  for (int k = 0; k < n_cam; ++k) pose_backup[k] = keyframes[kf_i + k].T_w_c;
  vector<std::pair<int, Vector3d>> point_backup;

  const Sophus::SE3d initialPose = keyframes[kf_i].T_w_c;          // :231
  const Sophus::SE3d initialPoseInv = keyframes[kf_i].T_w_c.inverse();  // :232
  // The reference counts the admissible observations first (:242) because the count is the weight normaliser of every
  // residual; here the normaliser is the n_obs of the upload (the same number by construction), so the extra walk over all
  // hash maps is replaced by an upper bound for the reservations.
  size_t obs_bound = 0;
  for (int kf_n = kf_i; kf_n <= kf_f; kf_n++) obs_bound += keyframes[kf_n].global_points_map.size();

  // ---- canonical enumeration (:244-294): container order, first-appearance point ids.
  // One hash lookup per observation (landmark id -> point index, inserted on first appearance) and one map
  // lookup per DISTINCT landmark; the Landmark addresses are kept (unordered_map nodes do not move), so the
  // gather of the points, the error path and the write-back never search the map again.
  // landmark id -> point index: ids are small non-negative integers in the reference (a running counter, src/main.cpp), so
  // the lookup is a flat epoch-stamped table that persists across calls (no clearing, no hashing); any other id falls back
  // to a hash map
  struct Stamp {
    int epoch, pt;
  };
  static thread_local vector<Stamp> flat;
  static thread_local int epoch = 0;
  if (++epoch == 0x7fffffff) {
    flat.assign(flat.size(), Stamp{0, 0});
    epoch = 1;
  }
  constexpr int kFlatMax = 1 << 24;
  std::unordered_map<int, int> pt_of_landmark;
  vector<int> landmark_of_pt;
  vector<Landmark *> landmark_ptr;
  vector<int32_t> cam_idx, pt_idx;
  vector<double> uv2, depthv, pose7((size_t)n_cam * 7), pt3;
  cam_idx.reserve(obs_bound);
  pt_idx.reserve(obs_bound);
  uv2.reserve(obs_bound * 2);
  depthv.reserve(obs_bound);
  bool missing_landmark = false;
  for (int kf_n = kf_i; kf_n <= kf_f && !missing_landmark; kf_n++) {
    KeyFrame &curr_kf = keyframes[kf_n];
    curr_kf.T_w_c = Sophus::SE3d(initialPoseInv * curr_kf.T_w_c);  // :248, in place
    for (const auto &index_pair : curr_kf.global_points_map) {
      const int landmarkId = index_pair.second;
      const int localId = index_pair.first;
      const double depth = curr_kf.points3d_local[localId](2);
      if (depth <= 1e-15) continue;  // :265-268
      int *pt_slot;
      bool first;
      if (landmarkId >= 0 && landmarkId < kFlatMax) {
        if ((size_t)landmarkId >= flat.size()) flat.resize((size_t)landmarkId + 1 + flat.size() / 2, Stamp{0, 0});
        Stamp &st = flat[landmarkId];
        first = st.epoch != epoch;
        if (first) {
          st.epoch = epoch;
          st.pt = (int)landmark_of_pt.size();
        }
        pt_slot = &st.pt;
      } else {
        const auto ins = pt_of_landmark.try_emplace(landmarkId, (int)landmark_of_pt.size());
        first = ins.second;
        pt_slot = &ins.first->second;
      }
      if (first) {  // first appearance in the window (:271)
        auto found = map.find(landmarkId);
        if (found == map.end()) {  // the reference would throw from map.at (:270)
          missing_landmark = true;
          break;
        }
        Landmark &map_point = found->second;
        point_backup.emplace_back(landmarkId, map_point.point);
        map_point.point = initialPoseInv * map_point.point;  // :274, in place
        landmark_of_pt.push_back(landmarkId);
        landmark_ptr.push_back(&map_point);
      }
      cam_idx.push_back(kf_n - kf_i);
      pt_idx.push_back(*pt_slot);
      uv2.push_back((double)curr_kf.keypoints[localId].pt.x);  // float -> double (:262)
      uv2.push_back((double)curr_kf.keypoints[localId].pt.y);
      depthv.push_back(depth);
    }
  }
  auto restore = [&]() {
    for (int k = 0; k < n_cam; ++k) keyframes[kf_i + k].T_w_c = pose_backup[k];
    for (size_t p = 0; p < landmark_ptr.size(); ++p) landmark_ptr[p]->point = point_backup[p].second;
  };
  if (missing_landmark) {
    std::fprintf(stderr, "windowOptimize: keyframe references a landmark that is not in the map\n");
    restore();
    return false;
  }
  const int n_pt = (int)landmark_of_pt.size(), n_obs = (int)cam_idx.size();
  for (int k = 0; k < n_cam; ++k)
    for (int j = 0; j < 7; ++j) pose7[(size_t)k * 7 + j] = keyframes[kf_i + k].T_w_c.data()[j];
  pt3.resize((size_t)n_pt * 3);
  for (int p = 0; p < n_pt; ++p)
    for (int j = 0; j < 3; ++j) pt3[(size_t)p * 3 + j] = landmark_ptr[p]->point(j);
  double intr[4], prior[4];
  for (int j = 0; j < 4; ++j) {
    intr[j] = intrinsics_optimized(j);
    prior[j] = intrinsics_initial(j);
  }
  g_last.admissible_obs = n_obs;  // == countConstraints(map, keyframes, kf_i, kf_f)
  g_last.ms_extract = ms_since(t_begin);

  // ---- ceres::Solve (:300) -> GPU
  int rc = BA_OK;
  if (!g_ctx.ctx)
    rc = ba_gpu_create(&opt, &g_ctx.ctx);
  else
    rc = ba_gpu_set_options(g_ctx.ctx, &opt);
  ba_gpu_summary summary;
  auto t_phase = std::chrono::steady_clock::now();
  if (rc == BA_OK)
    rc = ba_gpu_upload(g_ctx.ctx, n_cam, pose7.data(), /*fixed_cam=*/0 /* :299 */, n_pt, pt3.data(), n_obs, cam_idx.data(),
                       pt_idx.data(), uv2.data(), depthv.data(), intr, prior);
  g_last.ms_upload = ms_since(t_phase);
  t_phase = std::chrono::steady_clock::now();
  if (rc == BA_OK) rc = ba_gpu_solve(g_ctx.ctx, &summary);
  g_last.ms_solve = ms_since(t_phase);
  t_phase = std::chrono::steady_clock::now();
  if (rc == BA_OK) rc = ba_gpu_download(g_ctx.ctx, pose7.data(), pt3.data(), intr);
  g_last.ms_download = ms_since(t_phase);
  t_phase = std::chrono::steady_clock::now();
  if (rc != BA_OK) {
    std::fprintf(stderr, "windowOptimize: GPU solve failed (%d): %s\n", rc, ba_gpu_last_error(g_ctx.ctx));
    restore();
    return false;
  }
  g_last.summary = summary;
  g_last.cam_idx.swap(cam_idx);
  g_last.pt_idx.swap(pt_idx);
  g_last.landmark_of_pt = landmark_of_pt;

  // ---- Ceres wrote the optimum into the caller-owned blocks: do the same
  for (int k = 0; k < n_cam; ++k) keyframes[kf_i + k].T_w_c = se3_from_raw(pose7.data() + (size_t)k * 7);
  for (int p = 0; p < n_pt; ++p) {
    Vector3d &x = landmark_ptr[p]->point;
    for (int j = 0; j < 3; ++j) x(j) = pt3[(size_t)p * 3 + j];
  }
  for (int j = 0; j < 4; ++j) intrinsics_optimized(j) = intr[j];

  // ---- back to the world frame (:303-310)
  for (int kf_n = kf_i; kf_n <= kf_f; kf_n++) {
    KeyFrame &curr_kf = keyframes[kf_n];
    curr_kf.T_w_c = Sophus::SE3d(initialPose * curr_kf.T_w_c);
  }
  for (Landmark *lm : landmark_ptr) lm->point = initialPose * lm->point;
  g_last.ms_writeback = ms_since(t_phase);
  return true;
}
