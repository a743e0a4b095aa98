// Flat C harness around the C++ drop-in (tests drive it through ctypes): builds
// vector<KeyFrame> + Map3D from arrays with the SAME std::unordered_map insert
// sequence the caller specifies, runs windowOptimize / countConstraints with the
// reference's signatures, and flattens the mutated state back.
#ifdef BA_USE_REFERENCE_HEADERS
#include "OptimizationUtils.h"
#else
#include "compat/reference_types.h"
#endif
#include "ba_host_debug.h"
#include "se3_raw.h"

#include <chrono>
#include <cstring>

extern "C" {
// obs arrays are in INSERTION order per keyframe: kf_ptr[n_kf+1] CSR,
// local ids are 0..cnt-1 in that order; landmark ids lm[]; pixels float; depth double.
// pose7 [n_kf*7], landmark table: lm_id[n_lm], lm_pt[n_lm*3].  All in/out.
// out_* (nullable): the enumeration windowOptimize produced and, independently,
// the container iteration order recomputed here.
int ba_host_window_optimize(int n_kf, double *pose7, const int32_t *kf_ptr, const int32_t *lm, const float *uv,
                            const double *depth, int n_lm, const int32_t *lm_id, double *lm_pt, int kf_i, int kf_f,
                            int max_num_iterations, const double *intr0, double *intr, int32_t *out_n_obs,
                            int32_t *out_cam_idx, int32_t *out_landmark, int32_t *ref_cam_idx, int32_t *ref_landmark,
                            int32_t *out_count, double *out_costs /*initial, final*/) {
  std::vector<KeyFrame> keyframes(n_kf);
  Map3D map;
  for (int k = 0; k < n_kf; ++k) {
    KeyFrame &kf = keyframes[k];
    kf.frame_id = (uint)k;
    kf.T_w_c = se3_from_raw(pose7 + (size_t)k * 7);
    const int a = kf_ptr[k], b = kf_ptr[k + 1];
    kf.keypoints.resize(b - a);
    kf.points3d_local.resize(b - a);
    for (int i = a; i < b; ++i) {
      const int local = i - a;
      kf.keypoints[local].pt.x = uv[2 * (size_t)i];
      kf.keypoints[local].pt.y = uv[2 * (size_t)i + 1];
      kf.points3d_local[local] = Vector3d(0.0, 0.0, depth[i]);
      kf.global_points_map.insert({local, lm[i]});
    }
  }
  for (int l = 0; l < n_lm; ++l) {
    Landmark L;
    L.point = Vector3d(lm_pt[3 * (size_t)l], lm_pt[3 * (size_t)l + 1], lm_pt[3 * (size_t)l + 2]);
    map.insert({lm_id[l], L});
  }
  // independent walk of the containers (what the reference's loops would visit)
  int nref = 0;
  for (int k = kf_i; k <= kf_f; ++k)
    for (const auto &pr : keyframes[k].global_points_map) {
      if (keyframes[k].points3d_local[pr.first](2) <= 1e-15) continue;
      if (ref_cam_idx) ref_cam_idx[nref] = k - kf_i;
      if (ref_landmark) ref_landmark[nref] = pr.second;
      ++nref;
    }
  if (out_count) *out_count = countConstraints(map, keyframes, kf_i, kf_f);
  ceresGlobalProblem gp;
  gp.options.max_num_iterations = max_num_iterations;
  Vector4d i0(intr0[0], intr0[1], intr0[2], intr0[3]), io(intr[0], intr[1], intr[2], intr[3]);
  const bool ok = windowOptimize(gp, kf_i, kf_f, keyframes, map, i0, io);
  const BaHostLastProblem &last = ba_host_last_problem();
  if (ok) {
    if (out_n_obs) *out_n_obs = (int32_t)last.cam_idx.size();
    for (size_t i = 0; i < last.cam_idx.size(); ++i) {
      if (out_cam_idx) out_cam_idx[i] = last.cam_idx[i];
      if (out_landmark) out_landmark[i] = last.landmark_of_pt[last.pt_idx[i]];
    }
    if (out_costs) {
      out_costs[0] = last.summary.initial_cost;
      out_costs[1] = last.summary.final_cost;
    }
  }
  for (int k = 0; k < n_kf; ++k) std::memcpy(pose7 + (size_t)k * 7, keyframes[k].T_w_c.data(), 7 * sizeof(double));
  for (int l = 0; l < n_lm; ++l)
    for (int j = 0; j < 3; ++j) lm_pt[3 * (size_t)l + j] = map.at(lm_id[l]).point(j);
  for (int j = 0; j < 4; ++j) intr[j] = io(j);
  return ok ? 0 : -1;
}

// The reference's optimisation schedule (src/main.cpp:161-182) over a whole recorded sequence through the compiled
// drop-in: a window over the last `window_size` keyframes whenever the keyframe count is a multiple of
// `frame_frequency` (:162-166), the leftover window at the end of tracking (:169-175), and, if do_global != 0, the
// global optimisation over all keyframes instead (:178-182).  Containers are built once (as the tracking front end
// would have left them); every window is warm-started by the previous ones.  fixed_iterations != 0 switches the
// tolerances off, so that every call runs exactly max_num_iterations LM iterations (throughput measurement).
// out_ms[7]: accumulated host wall clock -- total, container walk + frame change, ba_gpu_upload, ba_gpu_solve,
// ba_gpu_download, write-back -- and the number of calls the device-resident store solved.  Returns the number of windowOptimize calls, or -1 if one failed.
int ba_host_sliding_sequence(int n_kf, double *pose7, const int32_t *kf_ptr, const int32_t *lm, const float *uv,
                             const double *depth, int n_lm, const int32_t *lm_id, double *lm_pt, int window_size,
                             int frame_frequency, int do_global, int max_num_iterations, int fixed_iterations,
                             const double *intr0, double *intr, double *out_ms, int64_t *out_lm_iterations, int use_device_store) {
  if (n_kf <= 0 || frame_frequency <= 0 || window_size <= 0 || window_size > n_kf) return -1;
  ba_host_device_store((use_device_store & 1) != 0);  // bit 0: device-resident store, bit 1: maps grow in two steps
  // Containers grow as the tracking front end would grow them (src/main.cpp:25-82, src/Map3D.cpp:29-74): keyframe k arrives
  // with its key points and the first part of its global_points_map (its matches as "new_frame"); the rest of its map is
  // inserted when keyframe k + 1 arrives (its inserts as "old_frame", :52) -- growing != 0 splits every list in two halves
  // that way, growing == 0 inserts the whole list at arrival.  A landmark enters the map when it is first referenced.
  const bool growing = (use_device_store & 2) != 0;
  std::vector<KeyFrame> keyframes;
  keyframes.reserve(n_kf);
  Map3D map;
  std::unordered_map<int, int> lm_row;  // landmark id -> row of lm_pt
  for (int l = 0; l < n_lm; ++l) lm_row[lm_id[l]] = l;
  auto insert_obs = [&](int k, int i0_, int i1_) {
    KeyFrame &kf = keyframes[k];
    for (int i = i0_; i < i1_; ++i) {
      kf.global_points_map.insert({i - kf_ptr[k], lm[i]});
      if (map.find(lm[i]) == map.end()) {
        const int l = lm_row.at(lm[i]);
        Landmark L;
        L.point = Vector3d(lm_pt[3 * (size_t)l], lm_pt[3 * (size_t)l + 1], lm_pt[3 * (size_t)l + 2]);
        map.insert({lm[i], L});
      }
    }
  };
  auto arrive = [&](int k) {
    keyframes.emplace_back();
    KeyFrame &kf = keyframes[k];
    kf.frame_id = (uint)k;
    kf.T_w_c = se3_from_raw(pose7 + (size_t)k * 7);
    const int a = kf_ptr[k], b = kf_ptr[k + 1];
    kf.keypoints.resize(b - a);
    kf.points3d_local.resize(b - a);
    for (int i = a; i < b; ++i) {
      kf.keypoints[i - a].pt.x = uv[2 * (size_t)i];
      kf.keypoints[i - a].pt.y = uv[2 * (size_t)i + 1];
      kf.points3d_local[i - a] = Vector3d(0.0, 0.0, depth[i]);
    }
    const int half = growing ? a + (b - a) / 2 : b;
    insert_obs(k, a, half);
    if (growing && k > 0) insert_obs(k - 1, kf_ptr[k - 1] + (kf_ptr[k] - kf_ptr[k - 1]) / 2, kf_ptr[k]);
  };
  ceresGlobalProblem gp;
  gp.options.max_num_iterations = max_num_iterations;
  Vector4d i0(intr0[0], intr0[1], intr0[2], intr0[3]), io(intr[0], intr[1], intr[2], intr[3]);
  double ms[7] = {0, 0, 0, 0, 0, 0, 0};
  int64_t lm_iterations = 0;
  int calls = 0;
  bool ok = true;
  ba_host_fixed_iterations(fixed_iterations != 0);
  auto run = [&](int kf_i, int kf_f) {
    const auto t0 = std::chrono::steady_clock::now();
    ok = ok && windowOptimize(gp, kf_i, kf_f, keyframes, map, i0, io);
    ms[0] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    const BaHostLastProblem &last = ba_host_last_problem();
    ms[1] += last.ms_extract;
    ms[2] += last.ms_upload;
    ms[3] += last.ms_solve;
    ms[4] += last.ms_download;
    ms[5] += last.ms_writeback;
    if (ok && last.cam_idx.empty() && last.admissible_obs > 0) ms[6] += 1;  // (the store path keeps no host index arrays)
    lm_iterations += last.summary.num_iterations;
    ++calls;
  };
  if (do_global) {
    for (int k = 0; k < n_kf; ++k) arrive(k);
    if (growing) insert_obs(n_kf - 1, kf_ptr[n_kf - 1] + (kf_ptr[n_kf] - kf_ptr[n_kf - 1]) / 2, kf_ptr[n_kf]);
    run(0, n_kf - 1);
  } else {
    for (int size = 1; size <= n_kf && ok; ++size) {  // keyframes.size() after every tracking step
      arrive(size - 1);
      if (size % frame_frequency == 0 && size >= window_size) run(size - window_size, size - 1);
    }
    if (ok && n_kf % frame_frequency != 0) run(n_kf - window_size, n_kf - 1);  // leftovers
  }
  ba_host_fixed_iterations(false);
  ba_host_device_store(false);
  if (out_ms) std::memcpy(out_ms, ms, sizeof(ms));
  if (out_lm_iterations) *out_lm_iterations = lm_iterations;
  for (int k = 0; k < n_kf; ++k) std::memcpy(pose7 + (size_t)k * 7, keyframes[k].T_w_c.data(), 7 * sizeof(double));
  for (int l = 0; l < n_lm; ++l) {
    auto found = map.find(lm_id[l]);  // (a landmark nobody referenced never entered the map)
    if (found != map.end())
      for (int j = 0; j < 3; ++j) lm_pt[3 * (size_t)l + j] = found->second.point(j);
  }
  for (int j = 0; j < 4; ++j) intr[j] = io(j);
  return ok ? calls : -1;
}

int ba_host_count_constraints(int n_kf, const int32_t *kf_ptr, const double *depth, int kf_i, int kf_f) {
  std::vector<KeyFrame> keyframes(n_kf);
  Map3D map;
  for (int k = 0; k < n_kf; ++k) {
    const int a = kf_ptr[k], b = kf_ptr[k + 1];
    keyframes[k].points3d_local.resize(b - a);
    for (int i = a; i < b; ++i) {
      keyframes[k].points3d_local[i - a] = Vector3d(0.0, 0.0, depth[i]);
      keyframes[k].global_points_map.insert({i - a, i});
    }
  }
  return countConstraints(map, keyframes, kf_i, kf_f);
}

// ---- flat wrappers of host/TrajectoryIO.cpp (tests/test_trajectory_eval.py)
int ba_host_read_intrinsics(const char *path, double out4[4]) {
  const Vector4d k = read_camera_intrinsics_from_file(path);
  for (int i = 0; i < 4; ++i) out4[i] = k[i];
  return 0;
}
int ba_host_get_first_pose(const char *first_timestamp, const char *gt_path, double out7[7]) {
  const Sophus::SE3d T = getFirstPose(first_timestamp, gt_path);
  std::memcpy(out7, T.data(), 7 * sizeof(double));
  return 0;
}
// timestamps: n NUL-terminated strings back to back
int ba_host_write_poses(const char *path, int n, const char *timestamps, const double *pose7) {
  std::vector<KeyFrame> kfs(n);
  const char *t = timestamps;
  for (int i = 0; i < n; ++i) {
    kfs[i].timestamp = t;
    t += kfs[i].timestamp.size() + 1;
    kfs[i].T_w_c = se3_from_raw(pose7 + (size_t)i * 7);
  }
  write_keyframe_poses_to_file(path, kfs);
  return 0;
}
int ba_host_pose_offset(int n, double *pose7, const double *initial7) {
  std::vector<KeyFrame> kfs(n);
  for (int i = 0; i < n; ++i) kfs[i].T_w_c = se3_from_raw(pose7 + (size_t)i * 7);
  poseOffset(kfs, se3_from_raw(initial7));
  for (int i = 0; i < n; ++i) std::memcpy(pose7 + (size_t)i * 7, kfs[i].T_w_c.data(), 7 * sizeof(double));
  return 0;
}
}
