// Introspection of the last problem windowOptimize handed to the GPU (tests only).
#pragma once
#include <stdint.h>

#include <vector>

#include "../../include/ba_gpu.h"

struct BaHostLastProblem {
  std::vector<int32_t> cam_idx, pt_idx;
  std::vector<int> landmark_of_pt;
  int admissible_obs = 0;
  ba_gpu_summary summary{};
  // host wall clock of the last call, per phase: container walk + frame change, ba_gpu_upload, ba_gpu_solve,
  // ba_gpu_download, write-back into the caller's containers
  double ms_extract = 0, ms_upload = 0, ms_solve = 0, ms_download = 0, ms_writeback = 0;
};
const BaHostLastProblem &ba_host_last_problem();
// measurement only: tolerances off, so that every call runs exactly options.max_num_iterations LM iterations
void ba_host_fixed_iterations(bool on);
// Device-resident keyframe / landmark store (SURVEY.md 8f row N1; ba_store_* of include/ba_gpu.h) behind windowOptimize: on =
// windows upload only the keyframes that are new or whose global_points_map grew since the last
// call, and enumerate / change frames on the device; off (default) = every call walks and uploads the whole window.
// Assumes what holds in the reference's main loop: between two calls only new keyframes / landmarks appear, a keyframe's
// map only GROWS (src/Map3D.cpp:52-53, 73), and world points are changed by windowOptimize alone.  Calling it (on or off)
// drops what is on the device -- call it again after anything else edited poses of old keyframes or landmark points.
void ba_host_device_store(bool on);
