// pose_select.hpp — the step right after the path (SURVEY.md 8f rank 3): which refined hypothesis the node returns and
// how it is packed into the 7 floats it publishes (pose_estimation/src/opencv_surface_match.cpp:100-142).  Host-side, no
// device work; shared by the C++ facade (pcl_facade.hpp) and the library itself (peb_surface_match), so that both run the
// same rule.  Plain C++ over the C ABI's types, nothing else.
#pragma once

#include <cstddef>

#include "../pe_b200.h"

namespace pe_b200 {

// Which refined hypothesis the node returns: pose_estimation/src/opencv_surface_match.cpp:100-124.
// Most votes wins; but if the matcher produced more than 5 results in total, the lowest residual among
// the refined poses with more than 400 votes overrides it (the loop keeps the LAST assignment, so a later
// pose with more votes still takes over — reproduced as written).
inline size_t select_best_pose(const int* num_votes, const double* residual, size_t n_subset, size_t n_results_total) {
  int max_votes = 0;
  float min_res = 10000.0f;
  size_t best_idx = 0;
  for (size_t i = 0; i < n_subset; ++i) {
    if (num_votes[i] > max_votes) {
      max_votes = num_votes[i];
      best_idx = i;
    }
    if (n_results_total > 5) {
      if (residual[i] < min_res && num_votes[i] > 400) {
        min_res = static_cast<float>(residual[i]);
        best_idx = i;
      }
    }
  }
  return best_idx;
}

// The 7 floats {x, y, z, qx, qy, qz, qw} from the selected cv::ppf_match_3d::Pose3D itself, the way
// opencv_surface_match.cpp:133-142 builds them: t, then q (w x y z) as x y z w (pcl_facade.hpp's pack_pose packs a 4 x 4).  reference_layout = true writes it literally: pose[5] (qz) is never written and left 0,
// pose[6] receives q[3] and is then overwritten with q[0].
inline void pack_pose3d(const peb_ppf_pose& p, float pose7[7], bool reference_layout = false) {
  for (int i = 0; i < 3; ++i) pose7[i] = static_cast<float>(p.t[i]);
  pose7[3] = static_cast<float>(p.q[1]);
  pose7[4] = static_cast<float>(p.q[2]);
  if (reference_layout) {
    pose7[5] = 0.0f;
    pose7[6] = static_cast<float>(p.q[3]);
    pose7[6] = static_cast<float>(p.q[0]);
  } else {
    pose7[5] = static_cast<float>(p.q[3]);
    pose7[6] = static_cast<float>(p.q[0]);
  }
}

}  // namespace pe_b200
