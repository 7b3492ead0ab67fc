// pcl_facade.hpp — header-only C++ facade over the C ABI of libpe_b200.so (include/pe_b200.h).
//
// The classes carry the names, setters, defaults and enum values of the PCL 1.10 classes the
// north-star path substitutes into the reference's slots, so host code written against PCL ports
// by a namespace swap (pcl:: -> pe_b200::):
//
//   pe_b200::VoxelGrid                         pcl::VoxelGrid<pcl::PointXYZ>
//        down-sample slot  pose_estimation/src/pose_estimation.cpp:261-263
//   pe_b200::NormalEstimation                  pcl::NormalEstimation<pcl::PointXYZ, pcl::Normal>
//        normals slot      pose_estimation/src/opencv_surface_match.cpp:57-59
//   pe_b200::IterativeClosestPoint             pcl::IterativeClosestPoint<PointXYZ, PointXYZ>
//   pe_b200::IterativeClosestPointWithNormals  pcl::IterativeClosestPointWithNormals<PointNormal, PointNormal>
//        refinement slot   pose_estimation/src/opencv_surface_match.cpp:85-94
//
// Clouds are passed as (pointer, count, stride in bytes): pcl::PointCloud<PointXYZ>::points.data()
// with stride 16, pcl::PointNormal with stride 48, rows of a cv::Mat N x 3 / N x 6 CV_32F with
// stride 12 / 24 (cv::Mat::step).  Matrices are 16 floats column-major, i.e.
// Eigen::Matrix4f::data().  No dependency on PCL, Eigen or OpenCV.  Errors throw pe_b200::Error
// (the C ABI itself never throws); numerical outcomes are reported like PCL reports them.
#pragma once

#include <cfloat>
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../pe_b200.h"

namespace pe_b200 {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct CloudView {
  const void* data = nullptr;
  size_t size = 0;
  size_t stride = 16;
};

// owns one peb_ctx; share one Context between the objects used by one thread
class Context {
 public:
  explicit Context(int device = 0) {
    if (int rc = peb_ctx_create(device, &ctx_)) throw Error(rc, peb_last_error(nullptr));
  }
  ~Context() { peb_ctx_destroy(ctx_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  peb_ctx* get() const { return ctx_; }
  void check(int rc) const {
    if (rc != PEB_OK) throw Error(rc, peb_last_error(ctx_));
  }

 private:
  peb_ctx* ctx_ = nullptr;
};

// NaN removal + sphere filter + plane-band removal in front of VoxelGrid: the deterministic part of
// PoseEstimation::create_surface_match_pc (pose_estimation/src/pose_estimation.cpp:246-261, 309-333, 347-372)
class ScenePrefilter {
 public:
  explicit ScenePrefilter(Context& c) : c_(c) {
    std::memset(&p_, 0, sizeof(p_));
    p_.plane_band = 0.005f;
  }
  void setInputCloud(const void* pts, size_t n, size_t stride = 16) { in_ = {pts, n, stride}; }
  // filter_out == "inliers" drops the points inside the sphere, anything else keeps only them
  void setSphereFilter(const float center[3], float radius, const std::string& filter_out) {
    p_.use_sphere = radius > 0.0f ? 1 : 0;
    p_.remove_inliers = filter_out == "inliers" ? 1 : 0;
    for (int i = 0; i < 3; ++i) p_.sphere_center[i] = center[i];
    p_.sphere_radius = radius;
  }
  void addPlane(float a, float b, float c, float d) {
    if (p_.n_planes >= PEB_PREFILTER_MAX_PLANES) throw Error(PEB_E_INVALID_ARG, "ScenePrefilter: too many planes");
    float* v = p_.planes + 4 * p_.n_planes++;
    v[0] = a, v[1] = b, v[2] = c, v[3] = d;
  }
  void filter(std::vector<float>& out_xyz4) {
    out_xyz4.resize(4 * (in_.size ? in_.size : 1));
    size_t m = 0;
    c_.check(peb_scene_prefilter(c_.get(), in_.data, in_.size, in_.stride, &p_, out_xyz4.data(), &m));
    out_xyz4.resize(4 * m);
  }

 private:
  Context& c_;
  CloudView in_;
  peb_prefilter_params p_;
};

// PoseEstimation::create_surface_match_pc (pose_estimation/src/pose_estimation.cpp:246-261 + remove_planes :281-345) in ONE
// library call: NaN removal, optional sphere filter, num_planes rounds of plane RANSAC + band removal, optional VoxelGrid.
// The cloud crosses PCIe once in each direction.  planes (optional): num_planes x 4 coefficients.
inline void create_surface_match_pc(Context& c, const void* pts, size_t n, size_t stride, const float* filter_pose,
                                    float filter_radius, const std::string& filter_out, int num_planes, float leaf,
                                    std::vector<float>& out_xyz4, std::vector<float>* planes = nullptr) {
  peb_prefilter_params f;
  std::memset(&f, 0, sizeof(f));
  f.plane_band = 0.005f;                                    // :320
  if (filter_pose && filter_radius > 0.0f) {                // :250-256
    f.use_sphere = 1;
    f.remove_inliers = filter_out == "inliers" ? 1 : 0;
    for (int i = 0; i < 3; ++i) f.sphere_center[i] = filter_pose[i];
    f.sphere_radius = filter_radius;
  }
  peb_sac_params sac;
  peb_sac_params_default(&sac);
  sac.distance_threshold = 0.0001;                          // :294
  sac.max_iterations = 100;                                 // :295
  out_xyz4.resize(4 * (n ? n : 1));
  std::vector<float> pl(4 * static_cast<size_t>(num_planes > 0 ? num_planes : 1), 0.0f);
  size_t m = 0;
  c.check(peb_scene_prepare(c.get(), pts, n, stride, &f, num_planes, &sac, leaf, out_xyz4.data(), &m, pl.data()));
  out_xyz4.resize(4 * m);
  if (planes) planes->assign(pl.begin(), pl.begin() + 4 * static_cast<size_t>(num_planes > 0 ? num_planes : 0));
}

// pcl::SACSegmentation<pcl::PointXYZ> for SACMODEL_PLANE + SAC_RANSAC: the plane fit of remove_planes
// (pose_estimation/src/pose_estimation.cpp:285-297).  Same setters and defaults as
// [PCL] segmentation/include/pcl/segmentation/sac_segmentation.h; other model / method types throw
// PEB_E_UNSUPPORTED (no CPU fallback).
class SACSegmentation {
 public:
  enum { SACMODEL_PLANE = 0, SAC_RANSAC = 0 };  // pcl::SacModel / pcl::SAC_RANSAC values
  explicit SACSegmentation(Context& c) : c_(c) { peb_sac_params_default(&p_); }
  void setInputCloud(const void* pts, size_t n, size_t stride = 16) { in_ = {pts, n, stride}; }
  void setModelType(int model) {
    if (model != SACMODEL_PLANE) throw Error(PEB_E_UNSUPPORTED, "SACSegmentation: only SACMODEL_PLANE has a CUDA implementation");
    have_model_ = true;
  }
  void setMethodType(int method) {
    if (method != SAC_RANSAC) throw Error(PEB_E_UNSUPPORTED, "SACSegmentation: only SAC_RANSAC has a CUDA implementation");
  }
  void setOptimizeCoefficients(bool on) { p_.optimize_coefficients = on ? 1 : 0; }
  void setDistanceThreshold(double t) { p_.distance_threshold = t; }
  void setMaxIterations(int n) { p_.max_iterations = n; }
  void setProbability(double p) { p_.probability = p; }
  // inliers: ascending indices; coefficients: a b c d, or empty when no model was found (as PCL clears them)
  void segment(std::vector<int32_t>& inliers, std::vector<float>& coefficients) {
    if (!have_model_) throw Error(PEB_E_INVALID_ARG, "SACSegmentation::segment: no model type given (setModelType)");
    inliers.resize(in_.size ? in_.size : 1);
    coefficients.assign(4, 0.0f);
    size_t m = 0;
    int32_t its = 0;
    c_.check(peb_sac_plane(c_.get(), in_.data, in_.size, in_.stride, &p_, coefficients.data(), inliers.data(), &m, &its));
    inliers.resize(m);
    iterations_ = its;
    if (m == 0 && coefficients[0] == 0.0f && coefficients[1] == 0.0f && coefficients[2] == 0.0f && coefficients[3] == 0.0f)
      coefficients.clear();
  }
  int iterations() const { return iterations_; }

 private:
  Context& c_;
  CloudView in_;
  peb_sac_params p_;
  bool have_model_ = false;
  int iterations_ = 0;
};

class VoxelGrid {
 public:
  explicit VoxelGrid(Context& c) : c_(c) {}
  void setInputCloud(const void* pts, size_t n, size_t stride = 16) { in_ = {pts, n, stride}; }
  void setLeafSize(float lx, float ly, float lz) { leaf_[0] = lx, leaf_[1] = ly, leaf_[2] = lz; }
  void setMinimumPointsNumberPerVoxel(unsigned n) { min_pts_ = n; }
  unsigned getMinimumPointsNumberPerVoxel() const { return min_pts_; }
  // output: x y z 1 records (pcl::PointXYZ memory image), ascending voxel index
  void filter(std::vector<float>& out_xyz4) {
    out_xyz4.resize(4 * (in_.size ? in_.size : 1));
    size_t m = 0;
    c_.check(peb_voxel_grid(c_.get(), in_.data, in_.size, in_.stride, leaf_[0], leaf_[1], leaf_[2], min_pts_,
                            out_xyz4.data(), &m));
    out_xyz4.resize(4 * m);
  }

 private:
  Context& c_;
  CloudView in_;
  float leaf_[3] = {0, 0, 0};
  unsigned min_pts_ = 0;
};

class NormalEstimation {
 public:
  explicit NormalEstimation(Context& c) : c_(c) {}
  void setInputCloud(const void* pts, size_t n, size_t stride = 16) { in_ = {pts, n, stride}; }
  void setKSearch(int k) { k_ = k; }
  int getKSearch() const { return k_; }
  void setRadiusSearch(double r) {
    if (r != 0.0) throw Error(PEB_E_UNSUPPORTED, "NormalEstimation::setRadiusSearch has no CUDA path (no CPU fallback)");
  }
  void setViewPoint(float x, float y, float z) { vp_[0] = x, vp_[1] = y, vp_[2] = z; }
  // output: pcl::Normal records (nx ny nz 0 | curvature 0 0 0), 8 floats each
  void compute(std::vector<float>& out_normal8) {
    out_normal8.resize(8 * in_.size);
    c_.check(peb_normals_knn(c_.get(), in_.data, in_.size, in_.stride, k_, vp_, out_normal8.data()));
  }

 private:
  Context& c_;
  CloudView in_;
  int k_ = 0;
  float vp_[3] = {0, 0, 0};
};

// cv::ppf_match_3d::computeNormalsPC3d(pc, pc_normals, num_neighbors, flip_viewpoint, viewpoint) — the reference's
// normals slot (pose_estimation/src/opencv_surface_match.cpp:57-59) with OpenCV's arithmetic (peb_cv_normals).
// pc: rows of `stride` bytes whose first three floats are x y z (a CV_32F N x 3 or N x 6 Mat: ptr<float>(0), step);
// out6: rows x 6 floats x y z nx ny nz, e.g. pc_normals.ptr<float>(0) of a continuous CV_32F rows x 6 Mat.
inline void computeNormalsPC3d(Context& c, const float* pc, size_t rows, size_t stride, int num_neighbors, bool flip_viewpoint,
                               const float viewpoint[3], float* out6) {
  c.check(peb_cv_normals(c.get(), pc, rows, stride, num_neighbors, flip_viewpoint ? 1 : 0, viewpoint, out6, nullptr));
}

// pcl::registration::DefaultConvergenceCriteria<float>, the part reachable through getConvergeCriteria()
class ConvergenceCriteria {
 public:
  enum ConvergenceState {
    CONVERGENCE_CRITERIA_NOT_CONVERGED = PEB_NOT_CONVERGED,
    CONVERGENCE_CRITERIA_ITERATIONS = PEB_ITERATIONS,
    CONVERGENCE_CRITERIA_TRANSFORM = PEB_TRANSFORM,
    CONVERGENCE_CRITERIA_ABS_MSE = PEB_ABS_MSE,
    CONVERGENCE_CRITERIA_REL_MSE = PEB_REL_MSE,
    CONVERGENCE_CRITERIA_NO_CORRESPONDENCES = PEB_NO_CORRESPONDENCES,
    CONVERGENCE_CRITERIA_FAILURE_AFTER_MAX_ITERATIONS = PEB_FAILURE_AFTER_MAX_ITERATIONS
  };
  explicit ConvergenceCriteria(peb_icp_params& p) : p_(p) {}
  void setAbsoluteMSE(double v) { p_.abs_mse_threshold = v; }
  double getAbsoluteMSE() const { return p_.abs_mse_threshold; }
  void setMaximumIterationsSimilarTransforms(int n) { p_.max_iterations_similar = n; }
  ConvergenceState getConvergenceState() const { return static_cast<ConvergenceState>(state_); }

 private:
  friend class IterativeClosestPoint;
  peb_icp_params& p_;
  int state_ = PEB_NOT_CONVERGED;
};

class IterativeClosestPoint {
 public:
  explicit IterativeClosestPoint(Context& c, int estimator = PEB_ESTIMATOR_SVD) : c_(c), criteria_(params_) {
    peb_icp_params_default(&params_);
    params_.estimator = estimator;
    std::memset(&result_, 0, sizeof(result_));
    for (int i = 0; i < 4; ++i) result_.T[5 * i] = 1.0f;
  }
  virtual ~IterativeClosestPoint() = default;

  void setInputSource(const void* pts, size_t n, size_t stride = 16) {
    c_.check(peb_source_set(c_.get(), pts, n, stride));
    n_src_ = n;
  }
  // normals: nullable; pcl::Normal records have stride 32, the normal inside a pcl::PointNormal
  // is at (pts + 16 bytes, stride 48)
  void setInputTarget(const void* pts, size_t n, size_t stride = 16, const void* normals = nullptr, size_t nstride = 32) {
    c_.check(peb_target_set(c_.get(), pts, n, stride, normals, nstride));
  }
  void setMaximumIterations(int n) { params_.max_iterations = n; }
  int getMaximumIterations() const { return params_.max_iterations; }
  void setMaxCorrespondenceDistance(double d) { params_.max_corr_dist = d; }
  double getMaxCorrespondenceDistance() const { return params_.max_corr_dist; }
  void setTransformationEpsilon(double e) { params_.transformation_epsilon = e; }
  void setTransformationRotationEpsilon(double e) { params_.rotation_epsilon = e; }
  void setEuclideanFitnessEpsilon(double e) { params_.euclidean_fitness_epsilon = e; }
  void setUseReciprocalCorrespondences(bool on) {
    if (on) throw Error(PEB_E_UNSUPPORTED, "reciprocal correspondences have no CUDA path (no CPU fallback)");
  }
  void setRANSACIterations(int n) {
    if (n) throw Error(PEB_E_UNSUPPORTED, "the RANSAC rejector has no CUDA path (no CPU fallback)");
  }
  // addCorrespondenceRejector(CorrespondenceRejectorDistance with setMaximumDistance(d)): before any other rejector it
  // sets params().rejector_max_dist, the head of the chain; after one it joins the chain, so PCL's order is kept
  void addCorrespondenceRejectorDistance(double max_distance) {
    if (chain_.empty()) params_.rejector_max_dist = max_distance;
    else add_rejector(PEB_REJECTOR_DISTANCE, max_distance, 0);
  }
  // addCorrespondenceRejector(CorrespondenceRejectorMedianDistance with setMedianFactor(factor))
  void addCorrespondenceRejectorMedianDistance(double factor = 1.0) { add_rejector(PEB_REJECTOR_MEDIAN_DISTANCE, factor, 0); }
  // addCorrespondenceRejector(CorrespondenceRejectorOneToOne)
  void addCorrespondenceRejectorOneToOne() { add_rejector(PEB_REJECTOR_ONE_TO_ONE, 0.0, 0); }
  // addCorrespondenceRejector(CorrespondenceRejectorTrimmed with setOverlapRatio(ratio), setMinCorrespondences(min_corr))
  void addCorrespondenceRejectorTrimmed(double ratio = 0.5, int min_corr = 0) { add_rejector(PEB_REJECTOR_TRIMMED, ratio, min_corr); }
  // the rejectors after params().rejector_max_dist, in the order they were added (peb_icp_align_ex)
  const std::vector<peb_rejector>& correspondenceRejectors() const { return chain_; }
  ConvergenceCriteria* getConvergeCriteria() { return &criteria_; }

  // align(output, guess): out_xyz4 (nullable) receives final * input as x y z 1 records
  void align(std::vector<float>* out_xyz4 = nullptr, const float* guess16 = nullptr) {
    if (out_xyz4) out_xyz4->resize(4 * n_src_);
    float* out = out_xyz4 && n_src_ ? out_xyz4->data() : nullptr;
    if (chain_.empty()) c_.check(peb_icp_align(c_.get(), guess16, &params_, &result_, out, nullptr, nullptr));
    else c_.check(peb_icp_align_ex(c_.get(), guess16, &params_, chain_.data(), chain_.size(), &result_, out, nullptr, nullptr));
    criteria_.state_ = result_.state;
  }
  // H initial poses against one source / one target: the call shape of
  // cv::ppf_match_3d::ICP::registerModelToScene(model, scene, poses), opencv_surface_match.cpp:94
  void alignBatch(const float* guesses16, size_t n_guesses, std::vector<peb_icp_result>& results) {
    results.resize(n_guesses);
    if (chain_.empty()) c_.check(peb_icp_align_batch(c_.get(), guesses16, n_guesses, &params_, results.data()));
    else c_.check(peb_icp_align_batch_ex(c_.get(), guesses16, n_guesses, &params_, chain_.data(), chain_.size(), results.data()));
  }
  bool hasConverged() const { return result_.converged != 0; }
  const float* getFinalTransformation() const { return result_.T; }  // column-major 4x4
  double getFitnessScore(double max_range = DBL_MAX) {
    if (max_range == params_.fitness_max_range) return result_.fitness;
    double f = 0;
    c_.check(peb_fitness_score(c_.get(), result_.T, max_range, &f, nullptr));
    return f;
  }
  int nr_iterations() const { return result_.iterations; }
  const peb_icp_result& result() const { return result_; }
  const peb_icp_params& params() const { return params_; }

 private:
  void add_rejector(int kind, double value, int min_corr) {
    if (chain_.size() >= PEB_MAX_REJECTORS)
      throw Error(PEB_E_INVALID_ARG, "at most " + std::to_string(PEB_MAX_REJECTORS) + " correspondence rejectors after the distance one");
    peb_rejector r;
    r.kind = kind;
    r.min_correspondences = min_corr;
    r.value = value;
    chain_.push_back(r);
  }
  std::vector<peb_rejector> chain_;

 protected:
  Context& c_;
  peb_icp_params params_;
  peb_icp_result result_;
  ConvergenceCriteria criteria_;
  size_t n_src_ = 0;
};

// ---- the step right after the path (SURVEY.md 8f rank 3): host-side, no device work ----------------
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

// rotation part of a column-major 4x4 -> unit quaternion (w, x, y, z), w >= 0
inline void rotation_to_quat(const float* T16, double q[4]) {
  const double m00 = T16[0], m10 = T16[1], m20 = T16[2], m01 = T16[4], m11 = T16[5], m21 = T16[6], m02 = T16[8],
               m12 = T16[9], m22 = T16[10];
  const double tr = m00 + m11 + m22;
  if (tr > 0.0) {
    const double s = std::sqrt(tr + 1.0) * 2.0;
    q[0] = 0.25 * s, q[1] = (m21 - m12) / s, q[2] = (m02 - m20) / s, q[3] = (m10 - m01) / s;
  } else if (m00 > m11 && m00 > m22) {
    const double s = std::sqrt(1.0 + m00 - m11 - m22) * 2.0;
    q[0] = (m21 - m12) / s, q[1] = 0.25 * s, q[2] = (m01 + m10) / s, q[3] = (m02 + m20) / s;
  } else if (m11 > m22) {
    const double s = std::sqrt(1.0 + m11 - m00 - m22) * 2.0;
    q[0] = (m02 - m20) / s, q[1] = (m01 + m10) / s, q[2] = 0.25 * s, q[3] = (m12 + m21) / s;
  } else {
    const double s = std::sqrt(1.0 + m22 - m00 - m11) * 2.0;
    q[0] = (m10 - m01) / s, q[1] = (m02 + m20) / s, q[2] = (m12 + m21) / s, q[3] = 0.25 * s;
  }
  if (q[0] < 0.0)
    for (int i = 0; i < 4; ++i) q[i] = -q[i];
}

// The 7 floats the node publishes, {x, y, z, qx, qy, qz, qw} (pose_estimation/include/pose_estimation.hpp:83-88).
// reference_layout = true reproduces opencv_surface_match.cpp:133-142 literally: pose[5] (qz) is never
// written and pose[6] receives q[3] and is then overwritten with q[0] — so qz is lost and left 0.
inline void pack_pose(const float* T16, float pose7[7], bool reference_layout = false) {
  double q[4];
  rotation_to_quat(T16, q);
  for (int i = 0; i < 3; ++i) pose7[i] = T16[12 + i];
  pose7[3] = static_cast<float>(q[1]);
  pose7[4] = static_cast<float>(q[2]);
  if (reference_layout) {
    pose7[5] = 0.0f;
    pose7[6] = static_cast<float>(q[3]);
    pose7[6] = static_cast<float>(q[0]);
  } else {
    pose7[5] = static_cast<float>(q[3]);
    pose7[6] = static_cast<float>(q[0]);
  }
}

// cv::ppf_match_3d::ICP as the reference constructs and calls it (pose_estimation/src/opencv_surface_match.cpp:85-94):
// ICP icp(250, 0.005f, 2.5f, 8); icp.registerModelToScene(model, scene_with_normals, poses).  Clouds are the N x 6
// CV_32F rows of OpenCV (x y z nx ny nz, cv::Mat::ptr<float>(0) of a continuous Mat); a pose is the 16 doubles of
// Pose3D::pose (cv::Matx44d::val, row-major) and is updated in place like Pose3D::appendPose; residual -> Pose3D::residual.
class CvIcp {
 public:
  CvIcp(Context& c, int iterations = 250, float tolerance = 0.05f, float rejection_scale = 2.5f, int num_levels = 6) : c_(c) {
    p_.iterations = iterations;
    p_.num_levels = num_levels;
    p_.tolerance = tolerance;
    p_.rejection_scale = rejection_scale;
  }
  void registerModelToScene(const float* model_xyzn, size_t n_model, const float* scene_xyzn, size_t n_scene, double* poses16,
                            size_t n_poses, double* residuals) {
    c_.check(peb_cvicp_register(c_.get(), model_xyzn, n_model, scene_xyzn, n_scene, &p_, poses16, n_poses, residuals));
  }

 private:
  Context& c_;
  peb_cvicp_params p_;
};

// cv::ppf_match_3d::PPF3DDetector as the reference constructs and calls it
// (pose_estimation/src/opencv_surface_match.cpp:45-46: detectors_[name] = PPF3DDetector(0.03, 0.03, 40);
// detectors_[name].trainModel(models_[name]); :65: detectors_[object].match(pc_scene_normals, results, 1.0, 0.03)).
// Clouds are the N x 6 CV_32F rows of OpenCV; a result is peb_ppf_pose = cv::ppf_match_3d::Pose3D (pose row-major like
// cv::Matx44d::val, q = w x y z, t, angle, numVotes, modelIndex, residual), clustered, most votes first — the vector the
// reference truncates to six poses and hands to ICP::registerModelToScene (CvIcp above).
class PPF3DDetector {
 public:
  explicit PPF3DDetector(Context& c, double relativeSamplingStep = 0.05, double relativeDistanceStep = 0.05, double numAngles = 30)
      : c_(c) {
    peb_ppf_params_default(&p_);
    p_.relative_sampling_step = relativeSamplingStep;
    p_.relative_distance_step = relativeDistanceStep;
    p_.num_angles = numAngles;
  }
  ~PPF3DDetector() { peb_ppf_model_destroy(m_); }
  PPF3DDetector(const PPF3DDetector&) = delete;
  PPF3DDetector& operator=(const PPF3DDetector&) = delete;
  void setSearchParams(double positionThreshold = -1, double rotationThreshold = -1, bool useWeightedClustering = false) {
    p_.position_threshold = positionThreshold;
    p_.rotation_threshold = rotationThreshold;
    p_.use_weighted_avg = useWeightedClustering ? 1 : 0;
  }
  void trainModel(const float* model_xyzn, size_t n_model) {
    peb_ppf_model_destroy(m_);
    m_ = nullptr;
    c_.check(peb_ppf_train(c_.get(), model_xyzn, n_model, &p_, &m_));
  }
  void match(const float* scene_xyzn, size_t n_scene, std::vector<peb_ppf_pose>& results, double relativeSceneSampleStep = 1.0 / 5.0,
             double relativeSceneDistance = 0.03) {
    if (!m_) throw Error(PEB_E_INVALID_ARG, "PPF3DDetector::match: the model is not trained");
    size_t n = 0;
    results.resize(64);
    c_.check(peb_ppf_match(c_.get(), m_, scene_xyzn, n_scene, relativeSceneSampleStep, relativeSceneDistance, results.data(),
                           results.size(), &n, nullptr, 0, nullptr));
    if (n > results.size()) {  // more clusters than the first guess: ask again with room for all of them
      results.resize(n);
      c_.check(peb_ppf_match(c_.get(), m_, scene_xyzn, n_scene, relativeSceneSampleStep, relativeSceneDistance, results.data(),
                             results.size(), &n, nullptr, 0, nullptr));
    }
    results.resize(n);
  }

 private:
  Context& c_;
  peb_ppf_params p_;
  peb_ppf_model* m_ = nullptr;
};

// The manager's side of the pose (pose_estimation_manager/src/pose_transformer.cpp:78-121, PoseTransformer::obj_in_base_frame):
// the published {x, y, z, qx, qy, qz, qw} (camera frame) -> hand-eye calibration (row-major 4x4, he_calibration_mat_) -> the
// grasp frame sent to the robot: the object's y axis is kept, z is the base's -z (or +x when y is more than ~37 degrees out of
// the horizontal) made orthogonal to y, x = y x z.  float like the reference's Eigen types; out7 = 7 doubles.
inline void obj_in_base_frame(const float pose7[7], const float he16[16], double out7[7]) {
  float q[4] = {pose7[3], pose7[4], pose7[5], pose7[6]};  // x y z w
  const float qn = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (float& v : q) v /= qn;
  const float x = q[0], y = q[1], z = q[2], w = q[3];
  const float R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * w),     2 * (x * z + y * w),
                      2 * (x * y + z * w),     1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                      2 * (x * z - y * w),     2 * (y * z + x * w),     1 - 2 * (x * x + y * y)};
  float cam[16] = {R[0], R[1], R[2], pose7[0], R[3], R[4], R[5], pose7[1], R[6], R[7], R[8], pose7[2], 0, 0, 0, 1};
  float base[16];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      float a = 0.0f;
      for (int k = 0; k < 4; ++k) a += he16[4 * r + k] * cam[4 * k + c];
      base[4 * r + c] = a;
    }
  const float yv[3] = {base[1], base[5], base[9]};
  float zb[3] = {0.0f, 0.0f, -1.0f};
  if (std::fabs(yv[2]) > 0.6f) zb[0] = 1.0f, zb[2] = 0.0f;
  const float f = (zb[0] * yv[0] + zb[1] * yv[1] + zb[2] * yv[2]) / (yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
  const float zv[3] = {zb[0] - f * yv[0], zb[1] - f * yv[1], zb[2] - f * yv[2]};
  const float xv[3] = {yv[1] * zv[2] - yv[2] * zv[1], yv[2] * zv[0] - yv[0] * zv[2], yv[0] * zv[1] - yv[1] * zv[0]};
  auto norm3 = [](const float* v) { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); };
  const float nx = norm3(xv), ny = norm3(yv), nz = norm3(zv);
  float T[16] = {0};  // column-major for rotation_to_quat: columns x, y, z
  for (int i = 0; i < 3; ++i) {
    T[i] = xv[i] / nx;
    T[4 + i] = yv[i] / ny;
    T[8 + i] = zv[i] / nz;
  }
  // Eigen::Quaternionf(Matrix3f): no sign normalisation
  const float m00 = T[0], m10 = T[1], m20 = T[2], m01 = T[4], m11 = T[5], m21 = T[6], m02 = T[8], m12 = T[9], m22 = T[10];
  const float m[3][3] = {{m00, m01, m02}, {m10, m11, m12}, {m20, m21, m22}};
  float qo[4];  // x y z w
  float t = m00 + m11 + m22;
  if (t > 0.0f) {
    t = std::sqrt(t + 1.0f);
    qo[3] = 0.5f * t;
    t = 0.5f / t;
    qo[0] = (m21 - m12) * t;
    qo[1] = (m02 - m20) * t;
    qo[2] = (m10 - m01) * t;
  } else {
    int i = 0;
    if (m11 > m00) i = 1;
    if (m22 > m[i][i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = std::sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0f);
    qo[i] = 0.5f * t;
    t = 0.5f / t;
    qo[3] = (m[k][j] - m[j][k]) * t;
    qo[j] = (m[j][i] + m[i][j]) * t;
    qo[k] = (m[k][i] + m[i][k]) * t;
  }
  const float qm = std::sqrt(qo[0] * qo[0] + qo[1] * qo[1] + qo[2] * qo[2] + qo[3] * qo[3]);
  out7[0] = base[3], out7[1] = base[7], out7[2] = base[11];
  for (int i = 0; i < 4; ++i) out7[3 + i] = qo[i] / qm;
}

class IterativeClosestPointWithNormals : public IterativeClosestPoint {
 public:
  explicit IterativeClosestPointWithNormals(Context& c) : IterativeClosestPoint(c, PEB_ESTIMATOR_POINT_TO_PLANE_LLS) {}
};

// ---- every GPU of the box from the node's one process (peb_multi_*, SURVEY.md 8e) ---------------------
// owns one peb_multi: one context per device, scene grid and model replicated on each
class MultiContext {
 public:
  explicit MultiContext(const std::vector<int>& devices) {
    if (int rc = peb_multi_create(static_cast<int>(devices.size()), devices.data(), &m_)) throw Error(rc, peb_multi_last_error(nullptr));
  }
  ~MultiContext() { peb_multi_destroy(m_); }
  MultiContext(const MultiContext&) = delete;
  MultiContext& operator=(const MultiContext&) = delete;
  peb_multi* get() const { return m_; }
  int size() const { return peb_multi_size(m_); }
  void check(int rc) const {
    if (rc != PEB_OK) throw Error(rc, peb_multi_last_error(m_));
  }

 private:
  peb_multi* m_ = nullptr;
};

// The batched refinement of the slot (opencv_surface_match.cpp:85-94) sharded over the devices of a MultiContext:
// contiguous blocks of the H poses per device, results in hypothesis order, identical to alignBatch on one device.
// Configure a pe_b200::IterativeClosestPoint(+WithNormals) with PCL's setters as usual and hand it over as `like`.
class MultiDeviceICP {
 public:
  MultiDeviceICP(MultiContext& m, const IterativeClosestPoint& like)
      : m_(m), params_(like.params()), chain_(like.correspondenceRejectors()) {}
  void setInputSource(const void* pts, size_t n, size_t stride = 16) { m_.check(peb_multi_source_set(m_.get(), pts, n, stride)); }
  void setInputTarget(const void* pts, size_t n, size_t stride = 16, const void* normals = nullptr, size_t nstride = 32) {
    m_.check(peb_multi_target_set(m_.get(), pts, n, stride, normals, nstride));
  }
  void alignBatch(const float* guesses16, size_t n_guesses, std::vector<peb_icp_result>& results) {
    results.resize(n_guesses);
    if (chain_.empty()) m_.check(peb_multi_icp_align_batch(m_.get(), guesses16, n_guesses, &params_, results.data()));
    else m_.check(peb_multi_icp_align_batch_ex(m_.get(), guesses16, n_guesses, &params_, chain_.data(), chain_.size(), results.data()));
  }

 private:
  MultiContext& m_;
  peb_icp_params params_;
  std::vector<peb_rejector> chain_;
};

}  // namespace pe_b200
