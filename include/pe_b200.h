/*
 * pe_b200.h — C ABI of libpe_b200.so, the B200 (sm_100a) pose-refinement path.
 *
 * This is the drop-in boundary. Every entry point replaces one PCL 1.10 call that the
 * north-star path substitutes into the refinement / normals / down-sample slots of
 * yumi-crew/pose_estimation:
 *
 *   refinement slot   pose_estimation/src/opencv_surface_match.cpp:85-94
 *   normals slot      pose_estimation/src/opencv_surface_match.cpp:57-59
 *   down-sample slot  pose_estimation/src/pose_estimation.cpp:261-263
 *
 * PCL itself is not vendored in the reference; "[PCL] file" below names the upstream
 * pcl-1.10.0 file whose behaviour the entry point reproduces (SURVEY.md section 8a).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++ or torch types, no exceptions across the ABI.
 *   - point clouds are passed as (pointer, count, stride-in-bytes); the first three
 *     floats of every record are x,y,z.  stride 16 = pcl::PointXYZ, 48 = pcl::PointNormal,
 *     12 / 24 = rows of a cv::Mat N x 3 / N x 6 CV_32F.
 *   - every call returns 0 (PEB_OK) or a negative peb_status; the text of the last error
 *     is available from peb_last_error().  Numerical outcomes (too few correspondences,
 *     iteration cap) are not errors: they are reported in peb_icp_result like PCL does.
 *   - a peb_ctx is bound to one CUDA device and one stream; calls on one context must be
 *     serialised by the caller (the node has a single executor thread).  Distinct
 *     contexts are independent.
 *   - there is no CPU fallback: every entry point either runs the CUDA path or fails.
 */
#ifndef PE_B200_H_
#define PE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PEB_API
#else
#define PEB_API __attribute__((visibility("default")))
#endif

typedef struct peb_ctx peb_ctx;

typedef enum peb_status {
  PEB_OK = 0,
  PEB_E_INVALID_ARG = -1,
  PEB_E_NO_TARGET = -2,  /* align / fitness called before peb_target_set            */
  PEB_E_NO_SOURCE = -3,  /* align called before peb_source_set                      */
  PEB_E_CUDA = -4,
  PEB_E_OOM = -5,
  PEB_E_UNSUPPORTED = -6 /* PCL option with no CUDA implementation (no CPU fallback) */
} peb_status;

/* pcl::registration::DefaultConvergenceCriteria<float>::ConvergenceState, same order.
 * [PCL] registration/include/pcl/registration/default_convergence_criteria.h */
typedef enum peb_convergence_state {
  PEB_NOT_CONVERGED = 0,
  PEB_ITERATIONS = 1,
  PEB_TRANSFORM = 2,
  PEB_ABS_MSE = 3,
  PEB_REL_MSE = 4,
  PEB_NO_CORRESPONDENCES = 5,
  PEB_FAILURE_AFTER_MAX_ITERATIONS = 6,
  /* not a PCL state: a device-side dependency wait between two iteration launches ran into its bound
   * (a bug, never data-dependent); every record of that align carries it and the host-buffer entry
   * points return PEB_E_CUDA */
  PEB_STATE_INTERNAL_ERROR = -1000
} peb_convergence_state;

enum { PEB_ESTIMATOR_SVD = 0, PEB_ESTIMATOR_POINT_TO_PLANE_LLS = 1 };

/* The setters of pcl::Registration / pcl::IterativeClosestPoint and of its
 * DefaultConvergenceCriteria, as one POD.  peb_icp_params_default() fills PCL 1.10's
 * defaults.  [PCL] registration/include/pcl/registration/registration.h, icp.h */
typedef struct peb_icp_params {
  int32_t max_iterations;             /* setMaximumIterations           (10)            */
  int32_t min_correspondences;        /* min_number_correspondences_    (3)             */
  int32_t estimator;                  /* PEB_ESTIMATOR_*                (SVD)           */
  int32_t max_iterations_similar;     /* setMaximumIterationsSimilarTransforms (0)      */
  double max_corr_dist;               /* setMaxCorrespondenceDistance   (sqrt(DBL_MAX)) */
  double transformation_epsilon;      /* setTransformationEpsilon       (0)             */
  double rotation_epsilon;            /* setTransformationRotationEpsilon (0)           */
  double euclidean_fitness_epsilon;   /* setEuclideanFitnessEpsilon     (-DBL_MAX)      */
  double abs_mse_threshold;           /* getConvergeCriteria()->setAbsoluteMSE (1e-12)  */
  double rejector_max_dist;           /* CorrespondenceRejectorDistance::setMaximumDistance;
                                         <= 0 : no rejector (PCL's ICP default)        */
  double fitness_max_range;           /* getFitnessScore(max_range)     (DBL_MAX)       */
} peb_icp_params;

/* What pcl::Registration exposes after align().  T is column-major, i.e. memcpy-compatible
 * with Eigen::Matrix4f::data() of getFinalTransformation(). */
typedef struct peb_icp_result {
  float T[16];
  double fitness;          /* getFitnessScore(fitness_max_range)                        */
  double last_mse;         /* correspondences_cur_mse_ of the last evaluated iteration  */
  int32_t iterations;      /* nr_iterations_                                            */
  int32_t converged;       /* hasConverged()                                            */
  int32_t state;           /* peb_convergence_state                                     */
  int32_t n_correspondences; /* size of the last correspondence set                     */
} peb_icp_result;

/* ---- context ------------------------------------------------------------------- */
PEB_API int peb_ctx_create(int device, peb_ctx** out);
PEB_API void peb_ctx_destroy(peb_ctx* ctx);
/* never NULL; valid until the next call on ctx (ctx == NULL: message of the last failed
 * peb_ctx_create on this thread) */
PEB_API const char* peb_last_error(const peb_ctx* ctx);
PEB_API const char* peb_version(void);
PEB_API void peb_icp_params_default(peb_icp_params* p);
/* the cudaStream_t all work of this context is ordered on (for event timing) */
PEB_API void* peb_ctx_stream(peb_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches claim) */
PEB_API uint64_t peb_ctx_launch_count(const peb_ctx* ctx);
/* tuning knobs that change speed, never results (tests/test_gpu_parity.py asserts bit-identical records for
 * every one of them; the exception are the block-count knobs "blocks_factor" / "blocks_factor_cold" — and "nn_group" in
 * a batch, which changes launch 0's block count —: they change the ORDER in which the per-block partial sums of the
 * double moments are added, i.e. at most their last bits): "nn_group" (lanes per COLD nearest-neighbour query: 1, 2, 4, 8, 16),
 * "grid_occupancy_x100" (wanted points per occupied target-grid cell x 100, default 500; takes effect at
 * the next peb_target_set), "source_sort_occupancy" (points per cell of the source's own sort grid = patch
 * compactness, default 32), "warm_start" (iterations >= 1 seed their search with the previous match),
 * "anchor_seed" / "seed_guard_x10" / "coop_max_rows" (first iteration of a batch: one anchor search per
 * 32-point patch, how far a point may be from its anchor in cells x 10, and up to how many grid rows a patch
 * verifies its candidates warp-cooperatively; 0 = per lane), "batch_streams" (independent chains of launches
 * of a batched align, 0 = auto), "blocks_factor" / "blocks_factor_cold" (blocks per SM and launch, 0 = auto),
 * "split_moments" (default 1: every iteration of a batch runs as a search launch — nearest neighbours only, more
 * resident warps — and a moment launch that recomputes the correspondences' distances, sums the moments in the order of
 * the fused kernel and solves — icp.cu : icp_search_kernel; byte-identical records; 0 = one fused launch per
 * iteration) in batches of at least "split_min_hyp" (default 256; smaller batches measured no faster split) hypotheses,
 * "blocks_factor_search" (blocks per SM of those search launches, 0 = like the iteration's moment launch; results do
 * not depend on it),
 * "flag_deps" (warm launches of a batch wait per hypothesis instead of for the whole previous grid),
 * "pdl" (programmatic dependent launch), "cert_margin_x1000" (search-skipping certificates, off),
 * "profile" (0 / 1 / 2, see peb_profile_read), "debug_timers" (development),
 * "warm_upfront" (default 0; 1 / 2: warm searches whose ball spans up to 2 x 2 grid rows fetch all row bounds up
 * front, 3: up to 3 x 3 — csrc/nn_upfront.cuh; bit-identical results, measured SLOWER on B200 (C4: -4 % and -19 %,
 * profiles/README.md round 2) and kept only as a recorded experiment; "warm_upfront_from": the first iteration
 * launch that uses it, default 2), "nn_cache_from" / "nn_cache_r_x100" (candidate cache of the warm launches,
 * csrc/nn_cache.cuh; bit-identical, measured slower, off), "warm_bin" (default 0; 1: the warm launches of a batch
 * sort the queries of a block by the number of grid rows their search walks before the warps search them —
 * icp.cu : icp_iteration_binned_kernel; bit-identical by construction, measured -6 % on C4,
 * profiles/r2_p_warm_bin.txt),
 * "warm_graph" (default 1: the warm launches of a batch of at least "warm_graph_min_hyp" (32) hypotheses search over a
 * 12-nearest-neighbour graph of the target, built once per target — csrc/nn_graph.cuh: the row of the previous match
 * proves most answers without a grid walk; byte-identical records, C4 11 480 -> 16 330 hypotheses/s),
 * "warm_graph_kappa_x100" (default 0 = every hypothesis from launch 1 on; > 0: a hypothesis takes the graph once
 * 4 x its last MSE x kappa is below the mean outer bound of the rows), "cold_graph" (default 1: launch 0 of such a batch
 * takes its candidates from a greedy descent on the graph instead of a 3 x 3 x 3 probe), "warm_graph_flat" (default 1) with "warm_graph_flat_from" / "warm_graph_flat_until"
 * (default 2 / 15: the iteration launches whose graph searches also try the flatness certificate of nn_graph.cuh — a residual
 * along the local surface normal is proven far beyond the triangle inequality), "warm_graph_peek" (default 1: in graph launches 1 .. this, a query whose row cannot certify
 * looks at the four nearest neighbours of its previous match before it walks the grid), "warm_graph_queue" (default 0;
 * 8 / 16: every warp queues the unproven queries of a tile of that many passes and walks the grid for them 32 at a
 * time — icp.cu : icp_iteration_graphq_kernel; byte-identical, measured -7 %, profiles/r2_ai_graph_queue.txt).
 * An align with a rejector chain (peb_icp_align_ex) always runs split with whole-grid launch dependencies: there
 * "split_moments", "split_min_hyp", "cert_margin_x1000", "warm_bin", "warm_graph_queue", "nn_cache_from",
 * "warm_upfront", "nn_group" and "flag_deps" have no effect. */
PEB_API int peb_ctx_set_int(peb_ctx* ctx, const char* key, int value);

/* ---- pcl::VoxelGrid<PointXYZ>::filter  [PCL] filters/.../impl/voxel_grid.hpp -------- */
/* out_xyz4 must hold n x 4 floats (the overflow guard returns the input unchanged).
 * Output order: ascending voxel index, x fastest, like PCL.  min_pts = setMinimumPointsNumberPerVoxel. */
PEB_API int peb_voxel_grid(peb_ctx* ctx, const void* pts, size_t n, size_t stride,
                           float leaf_x, float leaf_y, float leaf_z, unsigned min_pts,
                           float* out_xyz4, size_t* out_n);

/* ---- scene pre-filter: the deterministic part of PoseEstimation::create_surface_match_pc -------- */
/* (SURVEY.md 8f rank 1, the step right before the path)
 *   pcl::removeNaNFromPointCloud                      pose_estimation/src/pose_estimation.cpp:246-248
 *   PoseEstimation::filter_points (sphere filter)     pose_estimation/src/pose_estimation.cpp:347-372
 *   the 5 mm band removal of remove_planes            pose_estimation/src/pose_estimation.cpp:309-333
 * applied in that order, in one fused pass; survivors keep their original order (the reference's
 * own order depends on OpenMP scheduling).  The RANSAC fit that produces the plane coefficients
 * (pcl::SACSegmentation) is peb_sac_plane below: its coefficients are inputs of this call. */
enum { PEB_PREFILTER_MAX_PLANES = 8 };
typedef struct peb_prefilter_params {
  int32_t use_sphere;          /* filter_points() is applied                                   */
  int32_t remove_inliers;      /* filter_out == "inliers": drop the points INSIDE the sphere     */
  float sphere_center[3];      /* filter_pose_[0..2]                                             */
  float sphere_radius;         /* filter_radius_                                                 */
  int32_t n_planes;            /* plane coefficient sets applied one after the other             */
  float plane_band;            /* 0.005 in the reference                                         */
  float planes[4 * PEB_PREFILTER_MAX_PLANES]; /* a b c d of ax + by + cz + d = 0                 */
} peb_prefilter_params;
/* out_xyz4 must hold n x 4 floats; records are x y z 1 */
PEB_API int peb_scene_prefilter(peb_ctx* ctx, const void* pts, size_t n, size_t stride,
                                const peb_prefilter_params* params, float* out_xyz4, size_t* out_n);
PEB_API int peb_scene_prefilter_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const peb_prefilter_params* params,
                                    void* d_out_xyz4, size_t* out_n);

/* ---- pcl::SACSegmentation<pcl::PointXYZ>::segment, SACMODEL_PLANE + SAC_RANSAC ----------------
 * The plane fit of the reference's remove_planes (pose_estimation/src/pose_estimation.cpp:285-297:
 * distance threshold 0.0001, 100 iterations, optimised coefficients), the one step of the scene
 * preparation that peb_scene_prefilter takes as an input.
 * [PCL] segmentation/impl/sac_segmentation.hpp (segment), sample_consensus/impl/ransac.hpp
 * (computeModel: adaptive iteration count k = log(1 - p) / log(1 - w^3), skipped samples),
 * sample_consensus/sac_model.h (drawIndexSample: boost::mt19937 seeded with 12345 when the model is
 * not "random", uniform_int<>(0, INT_MAX), partial Fisher-Yates on the persistent index shuffle),
 * sample_consensus/impl/sac_model_plane.hpp (isSampleGood, computeModelCoefficients,
 * countWithinDistance, selectWithinDistance, optimizeModelCoefficients = PCA of the inliers).
 * The sample sequence does not depend on the data, so all candidate planes of a run are drawn on
 * the host first, their inliers are counted in ONE pass over the cloud on the device, and the
 * sequential loop (best-so-far, adaptive k) is replayed on the counts: same decisions as PCL's loop.
 * The inlier moments are accumulated in double (PCL 1.10: float, single pass — see DESIGN.md). */
typedef struct peb_sac_params {
  double distance_threshold;     /* setDistanceThreshold                      (PCL default 0)     */
  double probability;            /* setProbability                            (PCL default 0.99)  */
  int32_t max_iterations;        /* setMaxIterations                          (PCL default 50)    */
  int32_t optimize_coefficients; /* setOptimizeCoefficients                   (PCL default true)  */
  uint32_t seed;                 /* 12345: SampleConsensusModel(random = false)                   */
  int32_t reserved;
} peb_sac_params;
PEB_API void peb_sac_params_default(peb_sac_params* p);
/* out_coeff: a b c d of ax + by + cz + d = 0 (all 0 when no model was found);
 * out_inliers (nullable): up to n indices, ascending; out_iterations (nullable): RANSAC iterations run */
PEB_API int peb_sac_plane(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_sac_params* params,
                          float out_coeff[4], int32_t* out_inliers, size_t* out_n_inliers, int32_t* out_iterations);
/* d_out_inliers: nullable DEVICE buffer of n int32 */
PEB_API int peb_sac_plane_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const peb_sac_params* params,
                              float out_coeff[4], int32_t* d_out_inliers, size_t* out_n_inliers, int32_t* out_iterations);

/* ---- PoseEstimation::create_surface_match_pc in one call ------------------------------------------
 * pose_estimation/src/pose_estimation.cpp:246-261 (+ remove_planes :281-345): NaN removal, the optional sphere
 * filter, then num_planes times { plane RANSAC on what is left; removal of the plane band }, then — if
 * leaf > 0 — VoxelGrid.  Same arithmetic and results as peb_scene_prefilter / peb_sac_plane / peb_voxel_grid
 * called one after the other, but the cloud crosses PCIe once in each direction instead of seven times.
 * filter: use_sphere / remove_inliers / sphere_* / plane_band are read, its planes are ignored.
 * out_planes (nullable): num_planes x 4 coefficients; a plane that could not be estimated is all zeros and
 * removes nothing.  DELIBERATE DEVIATION: the reference's remove_planes applies its band test unconditionally
 * (pose_estimation.cpp:313-333) — after a failed segment() PCL leaves `coefficients->values` EMPTY, so the
 * reference indexes an empty vector there (undefined behaviour, there is nothing to reproduce); this library keeps
 * every point of such a pass (tests/test_sac.py::test_scene_prepare_keeps_everything_when_no_plane_is_found). */
PEB_API int peb_scene_prepare(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_prefilter_params* filter,
                              int num_planes, const peb_sac_params* sac, float leaf, float* out_xyz4, size_t* out_n,
                              float* out_planes);

/* ---- cv::ppf_match_3d::ICP::registerModelToScene(model, scene, poses) --------------------------
 * What the reference runs in the refinement slot (pose_estimation/src/opencv_surface_match.cpp:85-94:
 * ICP icp(250, 0.005f, 2.5f, 8); icp.registerModelToScene(models_[object], pc_scene_normals, <= 6 poses)).
 * [CV] opencv_contrib/modules/surface_matching/src/icp.cpp (not in the reference tree nor in this
 * image: restated from recollection, see DESIGN.md section 9): per pose the model is moved by the pose,
 * both clouds are centred and scaled, and a numLevels pyramid of point-to-plane ICP runs with
 * median/MAD rejection, many-to-one ("picky") elimination and the linearised 6-parameter step.
 * model, scene: n x 6 float rows (x y z nx ny nz = cv::Mat CV_32F with normals).
 * poses: n_poses x 16 doubles, row-major 4 x 4 (cv::Matx44d::val), updated IN PLACE like
 * Pose3D::appendPose (pose <- icp_pose * pose); out_residuals: n_poses doubles (Pose3D::residual). */
typedef struct peb_cvicp_params {
  int32_t iterations;      /* ICP(iterations, ...)      : 250 in the reference */
  int32_t num_levels;      /* ICP(..., numLevels)       : 8                    */
  float tolerance;         /* ICP(.., tolerance, ..)    : 0.005                */
  float rejection_scale;   /* ICP(.., rejectionScale,.) : 2.5 (<= 0: no robust rejection) */
} peb_cvicp_params;
PEB_API int peb_cvicp_register(peb_ctx* ctx, const float* model_xyzn, size_t n_model, const float* scene_xyzn,
                               size_t n_scene, const peb_cvicp_params* params, double* poses, size_t n_poses,
                               double* out_residuals);

/* ---- cv::ppf_match_3d::PPF3DDetector: trainModel / match (coarse matching, SURVEY.md 8f rank 4) -------------
 * What the reference runs in front of the refinement slot:
 *   detectors_[name] = cv::ppf_match_3d::PPF3DDetector(0.03, 0.03, 40); detectors_[name].trainModel(model)
 *                                                     (pose_estimation/src/opencv_surface_match.cpp:37-51)
 *   detectors_[object].match(pc_scene_normals, results, 1.0, 0.03)   (pose_estimation/src/opencv_surface_match.cpp:65)
 * [CV] opencv_contrib/modules/surface_matching/src/ppf_match_3d.cpp, ppf_helpers.cpp, pose_3d.cpp (not in the
 * reference tree nor in this image: restated from recollection, parity unpinned — DESIGN.md section 11).
 * train: both clouds are n x 6 float rows (x y z nx ny nz).  The model is sampled on a 1/step lattice of its bounding
 * box (samplePCByQuantization), every ordered pair of sampled points gives a four-component point-pair feature
 * (three angles quantised by 2 pi / num_angles, the distance by step * diameter) and the pair's planar angle alpha.
 * match: the scene is sampled the same way (relative_scene_distance); every 1/relative_scene_sample_step-th sampled
 * point is a reference point whose pairs with all other sampled points vote for (model reference, alpha bin); the
 * winner gives one pose per reference point, the poses are clustered greedily (position / rotation thresholds) and
 * averaged.  results: clustered poses, most votes first.
 * ONE DELIBERATE DIFFERENCE from OpenCV: a scene pair votes for the model pairs with the SAME quantised feature;
 * OpenCV additionally counts the pairs that merely share a bucket of its MurmurHash table (hash-collision votes,
 * walked without a key comparison) — noise that depends on the hash variant and cannot be restated. */
typedef struct peb_ppf_params {
  double relative_sampling_step;  /* PPF3DDetector(0.03, ., .)                                         */
  double relative_distance_step;  /* PPF3DDetector(., 0.03, .) — stored and never used by OpenCV either */
  double num_angles;              /* PPF3DDetector(., ., 40)                                            */
  double position_threshold;      /* setSearchParams: < 0 -> relative_sampling_step (an ABSOLUTE length, as upstream) */
  double rotation_threshold;      /* setSearchParams: < 0 -> (360 / angle_step) / 180 * pi              */
  int32_t use_weighted_avg;       /* setSearchParams(., ., useWeightedClustering)                       */
  int32_t reserved;
} peb_ppf_params;
/* cv::ppf_match_3d::Pose3D */
typedef struct peb_ppf_pose {
  double pose[16];       /* row-major 4 x 4 (cv::Matx44d::val): model -> scene */
  double q[4];           /* w x y z */
  double t[3];
  double angle;          /* rotation angle of pose (from the trace) */
  double alpha;          /* the winning alpha bin's angle           */
  double residual;       /* filled by the ICP afterwards            */
  uint64_t num_votes;
  uint64_t model_index;  /* the winning model reference point       */
} peb_ppf_pose;
typedef struct peb_ppf_model peb_ppf_model;
PEB_API void peb_ppf_params_default(peb_ppf_params* p); /* (0.03, 0.03, 40), thresholds -1, plain average */
/* trainModel: the trained detector lives on ctx's device and belongs to ctx (destroy it before the context) */
PEB_API int peb_ppf_train(peb_ctx* ctx, const float* model_xyzn, size_t n_model, const peb_ppf_params* params,
                          peb_ppf_model** out);
PEB_API void peb_ppf_model_destroy(peb_ppf_model* m);
/* sampled model points (rows of 6 floats, lattice order); out6 nullable */
PEB_API int peb_ppf_model_sampled(const peb_ppf_model* m, float* out6, size_t cap, size_t* out_n);
/* match: at most cap clustered poses are copied to results, *out_n = how many there are.
 * raw / cap_raw / out_n_raw (nullable): the un-clustered pose of every scene reference point, in reference order. */
PEB_API int peb_ppf_match(peb_ctx* ctx, const peb_ppf_model* m, const float* scene_xyzn, size_t n_scene,
                          double relative_scene_sample_step, double relative_scene_distance, peb_ppf_pose* results,
                          size_t cap, size_t* out_n, peb_ppf_pose* raw, size_t cap_raw, size_t* out_n_raw);

/* ---- pcl::NormalEstimation<PointXYZ,Normal>::compute  [PCL] features/.../impl/normal_3d.hpp */
/* out_normal8: n x 8 floats = pcl::Normal memory image (nx ny nz 0 | curvature 0 0 0). */
PEB_API int peb_normals_knn(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k,
                            const float viewpoint[3], float* out_normal8);
/* same, and also returns the neighbour lists KdTreeFLANN::nearestKSearch(p, k) would:
 * out_nn_idx (nullable) n x k original indices, ascending squared distance, -1 padded */
PEB_API int peb_normals_knn_ex(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k,
                               const float viewpoint[3], float* out_normal8, int32_t* out_nn_idx);

/* ---- cv::ppf_match_3d::computeNormalsPC3d(pc, out, k, flip, viewpoint) ------------------------------------------
 * What the reference runs in the normals slot (pose_estimation/src/opencv_surface_match.cpp:57-59:
 * computeNormalsPC3d(pc_scene, pc_scene_normals, 20, true, (0, 0, 0))).  [CV] opencv_contrib/modules/surface_matching/
 * src/ppf_helpers.cpp (restated from recollection, DESIGN.md section 13); the eigen solver is pinned bit for bit
 * against cv2.eigen of an OpenCV built without Eigen.
 *   neighbours  the k nearest points (the point itself included), ascending squared float distance: the exact
 *               search of KDTreeSingleIndexParams(8); equidistant neighbours may come in another order than FLANN's
 *   covariance  in list order: C(j,l) += (double)(float)(p_j * p_l), mu_j += p_j; then mu *= 1.0 / k, C *= 1.0 / k,
 *               C(j,l) -= mu_j mu_l, all double (meanCovLocalPCInd)
 *   normal      cv::eigen(C) = JacobiImpl_<double> (eigenvalues descending, eigenvectors as rows); row 2 rounded to float
 *   flip        flip_viewpoint != 0: d = viewpoint - p (float), cos = d0 n0 + d1 n1 + d2 n2 (float, left to right);
 *               cos < 0 negates n (flipNormalViewpoint)
 * out_xyzn6: n rows of 6 floats x y z nx ny nz (a CV_32F PCNormals Mat, e.g. pc_scene_normals.ptr<float>(0)); x y z
 * are copied from the input.  out_nn_idx (nullable): n x k original indices, -1 on rows of non-finite points.
 * Where the reference is undefined, this library defines:
 *   - a non-finite point is neither a query nor a neighbour; its row gets its x y z and a NaN normal;
 *   - k < 1, or k greater than the number of finite points (FLANN would leave indices unfilled and OpenCV would read
 *     row -1), is PEB_E_INVALID_ARG; k > 192 is PEB_E_UNSUPPORTED (the bound of peb_normals_knn); n == 0 is PEB_OK
 *     for any valid k and writes nothing. */
PEB_API int peb_cv_normals(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k, int flip_viewpoint,
                           const float viewpoint[3], float* out_xyzn6, int32_t* out_nn_idx);

/* ---- pcl::KdTreeFLANN::nearestKSearch over the resident target (k = 1) ------------ */
/* out_idx: original target index (-1 if the target is empty), out_d2: squared distance. */
PEB_API int peb_nn_search(peb_ctx* ctx, const void* queries, size_t nq, size_t stride,
                          int32_t* out_idx, float* out_d2);
/* the brute-force FP32 validator (shared-memory tiled, no grid): same outputs */
PEB_API int peb_nn_search_bruteforce(peb_ctx* ctx, const void* queries, size_t nq, size_t stride,
                                     int32_t* out_idx, float* out_d2);

/* ---- pcl::Registration::setInputTarget / setInputSource ---------------------------- */
/* normals: nullable; n records of nstride bytes whose first three floats are the normal
 * (pcl::Normal: 32, inside pcl::PointNormal: pass pts+16 and 48).  Builds the search grid;
 * it persists until the next peb_target_set (PCL: target_cloud_updated_). */
PEB_API int peb_target_set(peb_ctx* ctx, const void* pts, size_t n, size_t stride,
                           const void* normals, size_t nstride);
PEB_API int peb_source_set(peb_ctx* ctx, const void* pts, size_t n, size_t stride);
/* The two halves of peb_target_set / peb_source_set, and the replica of another context's cloud — the building
 * blocks of peb_multi_target_set / peb_multi_source_set (one host-to-device copy per box, not per device):
 *   *_stage  uploads the caller's records into the context (asynchronous; nothing is searchable yet),
 *   *_build  builds the search grid over the staged cloud (peb_target_set = stage + build),
 *   *_clone  copies src's STAGED cloud device to device into dst (cudaMemcpyPeerAsync, ordered after src's staging by
 *            an event: NVLink / NVSwitch between peers, through the host otherwise) and builds dst's grid — the build
 *            is deterministic, so the replica is identical to src's.  dst and src may live on the same device.
 * peb_ctx_enable_peer: direct peer access from ctx's device to peer's (PEB_E_UNSUPPORTED if the hardware has none —
 * the clones then still work, staged by the driver). */
PEB_API int peb_target_stage(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const void* normals, size_t nstride);
PEB_API int peb_target_build(peb_ctx* ctx);
PEB_API int peb_target_clone(peb_ctx* dst, peb_ctx* src);
PEB_API int peb_source_stage(peb_ctx* ctx, const void* pts, size_t n, size_t stride);
PEB_API int peb_source_build(peb_ctx* ctx);
PEB_API int peb_source_clone(peb_ctx* dst, peb_ctx* src);
PEB_API int peb_ctx_enable_peer(peb_ctx* ctx, const peb_ctx* peer);

/* ---- pcl::IterativeClosestPoint::align(output, guess) ------------------------------ */
/* guess: column-major 4x4 (NULL = identity).  Optional outputs (nullable):
 *   out_aligned_xyz4  n x 4 floats, final * input  (w = 1)
 *   out_corr_idx      n ints, the target index matched in the LAST iteration, -1 = rejected
 *   out_corr_d2       n floats, its squared distance */
PEB_API int peb_icp_align(peb_ctx* ctx, const float guess[16], const peb_icp_params* params,
                          peb_icp_result* result, float* out_aligned_xyz4,
                          int32_t* out_corr_idx, float* out_corr_d2);

/* one source, one target, H initial poses (guesses: H x 16 floats, column-major each):
 * the shape of cv::ppf_match_3d::ICP::registerModelToScene(model, scene, poses),
 * pose_estimation/src/opencv_surface_match.cpp:94.  results: H records. */
PEB_API int peb_icp_align_batch(peb_ctx* ctx, const float* guesses, size_t n_guesses,
                                const peb_icp_params* params, peb_icp_result* results);

/* ---- correspondence rejectors: pcl::Registration::addCorrespondenceRejector ---------------------------------
 * A chain of rejectors runs in every ICP iteration after the correspondence search, in the order given; each one
 * sees what the one before kept, and the pairs left at the end feed min_correspondences, the estimator, last_mse and
 * n_correspondences (getFitnessScore is not affected).  params->rejector_max_dist > 0 stays a DISTANCE rejector in
 * front of the chain.  [PCL] registration/src/correspondence_rejection_{distance,median_distance,one_to_one,trimmed}.cpp
 * (restated from recollection, DESIGN.md section 12):
 *   DISTANCE         keep iff d2 < value^2 (the limit stored as a float)
 *   MEDIAN_DISTANCE  score = the squared norm of (moved source - target) as a float Vector4f, ((dx dx + dz dz) + dy dy);
 *                    median = the (m / 2)-th smallest score (m pairs in); keep iff score <= median * value (value =
 *                    setMedianFactor, 1.0 in PCL: a factor on SQUARED distances)
 *   ONE_TO_ONE       per target point the pair of smallest d2; a tie goes to the smaller source index (value unused)
 *   TRIMMED          r = value clamped to [0, 1] (setOverlapRatio, 0.5 in PCL), n_keep = max(floor(r * m) in float,
 *                    min_correspondences); the n_keep pairs of smallest (d2, source index), all if n_keep >= m
 * An align with a chain runs every iteration as a search launch, one rejector launch and a moment launch (icp.cu :
 * icp_reject_kernel).  ONE_TO_ONE keeps a table of H x (finite target points) x 8 bytes on the device (4.1 GB for 1024
 * hypotheses and a 500 000-point scene); PEB_E_OOM if it cannot be allocated.  At most PEB_MAX_REJECTORS entries;
 * an unknown kind, a non-finite value, a negative min_correspondences or chain == NULL with n_chain > 0 is
 * PEB_E_INVALID_ARG.  n_chain == 0 is exactly the entry point without _ex. */
enum { PEB_REJECTOR_DISTANCE = 0, PEB_REJECTOR_MEDIAN_DISTANCE = 1, PEB_REJECTOR_ONE_TO_ONE = 2, PEB_REJECTOR_TRIMMED = 3 };
enum { PEB_MAX_REJECTORS = 8 };
typedef struct peb_rejector {
  int32_t kind;                 /* PEB_REJECTOR_*                                                       */
  int32_t min_correspondences;  /* TRIMMED: setMinCorrespondences (0); otherwise 0                      */
  double value;                 /* DISTANCE: max distance (m); MEDIAN: factor; TRIMMED: overlap ratio   */
} peb_rejector;
PEB_API int peb_icp_align_ex(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, const peb_rejector* chain,
                             size_t n_chain, peb_icp_result* result, float* out_aligned_xyz4, int32_t* out_corr_idx,
                             float* out_corr_d2);
PEB_API int peb_icp_align_batch_ex(peb_ctx* ctx, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                   const peb_rejector* chain, size_t n_chain, peb_icp_result* results);

/* pcl::Registration::getFitnessScore(max_range) for an arbitrary transform */
PEB_API int peb_fitness_score(peb_ctx* ctx, const float T[16], double max_range, double* out_fitness,
                              int32_t* out_n_inliers);

/* ---- several devices behind one handle (SURVEY.md 8e) -------------------------------- */
/* The reference node is one process (a component container with a single-threaded executor,
 * pose_estimation/launch/pose_estimation.launch.py:17-35), so the drop-in for the refinement slot
 * (pose_estimation/src/opencv_surface_match.cpp:85-94) that uses every GPU of the box lives behind
 * one handle: one context per device, a replica of the scene grid and of the model on each, the H
 * initial poses split into contiguous blocks (device i refines [lo, hi) of peb_multi_shard_range).
 * Hypotheses are independent: no collective; each device copies its records into `results`.
 * devices: ndev CUDA device indices (NULL = 0 .. ndev-1).  An index may repeat — the contexts are
 * independent, which is how the single-GPU tests exercise the sharding.  Calls on one peb_multi
 * must be serialised by the caller, like calls on one peb_ctx.  One persistent host thread per extra
 * device is parked between calls.  The scene and the model are uploaded once (device 0) and replicated
 * device to device (peb_target_clone).
 * Results: every hypothesis is refined exactly as by peb_icp_align_batch on one device given the same
 * block of hypotheses (byte-identical records; it is also what one rank of the one-process-per-GPU path
 * computes).  Against ONE context refining all H hypotheses the records can differ in the last bits of the
 * double moment sums: the number of blocks per hypothesis (hence the order in which the per-block partial
 * sums are added) is chosen from the batch size. */
typedef struct peb_multi peb_multi;
PEB_API int peb_multi_create(int ndev, const int* devices, peb_multi** out);
PEB_API void peb_multi_destroy(peb_multi* m);
/* message of the last failing call on m (m == NULL: of the last failing peb_multi_create of this thread) */
PEB_API const char* peb_multi_last_error(const peb_multi* m);
PEB_API int peb_multi_size(const peb_multi* m);
/* context i (borrowed; for per-device introspection, not for concurrent use) */
PEB_API peb_ctx* peb_multi_ctx(peb_multi* m, int i);
/* peb_ctx_set_int on every context */
PEB_API int peb_multi_set_int(peb_multi* m, const char* key, int value);
/* [lo, hi) of the n_items hypotheses device i of ndev refines: blocks of ceil(n_items / ndev) */
PEB_API void peb_multi_shard_range(size_t n_items, int ndev, int i, size_t* lo, size_t* hi);
/* peb_target_set / peb_source_set for every device: staged once on device 0, cloned to the others, built everywhere */
PEB_API int peb_multi_target_set(peb_multi* m, const void* pts, size_t n, size_t stride,
                                 const void* normals, size_t nstride);
PEB_API int peb_multi_source_set(peb_multi* m, const void* pts, size_t n, size_t stride);
/* peb_icp_align_batch, sharded: guesses H x 16 floats, results H records, hypothesis order */
PEB_API int peb_multi_icp_align_batch(peb_multi* m, const float* guesses, size_t n_guesses,
                                      const peb_icp_params* params, peb_icp_result* results);
/* peb_icp_align_batch_ex, sharded the same way */
PEB_API int peb_multi_icp_align_batch_ex(peb_multi* m, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                         const peb_rejector* chain, size_t n_chain, peb_icp_result* results);
/* kernel launches of all contexts so far */
PEB_API uint64_t peb_multi_launch_count(const peb_multi* m);

/* ---- device-resident variants (bench harness: inputs already in HBM) ---------------- */
/* d_*: device pointers on the context's device, float4 records (xyz + pad), 16-byte aligned.
 * Asynchronous on peb_ctx_stream(); *_dev results are device pointers too. */
PEB_API int peb_target_set_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const void* d_normal4);
PEB_API int peb_source_set_dev(peb_ctx* ctx, const void* d_xyz4, size_t n);
PEB_API int peb_icp_align_dev(peb_ctx* ctx, const float guess[16], const peb_icp_params* params,
                              peb_icp_result* d_result);
PEB_API int peb_icp_align_batch_dev(peb_ctx* ctx, const float* d_guesses, size_t n_guesses,
                                    const peb_icp_params* params, peb_icp_result* d_results);
PEB_API int peb_voxel_grid_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, float leaf_x, float leaf_y,
                               float leaf_z, unsigned min_pts, void* d_out_xyz4, size_t* out_n);
PEB_API int peb_normals_knn_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, int k,
                                const float viewpoint[3], void* d_out_normal8);
/* peb_cv_normals on the device: d_out_xyzn6 holds n x 6 floats (4-byte alignment suffices) */
PEB_API int peb_cv_normals_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, int k, int flip_viewpoint,
                               const float viewpoint[3], void* d_out_xyzn6);
/* waits for everything queued on the context.  PEB_E_CUDA if the last batched align raised its internal-error flag
 * (PEB_STATE_INTERNAL_ERROR): the asynchronous peb_icp_align_batch_dev cannot report it when it returns, and a
 * record written before another hypothesis hit the bound does not carry it. */
PEB_API int peb_sync(peb_ctx* ctx);

/* ---- introspection used by the parity tests ---------------------------------------- */
typedef struct peb_grid_info {
  float origin[3];
  float cell;          /* cell edge length                      */
  int32_t dims[3];
  int32_t n_points;    /* finite target points in the grid      */
  int64_t n_cells;
} peb_grid_info;
PEB_API int peb_target_grid_info(peb_ctx* ctx, peb_grid_info* out);
/* with peb_ctx_set_int(ctx, "profile", 2): device time (ms, CUDA events on the context's stream)
 * of every ICP kernel launch of the last align — the iteration launches, then the fitness launch.
 * With "profile" = 1: ONE value, the span from the first to the end of the last ITERATION launch (no events
 * between the iteration launches, so their overlap is not disturbed; the fitness launch is outside the span;
 * a batch that runs as several chains of launches reports its slowest chain). */
PEB_API int peb_profile_read(peb_ctx* ctx, float* out_ms, size_t cap, size_t* out_n);
/* per-iteration increments of the last peb_icp_align (column-major 4x4 each);
 * copies min(cap, iterations) matrices, returns the count via *out_n */
PEB_API int peb_icp_trace(peb_ctx* ctx, float* out_T, size_t cap, size_t* out_n);

#ifdef __cplusplus
}
#endif
#endif /* PE_B200_H_ */
