"""Host-side mirror of the PCL 1.10 classes the north-star path substitutes into the reference's
slots (SURVEY.md 8b): same method names, defaults and error behaviour as

    pcl::VoxelGrid<PointXYZ>                 down-sample slot  pose_estimation/src/pose_estimation.cpp:261-263
    pcl::NormalEstimation<PointXYZ, Normal>  normals slot      pose_estimation/src/opencv_surface_match.cpp:57-59
    pcl::IterativeClosestPoint(+WithNormals) refinement slot   pose_estimation/src/opencv_surface_match.cpp:85-94

Every method is a thin call into libpe_b200.so through its C ABI (include/pe_b200.h); this file
holds no arithmetic.  Clouds are numpy float32 arrays of shape (N, >=3); rows are the records,
so (N,3) cv::Mat-style, (N,4) pcl::PointXYZ-style and (N,12) pcl::PointNormal-style all work.
The C++ facade with the same surface is include/pe_b200/pcl_facade.hpp.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (CvIcpParams, IcpParams, IcpResult, GridInfo, PpfParams, PpfPose, PrefilterParams, SacParams, SurfaceMatchParams,
                   SurfaceMatchResult, lib)

DBL_MAX = float(np.finfo(np.float64).max)


class PebError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{_lib.STATUS_NAMES.get(code, code)}: {msg}")
        self.code = code


def _cloud(a) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3 or (a.shape[0] > 1 and a.strides[1] != 4):
        a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("point cloud must have shape (N, >=3)")
    return a


def _stride(a: np.ndarray) -> int:
    return int(a.strides[0]) if a.shape[0] > 1 else max(int(a.strides[0]), 12)


def _col_major(T) -> np.ndarray:
    """4x4 row-indexed numpy matrix -> the 16 floats of Eigen::Matrix4f::data()."""
    return np.ascontiguousarray(np.asarray(T, dtype=np.float32).reshape(4, 4).T).reshape(16)


def result_matrix(r: IcpResult) -> np.ndarray:
    return np.array(r.T, dtype=np.float32).reshape(4, 4).T.copy()


class Context:
    """peb_ctx: one CUDA device + stream.  Calls on one context must be serialised."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        rc = lib.peb_ctx_create(device, C.byref(h))
        if rc != 0:
            raise PebError(rc, lib.peb_last_error(None).decode())
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib.peb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check(self, rc: int):
        if rc != 0:
            raise PebError(rc, lib.peb_last_error(self._h).decode())

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return int(lib.peb_ctx_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(lib.peb_ctx_launch_count(self._h))

    def set_int(self, key: str, value: int):
        self.check(lib.peb_ctx_set_int(self._h, key.encode(), int(value)))

    def sync(self):
        self.check(lib.peb_sync(self._h))

    # ---- free functions of the ABI ---------------------------------------------------------
    def nn_search(self, queries, bruteforce: bool = False):
        q = _cloud(queries)
        idx = np.empty(q.shape[0], np.int32)
        d2 = np.empty(q.shape[0], np.float32)
        fn = lib.peb_nn_search_bruteforce if bruteforce else lib.peb_nn_search
        self.check(fn(self._h, q.ctypes.data, q.shape[0], _stride(q), idx.ctypes.data, d2.ctypes.data))
        return idx, d2

    def target_set(self, pts, normals=None):
        t = _cloud(pts)
        self._keep_t = t
        if normals is not None:
            nr = _cloud(normals)
            self.check(lib.peb_target_set(self._h, t.ctypes.data, t.shape[0], _stride(t), nr.ctypes.data, _stride(nr)))
        else:
            self.check(lib.peb_target_set(self._h, t.ctypes.data, t.shape[0], _stride(t), None, 0))

    def source_set(self, pts):
        s = _cloud(pts)
        self.check(lib.peb_source_set(self._h, s.ctypes.data, s.shape[0], _stride(s)))
        self._n_src = s.shape[0]

    def grid_info(self) -> GridInfo:
        gi = GridInfo()
        self.check(lib.peb_target_grid_info(self._h, C.byref(gi)))
        return gi

    def fitness_score(self, T, max_range: float = DBL_MAX):
        t = _col_major(T)
        f = C.c_double()
        n = C.c_int32()
        self.check(lib.peb_fitness_score(self._h, t.ctypes.data, max_range, C.byref(f), C.byref(n)))
        return f.value, n.value


_default_ctx: Context | None = None


class MultiContext:
    """peb_multi: several devices behind one handle (include/pe_b200.h, SURVEY.md 8e) — what the reference's single
    process binds to refine the poses of registerModelToScene(model, scene, poses) on every GPU of the box.  One context
    per device, the scene grid and the model replicated, the hypotheses of alignBatch split into contiguous blocks.
    Pass it as `ctx` to IterativeClosestPoint(+WithNormals); a single align() is not sharded (replicas only) and runs
    on the first device.  A device index may repeat (independent contexts on one GPU)."""

    is_multi = True

    def __init__(self, devices):
        devs = list(range(devices)) if isinstance(devices, int) else [int(d) for d in devices]
        arr = (C.c_int * max(len(devs), 1))(*devs)
        h = C.c_void_p()
        rc = lib.peb_multi_create(len(devs), arr, C.byref(h))
        if rc != 0:
            raise PebError(rc, lib.peb_multi_last_error(None).decode())
        self._h = h
        self.devices = devs

    def close(self):
        if getattr(self, "_h", None):
            lib.peb_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check(self, rc: int):
        if rc != 0:
            raise PebError(rc, lib.peb_multi_last_error(self._h).decode())

    @property
    def handle(self):
        return self._h

    @property
    def size(self) -> int:
        return int(lib.peb_multi_size(self._h))

    @property
    def launch_count(self) -> int:
        return int(lib.peb_multi_launch_count(self._h))

    def first(self) -> "Context":
        """Context 0, borrowed (closing it is a no-op): where the unsharded calls run."""
        c = Context.__new__(Context)
        c._h = C.c_void_p(lib.peb_multi_ctx(self._h, 0))
        c.close = lambda: None
        return c

    def shard_range(self, n_items: int, i: int) -> tuple[int, int]:
        lo, hi = C.c_size_t(0), C.c_size_t(0)
        lib.peb_multi_shard_range(n_items, self.size, i, C.byref(lo), C.byref(hi))
        return lo.value, hi.value

    def set_int(self, key: str, value: int):
        self.check(lib.peb_multi_set_int(self._h, key.encode(), int(value)))

    def target_set(self, pts, normals=None):
        p = _cloud(pts)
        if normals is None:
            self.check(lib.peb_multi_target_set(self._h, p.ctypes.data, p.shape[0], _stride(p), None, 0))
        else:
            nm = _cloud(normals)
            if nm.shape[0] != p.shape[0]:
                raise ValueError("target normals must have one row per target point")
            self.check(lib.peb_multi_target_set(self._h, p.ctypes.data, p.shape[0], _stride(p), nm.ctypes.data, _stride(nm)))

    def source_set(self, pts):
        p = _cloud(pts)
        self.check(lib.peb_multi_source_set(self._h, p.ctypes.data, p.shape[0], _stride(p)))

    def icp_align_batch(self, g16: np.ndarray, params: IcpParams, res, chain=()):
        """chain: correspondence rejectors (_lib.rejector_array), applied in order after rejector_max_dist."""
        if chain:
            arr, n = _lib.rejector_array(chain)
            self.check(lib.peb_multi_icp_align_batch_ex(self._h, g16.ctypes.data, g16.shape[0], C.byref(params), arr, n, res))
        else:
            self.check(lib.peb_multi_icp_align_batch(self._h, g16.ctypes.data, g16.shape[0], C.byref(params), res))


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class ScenePrefilter:
    """The deterministic part of PoseEstimation::create_surface_match_pc
    (pose_estimation/src/pose_estimation.cpp:246-261): NaN removal, the optional sphere filter around the
    last pose (filter_points, :347-372) and the 5 mm band removal of remove_planes (:309-333) for plane
    coefficients the caller supplies (SACSegmentation below computes them)."""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self._input = None
        self.params = PrefilterParams()
        self.params.plane_band = 0.005

    def setInputCloud(self, cloud):
        self._input = _cloud(cloud)

    def setSphereFilter(self, center, radius: float, filter_out: str = "outliers"):
        """filter_out == "inliers" removes the points inside the sphere, anything else keeps only them
        (EstimatePose.srv: filter_out / filter_radius)."""
        self.params.use_sphere = 1 if radius > 0 else 0
        self.params.remove_inliers = 1 if filter_out == "inliers" else 0
        self.params.sphere_center[:] = [float(v) for v in center[:3]]
        self.params.sphere_radius = float(radius)

    def addPlane(self, a: float, b: float, c: float, d: float):
        k = self.params.n_planes
        if k >= 8:
            raise PebError(-1, "ScenePrefilter: at most 8 planes")
        for j, v in enumerate((a, b, c, d)):
            self.params.planes[4 * k + j] = float(v)
        self.params.n_planes = k + 1

    def setPlaneBand(self, band: float):
        self.params.plane_band = float(band)

    def filter(self) -> np.ndarray:
        if self._input is None:
            raise ValueError("ScenePrefilter.filter: no input cloud (setInputCloud)")
        p = self._input
        out = np.empty((max(p.shape[0], 1), 4), np.float32)
        m = C.c_size_t(0)
        self.ctx.check(lib.peb_scene_prefilter(self.ctx.handle, p.ctypes.data, p.shape[0], _stride(p), C.byref(self.params),
                                               out.ctypes.data, C.byref(m)))
        return out[: m.value].copy()


def _surface_match_pc_params(filter_pose, filter_radius, filter_out, plane_band=0.005, distance_threshold=0.0001,
                             max_iterations=100):
    """The filter and RANSAC settings of create_surface_match_pc -> (PrefilterParams, SacParams)."""
    f = PrefilterParams()
    f.plane_band = float(plane_band)
    if filter_pose is not None and filter_radius > 0:
        f.use_sphere = 1
        f.remove_inliers = 1 if filter_out == "inliers" else 0
        f.sphere_center[:] = [float(v) for v in filter_pose[:3]]
        f.sphere_radius = float(filter_radius)
    sp = SacParams()
    lib.peb_sac_params_default(C.byref(sp))
    sp.distance_threshold = float(distance_threshold)
    sp.max_iterations = int(max_iterations)
    return f, sp


def create_surface_match_pc(cloud, ctx: Context | None = None, filter_pose=None, filter_radius: float = 0.0,
                            filter_out: str = "outliers", num_planes: int = 0, leaf: float = 0.0, plane_band: float = 0.005,
                            distance_threshold: float = 0.0001, max_iterations: int = 100):
    """PoseEstimation::create_surface_match_pc (pose_estimation/src/pose_estimation.cpp:211-279) from the organized cloud
    on: NaN removal, the optional sphere filter around the last pose, num_planes rounds of plane RANSAC + 5 mm band
    removal (remove_planes, :281-345, with the reference's RANSAC settings as defaults) and — leaf > 0 — the VoxelGrid,
    in ONE library call (peb_scene_prepare).  -> (points (M, 4) float32, plane coefficients (num_planes, 4))."""
    ctx = ctx or default_context()
    p = _cloud(cloud)
    f, sp = _surface_match_pc_params(filter_pose, filter_radius, filter_out, plane_band, distance_threshold, max_iterations)
    out = np.empty((max(p.shape[0], 1), 4), np.float32)
    planes = np.zeros((max(num_planes, 1), 4), np.float32)
    m = C.c_size_t(0)
    ctx.check(lib.peb_scene_prepare(ctx.handle, p.ctypes.data, p.shape[0], _stride(p), C.byref(f), int(num_planes), C.byref(sp),
                                    float(leaf), out.ctypes.data, C.byref(m), planes.ctypes.data))
    return out[: m.value].copy(), planes[:num_planes].copy()


class SACSegmentation:
    """pcl::SACSegmentation<pcl::PointXYZ> for SACMODEL_PLANE + SAC_RANSAC
    ([PCL] segmentation/include/pcl/segmentation/sac_segmentation.h), the plane fit of the reference's
    remove_planes (pose_estimation/src/pose_estimation.cpp:285-297).  Other model / method types have no
    CUDA implementation and raise PEB_E_UNSUPPORTED."""

    SACMODEL_PLANE = 0  # pcl::SacModel
    SAC_RANSAC = 0      # pcl::SAC_RANSAC

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self._input = None
        self.params = SacParams()
        lib.peb_sac_params_default(C.byref(self.params))
        self._model = None
        self._method = None
        self.iterations_ = 0

    def setInputCloud(self, cloud):
        self._input = _cloud(cloud)

    def setModelType(self, model: int):
        if model != self.SACMODEL_PLANE:
            raise PebError(-6, f"SACSegmentation: model type {model} has no CUDA implementation (SACMODEL_PLANE only)")
        self._model = model

    def setMethodType(self, method: int):
        if method != self.SAC_RANSAC:
            raise PebError(-6, f"SACSegmentation: method type {method} has no CUDA implementation (SAC_RANSAC only)")
        self._method = method

    def setOptimizeCoefficients(self, on: bool):
        self.params.optimize_coefficients = 1 if on else 0

    def setDistanceThreshold(self, t: float):
        self.params.distance_threshold = float(t)

    def setMaxIterations(self, n: int):
        self.params.max_iterations = int(n)

    def setProbability(self, p: float):
        self.params.probability = float(p)

    def segment(self):
        """-> (inlier indices int32 ascending, coefficients float32[4]); both empty when no model was found
        (pcl: inliers.indices.clear(), model_coefficients.values.clear())."""
        if self._input is None:
            raise ValueError("SACSegmentation.segment: no input cloud (setInputCloud)")
        if self._model is None:
            raise PebError(-1, "SACSegmentation.segment: no model type given (setModelType)")  # PCL: initSACModel fails
        p = self._input
        coeff = np.zeros(4, np.float32)
        inl = np.empty(max(p.shape[0], 1), np.int32)
        m = C.c_size_t(0)
        it = C.c_int32(0)
        self.ctx.check(lib.peb_sac_plane(self.ctx.handle, p.ctypes.data, p.shape[0], _stride(p), C.byref(self.params),
                                         coeff.ctypes.data, inl.ctypes.data, C.byref(m), C.byref(it)))
        self.iterations_ = it.value
        if m.value == 0 and not coeff.any():
            return np.empty(0, np.int32), np.empty(0, np.float32)
        return inl[: m.value].copy(), coeff


class CvIcp:
    """cv::ppf_match_3d::ICP (opencv_contrib surface_matching) as the reference constructs and calls it
    (pose_estimation/src/opencv_surface_match.cpp:85-94): ICP(iterations, tolerance, rejectionScale, numLevels) and
    registerModelToScene(model, scene, poses) with N x 6 float clouds (points + normals)."""

    def __init__(self, iterations: int = 250, tolerance: float = 0.05, rejection_scale: float = 2.5, num_levels: int = 6,
                 ctx: Context | None = None):
        # (defaults of cv::ppf_match_3d::ICP::ICP(); the reference passes 250, 0.005f, 2.5f, 8)
        self.ctx = ctx or default_context()
        self.params = CvIcpParams(int(iterations), int(num_levels), float(tolerance), float(rejection_scale))

    def registerModelToScene(self, model6, scene6, poses):
        """poses: (H, 4, 4) float64 -> (refined poses (H, 4, 4), residuals (H,)); the Pose3D list of OpenCV updated by
        appendPose, residual per pose."""
        m = np.ascontiguousarray(model6, np.float32)
        sc = np.ascontiguousarray(scene6, np.float32)
        if m.ndim != 2 or m.shape[1] != 6 or sc.ndim != 2 or sc.shape[1] != 6:
            raise PebError(-1, "CvIcp.registerModelToScene: model and scene must be N x 6 float (points + normals)")
        P = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 16)).copy()
        res = np.zeros(max(P.shape[0], 1), np.float64)
        self.ctx.check(lib.peb_cvicp_register(self.ctx.handle, m.ctypes.data, m.shape[0], sc.ctypes.data, sc.shape[0],
                                              C.byref(self.params), P.ctypes.data, P.shape[0], res.ctypes.data))
        return P.reshape(-1, 4, 4), res[: P.shape[0]]


class PPF3DDetector:
    """cv::ppf_match_3d::PPF3DDetector as the reference constructs and calls it
    (pose_estimation/src/opencv_surface_match.cpp:45-46: PPF3DDetector(0.03, 0.03, 40).trainModel(model); :65:
    match(scene_with_normals, results, 1.0, 0.03)).  Clouds are N x 6 float (points + normals); match returns the
    clustered poses (PpfPose = Pose3D: pose, q, t, angle, numVotes, modelIndex), most votes first."""

    def __init__(self, relativeSamplingStep: float = 0.05, relativeDistanceStep: float = 0.05, numAngles: float = 30,
                 ctx: Context | None = None):
        # (defaults of cv::ppf_match_3d::PPF3DDetector; the reference passes 0.03, 0.03, 40)
        self.ctx = ctx or default_context()
        self.params = PpfParams()
        lib.peb_ppf_params_default(C.byref(self.params))
        self.params.relative_sampling_step = float(relativeSamplingStep)
        self.params.relative_distance_step = float(relativeDistanceStep)
        self.params.num_angles = float(numAngles)
        self._model = C.c_void_p()

    def setSearchParams(self, positionThreshold: float = -1.0, rotationThreshold: float = -1.0, useWeightedClustering: bool = False):
        self.params.position_threshold = float(positionThreshold)
        self.params.rotation_threshold = float(rotationThreshold)
        self.params.use_weighted_avg = int(bool(useWeightedClustering))

    def trainModel(self, model6):
        m = np.ascontiguousarray(model6, np.float32)
        if m.ndim != 2 or m.shape[1] != 6:
            raise PebError(-1, "PPF3DDetector.trainModel: the model must be N x 6 float (points + normals)")
        self.close()
        self.ctx.check(lib.peb_ppf_train(self.ctx.handle, m.ctypes.data, m.shape[0], C.byref(self.params), C.byref(self._model)))

    def sampled_model(self) -> np.ndarray:
        n = C.c_size_t(0)
        self.ctx.check(lib.peb_ppf_model_sampled(self._model, None, 0, C.byref(n)))
        out = np.empty((n.value, 6), np.float32)
        self.ctx.check(lib.peb_ppf_model_sampled(self._model, out.ctypes.data, n.value, C.byref(n)))
        return out

    def match(self, scene6, relativeSceneSampleStep: float = 1.0 / 5.0, relativeSceneDistance: float = 0.03, return_raw: bool = False):
        if not self._model:
            raise PebError(-1, "PPF3DDetector.match: the model is not trained")
        sc = np.ascontiguousarray(scene6, np.float32)
        if sc.ndim != 2 or sc.shape[1] != 6:
            raise PebError(-1, "PPF3DDetector.match: the scene must be N x 6 float (points + normals)")
        # one pose per reference point at most, one reference point per occupied lattice cell at most (the buffers are kept)
        cap = max(1, min(sc.shape[0], (int(1.0 / np.float32(relativeSceneDistance)) + 1) ** 3))
        if getattr(self, "_cap", 0) < cap:
            self._res, self._raw, self._cap = (PpfPose * cap)(), (PpfPose * cap)(), cap
        n = C.c_size_t(0)
        n_raw = C.c_size_t(0)
        self.ctx.check(lib.peb_ppf_match(self.ctx.handle, self._model, sc.ctypes.data, sc.shape[0], float(relativeSceneSampleStep),
                                         float(relativeSceneDistance), self._res, self._cap, C.byref(n),
                                         self._raw if return_raw else None, self._cap if return_raw else 0, C.byref(n_raw)))
        out = [PpfPose.from_buffer_copy(p) for p in self._res[: n.value]]
        return (out, [PpfPose.from_buffer_copy(p) for p in self._raw[: n_raw.value]]) if return_raw else out

    def close(self):
        if self._model:
            lib.peb_ppf_model_destroy(self._model)
            self._model = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def surface_match_params(**overrides) -> SurfaceMatchParams:
    """peb_surface_match_params with the reference's values (peb_surface_match_params_default: k = 20 normals flipped
    towards (0, 0, 0), match(.., 1.0, 0.03), the first 6 results refined by ICP(250, 0.005f, 2.5f, 8), corrected pose7
    layout); keyword arguments override fields (icp=(iterations, tolerance, rejection_scale, num_levels))."""
    p = SurfaceMatchParams()
    lib.peb_surface_match_params_default(C.byref(p))
    for k, v in overrides.items():
        if k == "icp":
            it, tol, rej, lev = v
            p.icp = CvIcpParams(int(it), int(lev), float(tol), float(rej))
        elif k == "viewpoint":
            p.viewpoint[:] = [float(x) for x in v]
        else:
            setattr(p, k, type(getattr(p, k))(v))
    return p


def find_object_in_scene(detector: "PPF3DDetector", cloud, params: SurfaceMatchParams | None = None, prepare: bool = False,
                         filter_pose=None, filter_radius: float = 0.0, filter_out: str = "outliers", num_planes: int = 0,
                         leaf: float = 0.0, return_scene: bool = False):
    """OpenCVSurfaceMatch::find_object_in_scene (pose_estimation/src/opencv_surface_match.cpp:57-142) in ONE library call
    (peb_surface_match) on the detector's context: computeNormalsPC3d, detector.match, cv ICP of the first
    params.max_icp_poses results against the rows the detector was trained on, the selection rule and the packing.
    cloud: the (N, >=3) float cloud the function receives; prepare=True runs create_surface_match_pc's preparation in front
    of it (NaN removal, sphere filter, num_planes plane removals, leaf > 0: VoxelGrid) with its arguments.
    -> (refined PpfPose list, best (-1: nothing found), pose7 float32[7], n_results) [+ scene (M, 6) float32 with
    return_scene]; the same bytes as the step-by-step calls."""
    ctx = detector.ctx
    p = _cloud(cloud)
    params = params if params is not None else surface_match_params()
    f = sp = None
    if prepare:
        f, sp = _surface_match_pc_params(filter_pose, filter_radius, filter_out)
    refined = (PpfPose * max(int(params.max_icp_poses), 1))()
    res = SurfaceMatchResult()
    scene = np.empty((max(p.shape[0], 1), 6), np.float32) if return_scene else None
    m = C.c_size_t(0)
    ctx.check(lib.peb_surface_match(ctx.handle, detector._model, p.ctypes.data, p.shape[0], _stride(p),
                                    C.byref(f) if f is not None else None, int(num_planes), C.byref(sp) if sp is not None else None,
                                    float(leaf), C.byref(params), refined, C.byref(res),
                                    scene.ctypes.data if scene is not None else None, C.byref(m)))
    out = ([PpfPose.from_buffer_copy(r) for r in refined[: res.n_refined]], int(res.best), np.array(res.pose7, np.float32),
           int(res.n_results))
    return out + (scene[: m.value].copy(),) if return_scene else out


class VoxelGrid:
    """pcl::VoxelGrid<pcl::PointXYZ> ([PCL] filters/include/pcl/filters/voxel_grid.h)."""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self._input = None
        self._leaf = (0.0, 0.0, 0.0)
        self._min_pts = 0

    def setInputCloud(self, cloud):
        self._input = _cloud(cloud)

    def setLeafSize(self, lx: float, ly: float | None = None, lz: float | None = None):
        self._leaf = (float(lx), float(lx if ly is None else ly), float(lx if lz is None else lz))

    def getLeafSize(self):
        return self._leaf

    def setMinimumPointsNumberPerVoxel(self, n: int):
        self._min_pts = int(n)

    def getMinimumPointsNumberPerVoxel(self) -> int:
        return self._min_pts

    def filter(self) -> np.ndarray:
        """Returns the (M, 4) down-sampled cloud (x, y, z, 1), ascending voxel index like PCL."""
        if self._input is None:
            raise ValueError("VoxelGrid.filter: no input cloud (setInputCloud)")
        p = self._input
        out = np.empty((max(p.shape[0], 1), 4), np.float32)
        m = C.c_size_t(0)
        self.ctx.check(lib.peb_voxel_grid(self.ctx.handle, p.ctypes.data, p.shape[0], _stride(p), self._leaf[0],
                                          self._leaf[1], self._leaf[2], self._min_pts, out.ctypes.data, C.byref(m)))
        return out[: m.value].copy()


class NormalEstimation:
    """pcl::NormalEstimation<pcl::PointXYZ, pcl::Normal> with setKSearch ([PCL] features/normal_3d.h)."""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self._input = None
        self._k = 0
        self._vp = np.zeros(3, np.float32)

    def setInputCloud(self, cloud):
        self._input = _cloud(cloud)

    def setKSearch(self, k: int):
        self._k = int(k)

    def getKSearch(self) -> int:
        return self._k

    def setRadiusSearch(self, radius: float):
        if radius != 0:
            raise PebError(-6, "NormalEstimation.setRadiusSearch: radius search has no CUDA path (no CPU fallback)")

    def setViewPoint(self, x: float, y: float, z: float):
        self._vp = np.array([x, y, z], np.float32)

    def getViewPoint(self):
        return tuple(float(v) for v in self._vp)

    def compute(self, return_neighbours: bool = False):
        """(N, 8) float32 rows = pcl::Normal (nx ny nz 0 | curvature 0 0 0)."""
        if self._input is None:
            raise ValueError("NormalEstimation.compute: no input cloud (setInputCloud)")
        if self._k <= 0:
            raise ValueError("NormalEstimation.compute: setKSearch(k) first")
        p = self._input
        out = np.empty((p.shape[0], 8), np.float32)
        nn = np.empty((p.shape[0], self._k), np.int32) if return_neighbours else None
        self.ctx.check(lib.peb_normals_knn_ex(self.ctx.handle, p.ctypes.data, p.shape[0], _stride(p), self._k,
                                              self._vp.ctypes.data, out.ctypes.data,
                                              nn.ctypes.data if nn is not None else None))
        return (out, nn) if return_neighbours else out


def compute_normals_pc3d(pc, num_neighbors: int = 20, flip_viewpoint: bool = True, viewpoint=(0.0, 0.0, 0.0),
                         ctx: Context | None = None, return_neighbours: bool = False):
    """cv::ppf_match_3d::computeNormalsPC3d(pc, out, num_neighbors, flip_viewpoint, viewpoint), the reference's normals
    slot (pose_estimation/src/opencv_surface_match.cpp:57-59), with OpenCV's arithmetic (peb_cv_normals, DESIGN.md §13).
    pc: (N, >=3) float32 -> (N, 6) float32 rows x y z nx ny nz; with return_neighbours also the (N, k) int32 lists."""
    ctx = ctx or default_context()
    p = _cloud(pc)
    k = int(num_neighbors)
    vp = np.ascontiguousarray(np.asarray(viewpoint, np.float32).reshape(3))
    out = np.empty((p.shape[0], 6), np.float32)
    nn = np.empty((p.shape[0], max(k, 0)), np.int32) if return_neighbours else None
    ctx.check(lib.peb_cv_normals(ctx.handle, p.ctypes.data, p.shape[0], _stride(p), k, int(bool(flip_viewpoint)),
                                 vp.ctypes.data, out.ctypes.data, nn.ctypes.data if nn is not None else None))
    return (out, nn) if return_neighbours else out


class ConvergenceCriteria:
    """The part of pcl::registration::DefaultConvergenceCriteria<float> reachable through
    IterativeClosestPoint::getConvergeCriteria()."""

    def __init__(self, params: IcpParams):
        self._p = params
        self._state = _lib.CONVERGENCE_CRITERIA_NOT_CONVERGED

    def setAbsoluteMSE(self, v: float):
        self._p.abs_mse_threshold = float(v)

    def getAbsoluteMSE(self) -> float:
        return self._p.abs_mse_threshold

    def setMaximumIterationsSimilarTransforms(self, n: int):
        self._p.max_iterations_similar = int(n)

    def getConvergenceState(self) -> int:
        return self._state


class IterativeClosestPoint:
    """pcl::IterativeClosestPoint<PointXYZ, PointXYZ> ([PCL] registration/icp.h, registration.h)."""

    _estimator = _lib.ESTIMATOR_SVD

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.params = IcpParams()
        lib.peb_icp_params_default(C.byref(self.params))
        self.params.estimator = self._estimator
        self._criteria = ConvergenceCriteria(self.params)
        self._result: IcpResult | None = None
        self._have_source = False
        self._have_target = False
        self._n_src = 0
        self.correspondences = None
        self._chain: list[tuple] = []  # rejectors added after the first non-distance one, in PCL's order

    @property
    def _sctx(self) -> Context:
        """The context of the unsharded calls (align, fitness, trace): with a MultiContext, its first device."""
        if getattr(self.ctx, "is_multi", False):
            if getattr(self, "_first", None) is None:
                self._first = self.ctx.first()
            return self._first
        return self.ctx

    # -- pcl::Registration setters ------------------------------------------------------------
    def setInputSource(self, cloud):
        self.ctx.source_set(cloud)
        self._n_src = _cloud(cloud).shape[0]
        self._have_source = True

    def setInputTarget(self, cloud, normals=None):
        """normals: (N, >=3) target normals (needed by IterativeClosestPointWithNormals); a
        pcl::PointNormal-style (N, 12) cloud carries them in columns 4..6."""
        c = _cloud(cloud)
        if normals is None and c.shape[1] >= 7 and self._estimator == _lib.ESTIMATOR_POINT_TO_PLANE_LLS:
            normals = c[:, 4:7]
        self.ctx.target_set(c, normals)
        self._have_target = True

    def setMaximumIterations(self, n: int):
        self.params.max_iterations = int(n)

    def getMaximumIterations(self) -> int:
        return self.params.max_iterations

    def setMaxCorrespondenceDistance(self, d: float):
        self.params.max_corr_dist = float(d)

    def getMaxCorrespondenceDistance(self) -> float:
        return self.params.max_corr_dist

    def setTransformationEpsilon(self, e: float):
        self.params.transformation_epsilon = float(e)

    def setTransformationRotationEpsilon(self, e: float):
        self.params.rotation_epsilon = float(e)

    def setEuclideanFitnessEpsilon(self, e: float):
        self.params.euclidean_fitness_epsilon = float(e)

    def setUseReciprocalCorrespondences(self, on: bool):
        if on:
            raise PebError(-6, "reciprocal correspondences have no CUDA path (no CPU fallback)")

    def setRANSACIterations(self, n: int):
        if n:
            raise PebError(-6, "the RANSAC rejector has no CUDA path (no CPU fallback)")

    def addCorrespondenceRejectorDistance(self, max_distance: float):
        """addCorrespondenceRejector(CorrespondenceRejectorDistance with setMaximumDistance(d)).  Before any other
        rejector it sets params.rejector_max_dist (the head of the chain); after one, it joins the chain in order."""
        if self._chain:
            self._add_rejector((_lib.REJECTOR_DISTANCE, float(max_distance)))
        else:
            self.params.rejector_max_dist = float(max_distance)

    def addCorrespondenceRejectorMedianDistance(self, factor: float = 1.0):
        """addCorrespondenceRejector(CorrespondenceRejectorMedianDistance with setMedianFactor(factor)): keeps the
        pairs whose squared distance is at most factor x the median squared distance."""
        self._add_rejector((_lib.REJECTOR_MEDIAN_DISTANCE, float(factor)))

    def addCorrespondenceRejectorOneToOne(self):
        """addCorrespondenceRejector(CorrespondenceRejectorOneToOne): the closest source per target point."""
        self._add_rejector((_lib.REJECTOR_ONE_TO_ONE, 0.0))

    def addCorrespondenceRejectorTrimmed(self, ratio: float = 0.5, min_correspondences: int = 0):
        """addCorrespondenceRejector(CorrespondenceRejectorTrimmed with setOverlapRatio(ratio) and
        setMinCorrespondences(min_correspondences)): the closest max(floor(ratio * m), min) pairs."""
        self._add_rejector((_lib.REJECTOR_TRIMMED, float(ratio), int(min_correspondences)))

    def getCorrespondenceRejectors(self) -> list[tuple]:
        """The chain after params.rejector_max_dist: (kind, value[, min_correspondences]) in the order added."""
        return list(self._chain)

    def _add_rejector(self, r: tuple):
        if len(self._chain) >= _lib.MAX_REJECTORS:
            raise PebError(-1, f"at most {_lib.MAX_REJECTORS} correspondence rejectors after the distance one")
        self._chain.append(r)

    def getConvergeCriteria(self) -> ConvergenceCriteria:
        return self._criteria

    # -- align ------------------------------------------------------------------------------------
    def align(self, guess=None, want_output: bool = True, want_correspondences: bool = False) -> np.ndarray | None:
        """align(output, guess): returns the (N, 4) transformed source (or None)."""
        if not self._have_source or not self._have_target:
            # let the library produce its own status / message
            pass
        g = _col_major(guess) if guess is not None else None
        res = IcpResult()
        n = self._n_src
        out = np.empty((n, 4), np.float32) if (want_output and n) else None
        idx = np.empty(n, np.int32) if (want_correspondences and n) else None
        d2 = np.empty(n, np.float32) if (want_correspondences and n) else None
        outs = (out.ctypes.data if out is not None else None, idx.ctypes.data if idx is not None else None,
                d2.ctypes.data if d2 is not None else None)
        if self._chain:
            arr, nc = _lib.rejector_array(self._chain)
            self._sctx.check(lib.peb_icp_align_ex(self._sctx.handle, g.ctypes.data if g is not None else None,
                                                  C.byref(self.params), arr, nc, C.byref(res), *outs))
        else:
            self._sctx.check(lib.peb_icp_align(self._sctx.handle, g.ctypes.data if g is not None else None,
                                               C.byref(self.params), C.byref(res), *outs))
        self._result = res
        self._criteria._state = res.state
        self.correspondences = (idx, d2) if want_correspondences else None
        return out

    def alignBatch(self, guesses) -> list[IcpResult]:
        """One source, one target, H initial poses: the shape of
        cv::ppf_match_3d::ICP::registerModelToScene(model, scene, poses)
        (pose_estimation/src/opencv_surface_match.cpp:94)."""
        g = np.ascontiguousarray(np.asarray(guesses, np.float32).reshape(-1, 4, 4).transpose(0, 2, 1)).reshape(-1, 16)
        H = g.shape[0]
        res = (IcpResult * max(H, 1))()
        if getattr(self.ctx, "is_multi", False):
            self.ctx.icp_align_batch(g, self.params, res, self._chain)  # contiguous blocks of hypotheses per device
        elif self._chain:
            arr, nc = _lib.rejector_array(self._chain)
            self.ctx.check(lib.peb_icp_align_batch_ex(self.ctx.handle, g.ctypes.data, H, C.byref(self.params), arr, nc, res))
        else:
            self.ctx.check(lib.peb_icp_align_batch(self.ctx.handle, g.ctypes.data, H, C.byref(self.params), res))
        return list(res)[:H]

    def hasConverged(self) -> bool:
        return bool(self._result and self._result.converged)

    def getFinalTransformation(self) -> np.ndarray:
        if self._result is None:
            return np.eye(4, dtype=np.float32)
        return result_matrix(self._result)

    def getFitnessScore(self, max_range: float = DBL_MAX) -> float:
        if self._result is None:
            raise ValueError("getFitnessScore before align")
        if max_range == self.params.fitness_max_range:
            return self._result.fitness
        return self._sctx.fitness_score(self.getFinalTransformation(), max_range)[0]

    @property
    def nr_iterations_(self) -> int:
        return self._result.iterations if self._result else 0

    @property
    def result(self) -> IcpResult | None:
        return self._result

    def trace(self) -> np.ndarray:
        """Per-iteration increments of the last align, (iterations, 4, 4)."""
        cap = max(self.nr_iterations_, 1)
        buf = np.zeros((cap, 16), np.float32)
        n = C.c_size_t(0)
        self._sctx.check(lib.peb_icp_trace(self._sctx.handle, buf.ctypes.data, cap, C.byref(n)))
        return buf[: n.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()


class IterativeClosestPointWithNormals(IterativeClosestPoint):
    """pcl::IterativeClosestPointWithNormals<PointNormal, PointNormal>: the estimator is
    TransformationEstimationPointToPlaneLLS ([PCL] registration/icp.h)."""

    _estimator = _lib.ESTIMATOR_POINT_TO_PLANE_LLS
