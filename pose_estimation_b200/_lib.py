"""ctypes binding of libpe_b200.so (include/pe_b200.h).

The shared library is the product; this module only declares its entry points.  There is no
fallback of any kind: if the library is missing, import of the package fails, and if no B200 is
present, `Context()` raises with the library's own message.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
import os as _os

# PEB_LIB_VARIANT is a development switch (register-cap experiments build libpe_b200_<variant>.so)
LIB_PATH = _HERE / ("libpe_b200" + ("_" + _os.environ["PEB_LIB_VARIANT"] if _os.environ.get("PEB_LIB_VARIANT") else "") + ".so")

PEB_OK = 0
STATUS_NAMES = {
    0: "PEB_OK",
    -1: "PEB_E_INVALID_ARG",
    -2: "PEB_E_NO_TARGET",
    -3: "PEB_E_NO_SOURCE",
    -4: "PEB_E_CUDA",
    -5: "PEB_E_OOM",
    -6: "PEB_E_UNSUPPORTED",
}

# pcl::registration::DefaultConvergenceCriteria<float>::ConvergenceState
CONVERGENCE_CRITERIA_NOT_CONVERGED = 0
CONVERGENCE_CRITERIA_ITERATIONS = 1
CONVERGENCE_CRITERIA_TRANSFORM = 2
CONVERGENCE_CRITERIA_ABS_MSE = 3
CONVERGENCE_CRITERIA_REL_MSE = 4
CONVERGENCE_CRITERIA_NO_CORRESPONDENCES = 5
CONVERGENCE_CRITERIA_FAILURE_AFTER_MAX_ITERATIONS = 6

ESTIMATOR_SVD = 0
ESTIMATOR_POINT_TO_PLANE_LLS = 1


class IcpParams(C.Structure):
    """peb_icp_params."""

    _fields_ = [
        ("max_iterations", C.c_int32),
        ("min_correspondences", C.c_int32),
        ("estimator", C.c_int32),
        ("max_iterations_similar", C.c_int32),
        ("max_corr_dist", C.c_double),
        ("transformation_epsilon", C.c_double),
        ("rotation_epsilon", C.c_double),
        ("euclidean_fitness_epsilon", C.c_double),
        ("abs_mse_threshold", C.c_double),
        ("rejector_max_dist", C.c_double),
        ("fitness_max_range", C.c_double),
    ]


REJECTOR_DISTANCE = 0
REJECTOR_MEDIAN_DISTANCE = 1
REJECTOR_ONE_TO_ONE = 2
REJECTOR_TRIMMED = 3
MAX_REJECTORS = 8


class Rejector(C.Structure):
    """peb_rejector: one entry of a correspondence rejector chain."""

    _fields_ = [("kind", C.c_int32), ("min_correspondences", C.c_int32), ("value", C.c_double)]


def rejector_array(chain):
    """chain: Rejector records (or (kind, value[, min_correspondences]) tuples) -> (ctypes array, count)."""
    arr = (Rejector * max(len(chain), 1))()
    for k, r in enumerate(chain):
        if isinstance(r, Rejector):
            arr[k] = r
        else:
            arr[k].kind = int(r[0])
            arr[k].value = float(r[1]) if len(r) > 1 else 0.0
            arr[k].min_correspondences = int(r[2]) if len(r) > 2 else 0
    return arr, len(chain)


class IcpResult(C.Structure):
    """peb_icp_result (96 bytes)."""

    _fields_ = [
        ("T", C.c_float * 16),
        ("fitness", C.c_double),
        ("last_mse", C.c_double),
        ("iterations", C.c_int32),
        ("converged", C.c_int32),
        ("state", C.c_int32),
        ("n_correspondences", C.c_int32),
    ]


class GicpParams(C.Structure):
    """peb_gicp_params."""

    _fields_ = [
        ("max_iterations", C.c_int32),
        ("k_correspondences", C.c_int32),
        ("max_inner_iterations", C.c_int32),
        ("reserved", C.c_int32),
        ("max_corr_dist", C.c_double),
        ("transformation_epsilon", C.c_double),
        ("rotation_epsilon", C.c_double),
        ("fitness_max_range", C.c_double),
    ]


class PrefilterParams(C.Structure):
    """peb_prefilter_params."""

    _fields_ = [
        ("use_sphere", C.c_int32),
        ("remove_inliers", C.c_int32),
        ("sphere_center", C.c_float * 3),
        ("sphere_radius", C.c_float),
        ("n_planes", C.c_int32),
        ("plane_band", C.c_float),
        ("planes", C.c_float * 32),
    ]


class SacParams(C.Structure):
    """peb_sac_params."""

    _fields_ = [
        ("distance_threshold", C.c_double),
        ("probability", C.c_double),
        ("max_iterations", C.c_int32),
        ("optimize_coefficients", C.c_int32),
        ("seed", C.c_uint32),
        ("reserved", C.c_int32),
    ]


class CvIcpParams(C.Structure):
    """peb_cvicp_params."""

    _fields_ = [("iterations", C.c_int32), ("num_levels", C.c_int32), ("tolerance", C.c_float), ("rejection_scale", C.c_float)]


class PpfParams(C.Structure):
    """peb_ppf_params."""

    _fields_ = [("relative_sampling_step", C.c_double), ("relative_distance_step", C.c_double), ("num_angles", C.c_double),
                ("position_threshold", C.c_double), ("rotation_threshold", C.c_double), ("use_weighted_avg", C.c_int32),
                ("reserved", C.c_int32)]


class PpfPose(C.Structure):
    """peb_ppf_pose = cv::ppf_match_3d::Pose3D."""

    _fields_ = [("pose", C.c_double * 16), ("q", C.c_double * 4), ("t", C.c_double * 3), ("angle", C.c_double),
                ("alpha", C.c_double), ("residual", C.c_double), ("num_votes", C.c_uint64), ("model_index", C.c_uint64)]

    @property
    def matrix(self):
        import numpy as np

        return np.array(self.pose, np.float64).reshape(4, 4)


class SurfaceMatchParams(C.Structure):
    """peb_surface_match_params (64 bytes)."""

    _fields_ = [("normals_k", C.c_int32), ("flip_viewpoint", C.c_int32), ("viewpoint", C.c_float * 3), ("max_icp_poses", C.c_int32),
                ("relative_scene_sample_step", C.c_double), ("relative_scene_distance", C.c_double), ("icp", CvIcpParams),
                ("reference_layout", C.c_int32), ("reserved", C.c_int32)]


class SurfaceMatchResult(C.Structure):
    """peb_surface_match_result (48 bytes)."""

    _fields_ = [("n_results", C.c_uint64), ("n_refined", C.c_int32), ("best", C.c_int32), ("pose7", C.c_float * 7),
                ("reserved", C.c_int32)]


class GridInfo(C.Structure):
    _fields_ = [
        ("origin", C.c_float * 3),
        ("cell", C.c_float),
        ("dims", C.c_int32 * 3),
        ("n_points", C.c_int32),
        ("n_cells", C.c_int64),
    ]


# every symbol include/pe_b200.h declares: name -> (restype, argtypes)
_vp, _sz, _i, _f, _d = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_double
_pp = C.POINTER
SYMBOLS = {
    "peb_ctx_create": (_i, [_i, _pp(_vp)]),
    "peb_ctx_destroy": (None, [_vp]),
    "peb_last_error": (C.c_char_p, [_vp]),
    "peb_version": (C.c_char_p, []),
    "peb_icp_params_default": (None, [_pp(IcpParams)]),
    "peb_ctx_stream": (_vp, [_vp]),
    "peb_ctx_launch_count": (C.c_uint64, [_vp]),
    "peb_ctx_set_int": (_i, [_vp, C.c_char_p, _i]),
    "peb_voxel_grid": (_i, [_vp, _vp, _sz, _sz, _f, _f, _f, C.c_uint, _vp, _pp(_sz)]),
    "peb_scene_prefilter": (_i, [_vp, _vp, _sz, _sz, _pp(PrefilterParams), _vp, _pp(_sz)]),
    "peb_scene_prefilter_dev": (_i, [_vp, _vp, _sz, _pp(PrefilterParams), _vp, _pp(_sz)]),
    "peb_sac_params_default": (None, [_pp(SacParams)]),
    "peb_sac_plane": (_i, [_vp, _vp, _sz, _sz, _pp(SacParams), _vp, _vp, _pp(_sz), _pp(C.c_int32)]),
    "peb_sac_plane_dev": (_i, [_vp, _vp, _sz, _pp(SacParams), _vp, _vp, _pp(_sz), _pp(C.c_int32)]),
    "peb_scene_prepare": (_i, [_vp, _vp, _sz, _sz, _pp(PrefilterParams), _i, _pp(SacParams), _f, _vp, _pp(_sz), _vp]),
    "peb_cvicp_register": (_i, [_vp, _vp, _sz, _vp, _sz, _pp(CvIcpParams), _vp, _sz, _vp]),
    "peb_ppf_params_default": (None, [_pp(PpfParams)]),
    "peb_ppf_train": (_i, [_vp, _vp, _sz, _pp(PpfParams), _pp(_vp)]),
    "peb_ppf_model_destroy": (None, [_vp]),
    "peb_ppf_model_sampled": (_i, [_vp, _vp, _sz, _pp(_sz)]),
    "peb_ppf_match": (_i, [_vp, _vp, _vp, _sz, _d, _d, _vp, _sz, _pp(_sz), _vp, _sz, _pp(_sz)]),
    "peb_surface_match_params_default": (None, [_pp(SurfaceMatchParams)]),
    "peb_surface_match": (_i, [_vp, _vp, _vp, _sz, _sz, _pp(PrefilterParams), _i, _pp(SacParams), _f, _pp(SurfaceMatchParams), _vp,
                               _pp(SurfaceMatchResult), _vp, _pp(_sz)]),
    "peb_normals_knn": (_i, [_vp, _vp, _sz, _sz, _i, _vp, _vp]),
    "peb_normals_knn_ex": (_i, [_vp, _vp, _sz, _sz, _i, _vp, _vp, _vp]),
    "peb_cv_normals": (_i, [_vp, _vp, _sz, _sz, _i, _i, _vp, _vp, _vp]),
    "peb_nn_search": (_i, [_vp, _vp, _sz, _sz, _vp, _vp]),
    "peb_nn_search_bruteforce": (_i, [_vp, _vp, _sz, _sz, _vp, _vp]),
    "peb_target_set": (_i, [_vp, _vp, _sz, _sz, _vp, _sz]),
    "peb_source_set": (_i, [_vp, _vp, _sz, _sz]),
    "peb_target_stage": (_i, [_vp, _vp, _sz, _sz, _vp, _sz]),
    "peb_target_build": (_i, [_vp]),
    "peb_target_clone": (_i, [_vp, _vp]),
    "peb_source_stage": (_i, [_vp, _vp, _sz, _sz]),
    "peb_source_build": (_i, [_vp]),
    "peb_source_clone": (_i, [_vp, _vp]),
    "peb_ctx_enable_peer": (_i, [_vp, _vp]),
    "peb_icp_align": (_i, [_vp, _vp, _pp(IcpParams), _pp(IcpResult), _vp, _vp, _vp]),
    "peb_icp_align_batch": (_i, [_vp, _vp, _sz, _pp(IcpParams), _vp]),
    "peb_icp_align_ex": (_i, [_vp, _vp, _pp(IcpParams), _vp, _sz, _pp(IcpResult), _vp, _vp, _vp]),
    "peb_icp_align_batch_ex": (_i, [_vp, _vp, _sz, _pp(IcpParams), _vp, _sz, _vp]),
    "peb_gicp_params_default": (None, [_pp(GicpParams)]),
    "peb_gicp_align": (_i, [_vp, _vp, _pp(GicpParams), _pp(IcpResult), _vp, _vp, _vp]),
    "peb_gicp_align_batch": (_i, [_vp, _vp, _sz, _pp(GicpParams), _vp]),
    "peb_gicp_covariances": (_i, [_vp, _i, _i, _vp]),
    "peb_fitness_score": (_i, [_vp, _vp, _d, _pp(_d), _pp(C.c_int32)]),
    "peb_target_set_dev": (_i, [_vp, _vp, _sz, _vp]),
    "peb_source_set_dev": (_i, [_vp, _vp, _sz]),
    "peb_icp_align_dev": (_i, [_vp, _vp, _pp(IcpParams), _vp]),
    "peb_icp_align_batch_dev": (_i, [_vp, _vp, _sz, _pp(IcpParams), _vp]),
    "peb_voxel_grid_dev": (_i, [_vp, _vp, _sz, _f, _f, _f, C.c_uint, _vp, _pp(_sz)]),
    "peb_normals_knn_dev": (_i, [_vp, _vp, _sz, _i, _vp, _vp]),
    "peb_cv_normals_dev": (_i, [_vp, _vp, _sz, _i, _i, _vp, _vp]),
    "peb_sync": (_i, [_vp]),
    "peb_target_grid_info": (_i, [_vp, _pp(GridInfo)]),
    "peb_icp_trace": (_i, [_vp, _vp, _sz, _pp(_sz)]),
    "peb_profile_read": (_i, [_vp, _vp, _sz, _pp(_sz)]),
    "peb_multi_create": (_i, [_i, _pp(_i), _pp(_vp)]),
    "peb_multi_destroy": (None, [_vp]),
    "peb_multi_last_error": (C.c_char_p, [_vp]),
    "peb_multi_size": (_i, [_vp]),
    "peb_multi_ctx": (_vp, [_vp, _i]),
    "peb_multi_set_int": (_i, [_vp, C.c_char_p, _i]),
    "peb_multi_shard_range": (None, [_sz, _i, _i, _pp(_sz), _pp(_sz)]),
    "peb_multi_target_set": (_i, [_vp, _vp, _sz, _sz, _vp, _sz]),
    "peb_multi_source_set": (_i, [_vp, _vp, _sz, _sz]),
    "peb_multi_icp_align_batch": (_i, [_vp, _vp, _sz, _pp(IcpParams), _vp]),
    "peb_multi_icp_align_batch_ex": (_i, [_vp, _vp, _sz, _pp(IcpParams), _vp, _sz, _vp]),
    "peb_multi_launch_count": (C.c_uint64, [_vp]),
}


def load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C pose_estimation_b200/csrc).  pose_estimation_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()
