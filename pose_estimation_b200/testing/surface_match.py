"""OpenCVSurfaceMatch::find_object_in_scene made of the step entry points (peb_scene_prepare, peb_cv_normals, peb_ppf_match,
peb_cvicp_register, then the selection rule and the packing in Python): what peb_surface_match must reproduce byte for
byte.  Used by tests/test_gpu_surface_match.py and tools/bench_surface_match.py."""
from __future__ import annotations

import numpy as np


def steps(ctx, det, model6, cloud, params, prepare=False, filter_pose=None, filter_radius=0.0, filter_out="outliers",
          num_planes=0, leaf=0.0):
    """-> (scene (M, 6), refined PpfPose list, best, pose7, n_results), the fields of pcl.find_object_in_scene's result."""
    from .. import pcl, poses
    from .._lib import PpfPose

    pts = cloud
    if prepare:
        pts, _ = pcl.create_surface_match_pc(cloud, ctx, filter_pose, filter_radius, filter_out, num_planes, leaf)
    scene = pcl.compute_normals_pc3d(pts, params.normals_k, bool(params.flip_viewpoint), list(params.viewpoint), ctx=ctx)
    res = det.match(scene, params.relative_scene_sample_step, params.relative_scene_distance)
    sub = res[: params.max_icp_poses]
    if not sub:
        return scene, [], -1, np.zeros(7, np.float32), len(res)
    icp = pcl.CvIcp(params.icp.iterations, params.icp.tolerance, params.icp.rejection_scale, params.icp.num_levels, ctx=ctx)
    P, resid = icp.registerModelToScene(model6, scene, np.stack([r.matrix for r in sub]))
    refined = []
    for r, Pi, ri in zip(sub, P, resid):  # Pose3D::appendPose + residual
        x = PpfPose.from_buffer_copy(r)
        x.pose[:] = list(Pi.ravel())
        q, t, angle = poses.pose3d_from_matrix(Pi)
        x.q[:], x.t[:], x.angle, x.residual = list(q), list(t), angle, float(ri)
        refined.append(x)
    best = poses.select_best_pose([int(r.num_votes) for r in refined], [r.residual for r in refined], len(res))
    return scene, refined, best, poses.pack_pose3d(refined[best].t, refined[best].q, bool(params.reference_layout)), len(res)
