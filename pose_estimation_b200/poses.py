"""The step right after the path (SURVEY.md 8f rank 3): which refined hypothesis the node returns and
how it is packed into the 7 floats it publishes.  Host-side mirror of
pose_estimation/src/opencv_surface_match.cpp:100-142 (same functions as in include/pe_b200/pcl_facade.hpp);
no device work and no arithmetic of the hot path."""
from __future__ import annotations

import numpy as np


def select_best_pose(num_votes, residual, n_results_total: int) -> int:
    """opencv_surface_match.cpp:100-124: most votes wins; with more than 5 matcher results the lowest
    residual among poses with more than 400 votes overrides it (last assignment wins, as written)."""
    max_votes = 0
    min_res = np.float32(10000.0)
    best = 0
    for i, (v, r) in enumerate(zip(num_votes, residual)):
        if v > max_votes:
            max_votes = v
            best = i
        if n_results_total > 5 and r < min_res and v > 400:
            min_res = np.float32(r)
            best = i
    return best


def rotation_to_quat(T) -> np.ndarray:
    """4x4 (row-indexed) -> unit quaternion (w, x, y, z), w >= 0."""
    m = np.asarray(T, np.float64)[:3, :3]
    tr = m[0, 0] + m[1, 1] + m[2, 2]
    if tr > 0:
        s = np.sqrt(tr + 1.0) * 2
        q = [0.25 * s, (m[2, 1] - m[1, 2]) / s, (m[0, 2] - m[2, 0]) / s, (m[1, 0] - m[0, 1]) / s]
    elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
        s = np.sqrt(1.0 + m[0, 0] - m[1, 1] - m[2, 2]) * 2
        q = [(m[2, 1] - m[1, 2]) / s, 0.25 * s, (m[0, 1] + m[1, 0]) / s, (m[0, 2] + m[2, 0]) / s]
    elif m[1, 1] > m[2, 2]:
        s = np.sqrt(1.0 + m[1, 1] - m[0, 0] - m[2, 2]) * 2
        q = [(m[0, 2] - m[2, 0]) / s, (m[0, 1] + m[1, 0]) / s, 0.25 * s, (m[1, 2] + m[2, 1]) / s]
    else:
        s = np.sqrt(1.0 + m[2, 2] - m[0, 0] - m[1, 1]) * 2
        q = [(m[1, 0] - m[0, 1]) / s, (m[0, 2] + m[2, 0]) / s, (m[1, 2] + m[2, 1]) / s, 0.25 * s]
    q = np.array(q)
    return -q if q[0] < 0 else q


def pack_pose(T, reference_layout: bool = False) -> np.ndarray:
    """{x, y, z, qx, qy, qz, qw} float32.  reference_layout=True reproduces opencv_surface_match.cpp:133-142
    literally (qz is never written: pose[6] gets q[3] and is overwritten with q[0])."""
    T = np.asarray(T, np.float64)
    q = rotation_to_quat(T)
    pose = np.zeros(7, np.float32)
    pose[:3] = T[:3, 3]
    pose[3], pose[4] = q[1], q[2]
    if reference_layout:
        pose[6] = q[3]
        pose[6] = q[0]
    else:
        pose[5], pose[6] = q[3], q[0]
    return pose


def pack_pose3d(t, q, reference_layout: bool = False) -> np.ndarray:
    """{x, y, z, qx, qy, qz, qw} float32 from a Pose3D's t and q (w, x, y, z), as opencv_surface_match.cpp:133-142 builds
    it (pe_b200::pack_pose3d).  reference_layout=True: qz is never written, pose[6] gets q[3] and then q[0]."""
    t = np.asarray(t, np.float64)
    q = np.asarray(q, np.float64)
    pose = np.zeros(7, np.float32)
    pose[:3] = t[:3]
    pose[3], pose[4] = q[1], q[2]
    if reference_layout:
        pose[6] = q[3]
        pose[6] = q[0]
    else:
        pose[5], pose[6] = q[3], q[0]
    return pose


def pose3d_from_matrix(P):
    """Pose3D::appendPose's bookkeeping once the appended pose P (4 x 4, float64) is known: (q (w, x, y, z), t, angle) with
    OpenCV's dcmToQuat and the angle from the trace (the same operations as ppf.cu, so the same bits)."""
    import math

    P = np.asarray(P, np.float64).reshape(4, 4)
    R = [float(v) for v in P[:3, :3].ravel()]
    tr = R[0] + R[4] + R[8]
    q = [0.0] * 4
    if tr > 0:
        q[0], q[1], q[2], q[3] = tr + 1.0, R[5] - R[7], R[6] - R[2], R[1] - R[3]
    else:
        i = 0
        if R[4] > R[0]:
            i = 1
        if R[8] > R[3 * i + i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        q[i + 1] = R[3 * i + i] - R[3 * j + j] - R[3 * k + k] + 1.0
        q[j + 1] = R[3 * i + j] + R[3 * j + i]
        q[k + 1] = R[3 * i + k] + R[3 * k + i]
        q[0] = R[3 * j + k] - R[3 * k + j]
    s = 1.0 / math.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
    q = [v * s for v in q]
    eps = 1.192092896e-07
    angle = 0.0 if abs(tr - 3) <= eps else (math.pi if abs(tr + 1) <= eps else math.acos((tr - 1) / 2))
    return np.array(q), P[:3, 3].copy(), angle


def _eigen_quat_from_matrix(m: np.ndarray) -> np.ndarray:
    """Eigen::Quaternionf(Matrix3f) (Eigen/src/Geometry/Quaternion.h : quaternionbase_assign_impl), float32,
    -> (x, y, z, w), no sign normalisation."""
    f = np.float32
    m = np.asarray(m, f)
    t = f(m[0, 0] + m[1, 1] + m[2, 2])
    q = np.zeros(4, f)
    if t > 0:
        t = f(np.sqrt(f(t + f(1.0))))
        q[3] = f(0.5) * t
        t = f(0.5) / t
        q[0] = f(m[2, 1] - m[1, 2]) * t
        q[1] = f(m[0, 2] - m[2, 0]) * t
        q[2] = f(m[1, 0] - m[0, 1]) * t
    else:
        i = 0
        if m[1, 1] > m[0, 0]:
            i = 1
        if m[2, 2] > m[i, i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = f(np.sqrt(f(f(f(m[i, i] - m[j, j]) - m[k, k]) + f(1.0))))
        q[i] = f(0.5) * t
        t = f(0.5) / t
        q[3] = f(m[k, j] - m[j, k]) * t
        q[j] = f(m[j, i] + m[i, j]) * t
        q[k] = f(m[k, i] + m[i, k]) * t
    return q


def obj_in_base_frame(pose7, he_calibration) -> np.ndarray:
    """pose_estimation_manager/src/pose_transformer.cpp:78-121 (PoseTransformer::obj_in_base_frame): the published
    {x, y, z, qx, qy, qz, qw} in the camera frame -> hand-eye calibration -> the grasp frame the manager sends to the
    robot: the object's y axis is kept, z is the base's -z (or +x when y is more than ~37 degrees out of the
    horizontal) made orthogonal to y, x = y x z.  float32 like the reference's Eigen types; returns 7 doubles."""
    f = np.float32
    p = np.asarray(pose7, f)
    q = p[3:7].astype(f)
    q = (q / f(np.sqrt(f(q @ q)))).astype(f)  # Quaternionf::normalize
    x, y, z, w = q
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]], f)
    cam = np.eye(4, dtype=f)
    cam[:3, :3] = R
    cam[:3, 3] = p[:3]
    base = (np.asarray(he_calibration, f) @ cam).astype(f)  # apply_he_calibration
    yv = base[:3, 1].copy()
    z_base = np.array([0.0, 0.0, -1.0], f)
    if abs(yv[2]) > f(0.6):
        z_base = np.array([1.0, 0.0, 0.0], f)
    zv = (z_base - (f(z_base @ yv) / f(yv @ yv)) * yv).astype(f)
    xv = np.cross(yv, zv).astype(f)
    rot = np.stack([xv / f(np.linalg.norm(xv)), yv / f(np.linalg.norm(yv)), zv / f(np.linalg.norm(zv))], 1).astype(f)
    qb = _eigen_quat_from_matrix(rot)
    qb = (qb / f(np.sqrt(f(qb @ qb)))).astype(f)
    return np.array([base[0, 3], base[1, 3], base[2, 3], qb[0], qb[1], qb[2], qb[3]], np.float64)


def hover_pose(pose7, he_calibration, offset: float = 0.1) -> np.ndarray:
    """pose_transformer.cpp:70-75: the grasp pose lifted by 0.1 m along the base z axis."""
    out = obj_in_base_frame(pose7, he_calibration)
    out[2] += offset
    return out
