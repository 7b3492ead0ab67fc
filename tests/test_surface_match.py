"""peb_surface_match (OpenCVSurfaceMatch::find_object_in_scene in one call) without a GPU: the header compiles as pedantic
C99 and through the facade with the layout of the two new structs fixed, the packing of a refined record agrees between the
facade and pose_estimation_b200.poses, the reference's parameters are the defaults, and without a GPU the call fails loudly.
The chain itself is tested on the B200 in test_gpu_surface_match.py."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from surface_match_progs import build


def _has_gpu() -> bool:
    import torch

    return torch.cuda.is_available()


@pytest.mark.parametrize("which", ["c", "cpp"])
def test_header_and_facade_compile_with_the_struct_layout_fixed_and_fail_loudly_without_gpu(which, tmp_path):
    exe = build(tmp_path, which)
    if _has_gpu():
        return  # the run is checked in test_gpu_surface_match.py
    (tmp_path / "model.f32").write_bytes(np.zeros((4, 6), np.float32).tobytes())
    (tmp_path / "cloud.f32").write_bytes(np.zeros((4, 4), np.float32).tobytes())
    args = [str(tmp_path / "model.f32"), "4", str(tmp_path / "cloud.f32"), "4", "0", "0", str(tmp_path / "out")]
    r = subprocess.run([str(exe)] + (["run"] if which == "cpp" else []) + args, capture_output=True, text=True)
    assert r.returncode == 3 and "no CUDA device" in r.stderr and "no CPU fallback" in r.stderr, (r.returncode, r.stderr)
    assert not (tmp_path / "out.result").exists()


def _records(n, seed=0):
    from pose_estimation_b200._lib import PpfPose

    rng = np.random.default_rng(seed)
    recs = (PpfPose * n)()
    for i in range(n):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        if i % 3 == 0:
            q[0] = -abs(q[0])  # the packing takes q as it is (no sign normalisation)
        recs[i].q[:] = list(q)
        recs[i].t[:] = list(rng.normal(scale=0.5, size=3))
        recs[i].num_votes = int(rng.integers(0, 2000))
    return recs


def test_packing_from_a_refined_record_agrees_between_the_facade_and_python(tmp_path):
    from pose_estimation_b200 import poses

    exe = build(tmp_path, "cpp")
    recs = _records(50)
    (tmp_path / "recs.bin").write_bytes(bytes(recs))
    r = subprocess.run([str(exe), "pack", str(tmp_path / "recs.bin"), "50", str(tmp_path / "packed.f32")], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    packed = np.fromfile(tmp_path / "packed.f32", np.float32).reshape(50, 2, 7)
    for i, rec in enumerate(recs):
        ours = poses.pack_pose3d(rec.t, rec.q)
        lit = poses.pack_pose3d(rec.t, rec.q, reference_layout=True)
        assert packed[i, 0].tobytes() == ours.tobytes()
        assert packed[i, 1].tobytes() == lit.tobytes()
        assert lit[5] == 0.0 and lit[6] == np.float32(rec.q[0]) and ours[5] == np.float32(rec.q[3])
        assert np.array_equal(ours[:3], np.float32(rec.t[:])) and np.array_equal(ours[3:5], np.float32(rec.q[1:3]))


def test_pose3d_bookkeeping_matches_the_packed_rotation():
    """poses.pose3d_from_matrix (the Python side of Pose3D::appendPose): t is the pose's column, the angle the rotation's,
    and q the quaternion OpenCV's dcmToQuat (ppf.cu : dcm_to_quat) gives — that of the transposed rotation."""
    from pose_estimation_b200 import poses
    from pose_estimation_b200.testing import synth

    rng = np.random.default_rng(1)
    for k in range(40):
        R = synth.rotation_about(rng.normal(size=3), rng.uniform(0, np.pi) if k else np.pi - 1e-9)
        P = synth.make_pose(R, rng.normal(size=3))
        q, t, angle = poses.pose3d_from_matrix(P)
        w, x, y, z = q
        Rq = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                       [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                       [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        assert np.allclose(Rq, R.T, atol=1e-9) and np.array_equal(t, P[:3, 3])
        assert abs(angle - np.arccos(np.clip((np.trace(R) - 1) / 2, -1, 1))) < 1e-6


def test_defaults_are_the_reference_parameters_and_null_arguments_are_refused():
    from pose_estimation_b200 import _lib, pcl

    p = pcl.surface_match_params()
    assert (p.normals_k, p.flip_viewpoint, list(p.viewpoint), p.max_icp_poses) == (20, 1, [0.0, 0.0, 0.0], 6)
    assert (p.relative_scene_sample_step, p.relative_scene_distance) == (1.0, 0.03)
    assert (p.icp.iterations, p.icp.num_levels, p.icp.tolerance, p.icp.rejection_scale) == (250, 8, np.float32(0.005), 2.5)
    assert (p.reference_layout, p.reserved) == (0, 0)
    res = _lib.SurfaceMatchResult()
    assert _lib.lib.peb_surface_match(None, None, None, 0, 12, None, 0, None, 0.0, C.byref(p), (_lib.PpfPose * 6)(),
                                      C.byref(res), None, None) == -1


def test_python_call_fails_loudly_without_gpu():
    from pose_estimation_b200 import pcl

    if _has_gpu():
        pytest.skip("GPU present: covered by test_gpu_surface_match.py")
    with pytest.raises(pcl.PebError, match="no CPU fallback"):
        det = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=pcl.Context(0))
        pcl.find_object_in_scene(det, np.zeros((10, 3), np.float32))
