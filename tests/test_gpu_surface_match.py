"""peb_surface_match on the B200: OpenCVSurfaceMatch::find_object_in_scene in one call equals the step-by-step entry points
(peb_scene_prepare, peb_cv_normals, peb_ppf_match, peb_cvicp_register, the selection rule and the packing) bit for bit,
finds the rendered object, leaves no stage's buffers clobbered, fails like the steps do, and gives the same bytes from C,
C++ and Python."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from pose_estimation_b200.testing import surface_match, synth
from surface_match_progs import build

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as _pcl

    return _pcl


@pytest.fixture(scope="module")
def ctx(pcl):
    c = pcl.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def case():
    """model (n x 6, object frame), organised cloud (x y z 1 rows, NaNs, background plane, clutter), ground truth."""
    rng = np.random.default_rng(3)
    surf = synth.Surface(1)
    gt = synth.default_gt_pose(rng)
    mp, mn = surf.sample(20000, rng)
    model6 = np.concatenate([mp, mn], 1).astype(np.float32)
    cloud = synth.render_scene(surf, gt, rng, 486, 300)
    return model6, cloud, gt


@pytest.fixture(scope="module")
def det(pcl, ctx, case):
    d = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=ctx)
    d.trainModel(case[0])
    yield d
    d.close()  # before its context (the fixture order tears ctx down after)


def _bytes(a):
    return np.ascontiguousarray(a).tobytes()


def assert_same(one, ref):
    refined, best, pose7, n_results, scene = one
    s_scene, s_refined, s_best, s_pose7, s_n = ref
    assert _bytes(scene) == _bytes(s_scene)
    assert n_results == s_n and best == s_best and len(refined) == len(s_refined)
    for a, b in zip(refined, s_refined):
        assert bytes(a) == bytes(b)  # pose, q, t, angle, alpha, residual, votes, model index
    assert _bytes(pose7) == _bytes(s_pose7)


def run_both(pcl, ctx, det, case, params, **prep):
    model6, cloud, _ = case
    src = prep.pop("cloud", cloud)
    one = pcl.find_object_in_scene(det, src, params, return_scene=True, **prep)
    ref = surface_match.steps(ctx, det, model6, src, params, **prep)
    assert_same(one, ref)
    return one


@pytest.fixture(scope="module")
def prepared(pcl, ctx, case):
    """What find_object_in_scene receives in the reference: the cloud after create_surface_match_pc (one plane removed)."""
    pts, _ = pcl.create_surface_match_pc(case[1], ctx, num_planes=1)
    return pts


@pytest.mark.parametrize("stride", [12, 16])
def test_one_call_equals_the_steps_on_a_prepared_cloud(pcl, ctx, det, case, prepared, stride):
    cloud = np.ascontiguousarray(prepared[:, :3]) if stride == 12 else prepared
    assert cloud.strides[0] == stride
    refined, best, pose7, n_results, scene = run_both(pcl, ctx, det, case, pcl.surface_match_params(), cloud=cloud)
    assert n_results > 5 and len(refined) == 6 and best >= 0 and scene.shape == (len(cloud), 6)


@pytest.mark.parametrize("num_planes,leaf", [(0, 0.0), (1, 0.0), (2, 0.0), (1, 0.002)])
def test_one_call_equals_the_steps_with_the_preparation(pcl, ctx, det, case, num_planes, leaf):
    run_both(pcl, ctx, det, case, pcl.surface_match_params(), prepare=True, num_planes=num_planes, leaf=leaf)


@pytest.mark.parametrize("filter_out", ["outliers", "inliers"])
def test_one_call_equals_the_steps_with_the_sphere_filter(pcl, ctx, det, case, filter_out):
    gt = case[2]
    # outliers: keep the ball around the object; inliers: cut a ball out of the clutter side
    centre = gt[:3, 3] if filter_out == "outliers" else gt[:3, 3] + np.array([0.2, 0.0, 0.0])
    refined, *_ = run_both(pcl, ctx, det, case, pcl.surface_match_params(), prepare=True, filter_pose=centre, filter_radius=0.12,
                           filter_out=filter_out, num_planes=1)
    assert refined


@pytest.mark.parametrize("layout", [0, 1])
def test_pose7_layouts_and_the_ground_truth(pcl, ctx, det, case, layout):
    params = pcl.surface_match_params(reference_layout=layout)
    refined, best, pose7, n_results, _ = run_both(pcl, ctx, det, case, params, prepare=True, num_planes=1)
    rot, trans = synth.pose_error(refined[best].matrix, case[2])
    assert rot < 0.01 and trans < 0.002, (rot, trans)  # the bar of test_ppf.py
    q = refined[best].q
    assert pose7[3] == np.float32(q[1]) and pose7[6] == np.float32(q[0])
    assert pose7[5] == (0.0 if layout else np.float32(q[3]))


def test_fewer_clustered_results_than_max_icp_poses(pcl, ctx, det, case):
    gt = case[2]
    params = pcl.surface_match_params(max_icp_poses=4096, relative_scene_sample_step=0.25)
    refined, best, _, n_results, _ = run_both(pcl, ctx, det, case, params, prepare=True, filter_pose=gt[:3, 3], filter_radius=0.06,
                                              num_planes=1)
    assert 0 < n_results < 4096 and len(refined) == n_results and best >= 0


def test_icp_iterations_zero_equals_the_steps(pcl, ctx, det, case, prepared):
    params = pcl.surface_match_params(icp=(0, 0.005, 2.5, 8))
    refined, *_ = run_both(pcl, ctx, det, case, params, cloud=prepared)
    assert refined and all(r.residual == 9999999999.0 for r in refined)


def test_no_stage_clobbers_another(pcl, ctx, det, case, prepared):
    params = pcl.surface_match_params()
    model6, cloud, _ = case
    before_steps = surface_match.steps(ctx, det, model6, cloud, params, prepare=True, num_planes=1)
    first = pcl.find_object_in_scene(det, cloud, params, prepare=True, num_planes=1, return_scene=True)
    # other work on the same context: the step entry points and a batched PCL ICP
    other = prepared[::3]
    pcl.compute_normals_pc3d(other, 12, ctx=ctx)
    det.match(pcl.compute_normals_pc3d(other, 20, ctx=ctx), 0.5, 0.05)
    icp = pcl.IterativeClosestPoint(ctx)
    icp.setInputSource(model6[:, :3])
    icp.setInputTarget(prepared)
    g = np.stack([synth.perturb_pose(case[2], np.random.default_rng(i), 3.0, 0.005) for i in range(8)])
    icp.alignBatch(g)
    again = pcl.find_object_in_scene(det, cloud, params, prepare=True, num_planes=1, return_scene=True)
    assert_same(again, before_steps)
    assert_same(first, before_steps)
    after_steps = surface_match.steps(ctx, det, model6, cloud, params, prepare=True, num_planes=1)
    assert_same(first, after_steps)


def _call(pcl, ctx, det_handle, cloud, params, refined=True, out=True, prm=True):
    from pose_estimation_b200._lib import PpfPose, SurfaceMatchResult, lib

    res = SurfaceMatchResult()
    recs = (PpfPose * max(params.max_icp_poses, 1))()
    p = np.ascontiguousarray(cloud, np.float32)
    return lib.peb_surface_match(ctx.handle, det_handle, p.ctypes.data, p.shape[0], p.strides[0], None, 0, None, 0.0,
                                 C.byref(params) if prm else None, recs if refined else None, C.byref(res) if out else None, None,
                                 None), res


def test_errors_and_edges(pcl, ctx, det, case, prepared):
    model6, cloud, gt = case
    params = pcl.surface_match_params()
    # the scene empties during the preparation: PEB_OK, nothing found, no ICP
    refined, best, pose7, n_results, scene = pcl.find_object_in_scene(det, cloud, params, prepare=True, filter_pose=[5.0, 5.0, 5.0],
                                                                      filter_radius=0.01, return_scene=True)
    assert (refined, best, n_results, scene.shape) == ([], -1, 0, (0, 6)) and not pose7.any()
    assert pcl.find_object_in_scene(det, np.empty((0, 3), np.float32), params)[1:4:2] == (-1, 0)
    # k above the number of finite points: the error of peb_cv_normals, same code and message
    few = prepared[:10]
    with pytest.raises(pcl.PebError) as e_step:
        pcl.compute_normals_pc3d(few, 20, ctx=ctx)
    with pytest.raises(pcl.PebError) as e_one:
        pcl.find_object_in_scene(det, few, params)
    assert e_one.value.code == e_step.value.code == -1 and str(e_one.value) == str(e_step.value)
    # a model trained on another context
    ctx2 = pcl.Context(0)
    det2 = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=ctx2)
    det2.trainModel(model6)
    rc, _ = _call(pcl, ctx, det2._model, prepared, params)
    assert rc == -1 and b"another context" in pcl.lib.peb_last_error(ctx.handle)
    det2.close()
    ctx2.close()
    # max_icp_poses outside [1, 4096]
    for bad in (0, 4097):
        rc, _ = _call(pcl, ctx, det._model, prepared, pcl.surface_match_params(max_icp_poses=bad))
        assert rc == -1 and b"max_icp_poses" in pcl.lib.peb_last_error(ctx.handle)
    # NULL outputs / params
    for kw in ({"refined": False}, {"out": False}, {"prm": False}):
        rc, _ = _call(pcl, ctx, det._model, prepared, params, **kw)
        assert rc == -1
    # the context still works after every refusal
    run_both(pcl, ctx, det, case, params, cloud=prepared)


def test_same_bytes_from_c_cpp_and_python(pcl, ctx, det, case, tmp_path):
    model6, cloud, _ = case
    (tmp_path / "model.f32").write_bytes(_bytes(model6))
    (tmp_path / "cloud.f32").write_bytes(_bytes(cloud))
    refined, best, pose7, n_results, scene = pcl.find_object_in_scene(det, cloud, pcl.surface_match_params(), prepare=True,
                                                                      num_planes=1, return_scene=True)
    for which in ("c", "cpp"):
        exe = build(tmp_path, which)
        args = [str(tmp_path / "model.f32"), str(len(model6)), str(tmp_path / "cloud.f32"), str(len(cloud)), "1", "0",
                str(tmp_path / which)]
        r = subprocess.run([str(exe)] + (["run"] if which == "cpp" else []) + args, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert (tmp_path / f"{which}.scene").read_bytes() == _bytes(scene)
        assert (tmp_path / f"{which}.refined").read_bytes() == b"".join(bytes(x) for x in refined)
        res = np.frombuffer((tmp_path / f"{which}.result").read_bytes(), np.uint8)
        assert int(res[:8].view(np.uint64)[0]) == n_results and int(res[12:16].view(np.int32)[0]) == best
        assert res[16:44].tobytes() == _bytes(pose7)


def test_a_model_destroyed_after_its_context_leaves_later_work_alone(pcl, case, prepared):
    """peb_ppf_model_destroy never reads the context the model was trained on: destroying the model after the context
    (what a garbage collector may do with the two Python objects) frees its memory and leaves no CUDA error behind for the
    next call on another context."""
    c1 = pcl.Context(0)
    d1 = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=c1)
    d1.trainModel(case[0])
    c1.close()
    d1.close()
    c2 = pcl.Context(0)
    icp = pcl.IterativeClosestPoint(c2)
    icp.setInputSource(case[0][::4, :3])
    icp.setInputTarget(prepared)
    icp.align(case[2])
    assert icp.nr_iterations_ >= 1  # the align ran: no stale error from the destroy above
    c2.close()

