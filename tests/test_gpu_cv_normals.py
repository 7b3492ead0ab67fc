"""peb_cv_normals / peb_cv_normals_dev on the B200 against the oracle (tests/cv_normals_oracle.cpp : orc_cv_normals).

Wherever the device's neighbour list equals the oracle's, the row is bit-identical (uint32 view): the same float products,
double sums in the same order, the same Jacobi rotations (-fmad=false) and the same float flip.  The lists themselves
agree up to equidistant ties (tie_ok): the grid search orders ties by grid position, the kd-tree by its visiting order."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from pose_estimation_b200.testing import synth
from test_cv_normals import ROOT, same_bits, wavy_patch
import cv_normals_oracle as cvo
from util import tie_ok

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as m

    return m


@pytest.fixture(scope="module")
def ctx(pcl):
    return pcl.Context(0)


def check_against_oracle(pcl, ctx, oracle, P, k, flip=True, vp=(0.0, 0.0, 0.0), min_same=0.99):
    out, nn = pcl.compute_normals_pc3d(P, k, flip, vp, ctx=ctx, return_neighbours=True)
    ref, rnn = cvo.cv_normals(P, k, flip=flip, viewpoint=vp, want_nn=True, threads=0)
    xyz = np.asarray(P, np.float32)[:, :3]
    assert same_bits(out[:, :3], xyz).all()
    assert tie_ok(xyz, xyz, nn.reshape(-1), rnn.reshape(-1))
    same = (nn == rnn).all(1)
    assert same.mean() >= min_same, same.mean()
    assert same_bits(out[same], ref[same]).all()
    return out, nn, same


@pytest.mark.parametrize("k", [3, 8, 20, 24, 32, 33, 64, 192])
def test_device_matches_oracle_bitwise(pcl, ctx, oracle, k):
    P = wavy_patch(12000, seed=k)
    check_against_oracle(pcl, ctx, oracle, P, k)


@pytest.mark.parametrize("flip,vp", [(False, (0.0, 0.0, 0.0)), (True, (0.05, -0.2, 1.5)), (True, (0.0, 0.0, 0.72))])
@pytest.mark.parametrize("k", [20, 40])
def test_flip_and_viewpoint(pcl, ctx, oracle, flip, vp, k):
    P = wavy_patch(8000, seed=3)
    check_against_oracle(pcl, ctx, oracle, P, k, flip, vp)


@pytest.mark.parametrize("stride", [12, 16, 24])
def test_strides(pcl, ctx, oracle, stride):
    P = wavy_patch(6000, seed=4)
    rec = np.full((len(P), stride // 4), 7.0, np.float32)  # the padding must not be read
    rec[:, :3] = P
    out, _, _ = check_against_oracle(pcl, ctx, oracle, rec, 20)
    assert same_bits(out, pcl.compute_normals_pc3d(P, 20, ctx=ctx)).all()


def test_c2_scene(pcl, ctx, oracle):
    scene = synth.make_c2(downsample=lambda pts, leaf: oracle.voxel_grid(pts, leaf)[0]).target
    assert len(scene) > 150000
    out, _, same = check_against_oracle(pcl, ctx, oracle, scene[:, :3], 20)
    assert (out[:, 5] <= 0).mean() > 0.99  # towards the camera at the origin


def test_dev_entry_gives_the_host_entrys_bytes(pcl, ctx):
    import torch

    P = wavy_patch(20000, seed=8)
    P[17] = np.nan
    host = pcl.compute_normals_pc3d(P, 20, True, (0.0, 0.1, 0.0), ctx=ctx)
    d_in = torch.zeros((len(P), 4), dtype=torch.float32, device="cuda")
    d_in[:, :3] = torch.from_numpy(P).cuda()
    d_out = torch.empty((len(P), 6), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    vp = np.float32([0.0, 0.1, 0.0])
    ctx.check(pcl.lib.peb_cv_normals_dev(ctx.handle, d_in.data_ptr(), len(P), 20, 1, vp.ctypes.data, d_out.data_ptr()))
    ctx.sync()
    assert same_bits(d_out.cpu().numpy(), host).all()


def test_edge_cases(pcl, ctx, oracle):
    rng = np.random.default_rng(12)
    P = rng.normal(0, 0.01, (300, 3)).astype(np.float32) + np.float32([0, 0, 0.7])
    P[[5, 40, 41]] = np.nan
    P[77, 2] = np.inf
    out, nn, _ = check_against_oracle(pcl, ctx, oracle, P, 12, min_same=0.95)
    bad = [5, 40, 41, 77]
    assert np.isnan(out[bad, 3:]).all() and (nn[bad] == -1).all()
    assert out[77, 2] == np.inf and np.isnan(out[5, :3]).all()
    # duplicates with exact float products: zero covariance -> (0, 0, +-1)
    D = np.repeat(np.float32([[0.5, 0.25, 0.75]]), 40, 0)
    assert (pcl.compute_normals_pc3d(D, 10, ctx=ctx)[:, 3:] == np.float32([0, 0, -1])).all()
    assert (pcl.compute_normals_pc3d(D, 40, True, (0, 0, 2), ctx=ctx)[:, 3:] == np.float32([0, 0, 1])).all()
    assert (pcl.compute_normals_pc3d(D, 5, False, ctx=ctx)[:, 3:] == np.float32([0, 0, 1])).all()
    # collinear points
    L = np.zeros((200, 3), np.float32)
    L[:, 0] = np.linspace(0, 0.2, 200)
    L[:, 2] = 0.7
    out, _, _ = check_against_oracle(pcl, ctx, oracle, L, 6, min_same=0.0)  # evenly spaced: ties everywhere
    assert np.allclose(np.linalg.norm(out[:, 3:], axis=1), 1, atol=1e-6) and np.abs(out[:, 3]).max() < 1e-3
    # n = 0
    assert pcl.compute_normals_pc3d(np.empty((0, 3), np.float32), 20, ctx=ctx).shape == (0, 6)
    # the three error codes: k < 1, k > the finite points, k > 192
    Q = P[:20].copy()  # 19 finite points
    for cloud, k, code in ((P, 0, -1), (Q, 20, -1), (P, 193, -6)):
        with pytest.raises(pcl.PebError) as e:
            pcl.compute_normals_pc3d(cloud, k, ctx=ctx)
        assert e.value.code == code, (k, e.value)
    check_against_oracle(pcl, ctx, oracle, Q, 19, min_same=0.0)  # the largest k: every finite point is a neighbour
    allnan = np.full((10, 3), np.nan, np.float32)
    with pytest.raises(pcl.PebError) as e:
        pcl.compute_normals_pc3d(allnan, 1, ctx=ctx)
    assert e.value.code == -1


def test_facade_and_c_program_match_python(pcl, ctx, tmp_path):
    P = wavy_patch(3000, seed=9)
    (tmp_path / "in.f32").write_bytes(P.tobytes())
    ref = pcl.compute_normals_pc3d(P, 20, True, ctx=ctx)
    lib_dir = ROOT / "pose_estimation_b200"
    src = ROOT / "tests" / "cpp" / "cv_normals_check.cpp"
    for cc in (["gcc", "-x", "c", "-std=c99"], ["g++", "-std=c++17", "-O1"]):
        exe = tmp_path / "check"
        r = subprocess.run(cc + ["-I", str(ROOT / "include"), str(src), "-o", str(exe), "-L", str(lib_dir), "-lpe_b200",
                                 "-lm", f"-Wl,-rpath,{lib_dir}"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run([str(exe), str(tmp_path / "in.f32"), "3000", "20", "1", str(tmp_path / "out.f32")],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        got = np.frombuffer((tmp_path / "out.f32").read_bytes(), np.float32).reshape(-1, 6)
        assert same_bits(got, ref).all()


def test_ppf_then_cv_icp_recover_the_ground_truth_with_these_normals(pcl, ctx, oracle):
    """test_ppf.py's scene, with the scene normals from peb_cv_normals instead of the PCL formula."""
    rng = np.random.default_rng(3)
    surf = synth.Surface(1)
    gt = synth.default_gt_pose(rng)
    mp, mn = surf.sample(20000, rng)
    model6 = np.concatenate([mp, mn], 1).astype(np.float32)
    scene = synth.render_scene(surf, gt, rng, 486, 300)
    fin = scene[np.isfinite(scene).all(1)]
    ds = oracle.voxel_grid(fin[fin[:, 2] < 0.735], 0.002)[0]
    scene6 = pcl.compute_normals_pc3d(ds[:, :3], 20, True, (0.0, 0.0, 0.0), ctx=ctx)
    assert np.isfinite(scene6).all()
    det = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=ctx)
    det.trainModel(model6)
    res = det.match(scene6, 1.0, 0.03)
    det.close()
    rot, trans = synth.pose_error(res[0].matrix, gt)
    assert trans < 0.01 and rot < 0.35
    icp = pcl.CvIcp(250, 0.005, 2.5, 8, ctx=ctx)
    P, _ = icp.registerModelToScene(model6, scene6, np.array([res[0].matrix]))
    rot2, trans2 = synth.pose_error(P[0], gt)
    assert rot2 < 0.01 and trans2 < 0.002
