"""Correspondence rejector chains on the B200 (peb_icp_align_ex / peb_icp_align_batch_ex / peb_multi_icp_align_batch_ex):
against the CPU oracle's chain (tests/rejector_oracle.cpp : reject_chain), batch against single aligns, launch knobs that
must not change a record, and the facade's chain (tests/cpp/rejector_check.cpp)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import rejector_oracle as RO
from oracle import DBL_MAX, default_params
from pose_estimation_b200.testing import synth
from test_rejectors import CLUTTER_KW, clutter_problem
from util import pose_delta, tie_ok

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
D, MED, O2O, TRIM = 0, 1, 2, 3
CHAINS = [[(MED, 1.0)], [(O2O,)], [(TRIM, 0.8)], [(D, 0.004), (O2O,), (MED, 1.0)]]
ROT_TOL = TRANS_TOL = 1e-5


@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as m

    return m


@pytest.fixture(scope="module")
def ctx(pcl):
    c = pcl.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def c1():
    return synth.make_c1(20000, seed=1)


@pytest.fixture(scope="module")
def scene_small(oracle):
    return synth.make_c2(scale=0.25, downsample=lambda p, leaf: oracle.voxel_grid(p, leaf)[0])


def _icp(pcl, ctx, source, target, chain, normals=None, lls=False, **kw):
    icp = (pcl.IterativeClosestPointWithNormals if lls else pcl.IterativeClosestPoint)(ctx)
    icp.setInputSource(source)
    icp.setInputTarget(target, normals)
    for k, v in kw.items():
        setattr(icp.params, k, v)
    for r in chain:
        if r[0] == D:
            icp.addCorrespondenceRejectorDistance(r[1])
        elif r[0] == MED:
            icp.addCorrespondenceRejectorMedianDistance(r[1])
        elif r[0] == O2O:
            icp.addCorrespondenceRejectorOneToOne()
        else:
            icp.addCorrespondenceRejectorTrimmed(*r[1:])
    return icp


def _records(res):
    return b"".join(bytes(r) for r in res)


def _check_single(pcl, ctx, oracle, source, target, guess, chain, normals=None, lls=False, **kw):
    icp = _icp(pcl, ctx, source, target, chain, normals, lls, **kw)
    icp.align(guess, want_correspondences=True)
    got = icp.result
    prm = default_params(**kw)
    if lls:
        prm.estimator = 1
    ref = RO.ChainIcp(target, normals, wide_accum=True).align(source, guess, prm, chain=chain)
    r = ref["result"]
    assert got.state == r.state and got.iterations == r.iterations, (got.state, r.state, got.iterations, r.iterations)
    assert got.n_correspondences == r.n_correspondences
    rot, tr = pose_delta(icp.getFinalTransformation(), r.matrix())
    assert rot < ROT_TOL and tr < TRANS_TOL, (rot, tr)
    # the kept set of the last iteration: every difference is an equidistant tie
    idx, _ = icp.correspondences
    moved = synth.apply_pose(icp.getFinalTransformation(), np.asarray(source, np.float64)[:, :3])
    assert tie_ok(target, moved, idx, ref["corr_idx"], tol=1e-5)
    return icp


@pytest.mark.parametrize("chain", CHAINS)
def test_single_align_matches_oracle_c1(pcl, ctx, oracle, c1, chain):
    _check_single(pcl, ctx, oracle, c1.source, c1.target, c1.guess, chain, max_iterations=20, abs_mse_threshold=-1.0)


@pytest.mark.parametrize("chain", CHAINS)
def test_single_align_matches_oracle_scene_point_to_plane(pcl, ctx, oracle, scene_small, chain):
    p = scene_small
    nrm = oracle.normals(p.target, 10)[:, :3]
    _check_single(pcl, ctx, oracle, p.source, p.target, p.guess, chain, normals=nrm, lls=True, max_iterations=15,
                  max_corr_dist=0.01, abs_mse_threshold=-1.0)


@pytest.mark.parametrize("chain", CHAINS[:2])
def test_single_align_matches_oracle_scene_svd(pcl, ctx, oracle, scene_small, chain):
    p = scene_small
    _check_single(pcl, ctx, oracle, p.source, p.target, p.guess, chain, max_iterations=15, max_corr_dist=0.01,
                  transformation_epsilon=1e-10)


def _guesses(p, H, seed=3, spread=1.0):
    rng = np.random.default_rng(seed)
    return np.stack([synth.perturb_pose(p.guess, rng, 2.0 * spread, 0.003 * spread) for _ in range(H)])


KW_STOP = dict(max_iterations=40, transformation_epsilon=1e-9, max_corr_dist=0.01)


@pytest.mark.parametrize("chain", CHAINS)
def test_batch_matches_single_and_oracle(pcl, ctx, oracle, scene_small, chain):
    p = scene_small
    G = _guesses(p, 6, spread=2.0)  # hypotheses that stop at different iterations
    icp = _icp(pcl, ctx, p.source, p.target, chain, **KW_STOP)
    batch = icp.alignBatch(G)
    ref = RO.ChainIcp(p.target, wide_accum=True).align_batch(p.source, G, default_params(**KW_STOP), chain=chain)
    iters = set()
    for h in range(len(G)):
        icp.align(G[h], want_output=False)
        s, b, r = icp.result, batch[h], ref[h]
        iters.add(b.iterations)
        assert (b.state, b.iterations, b.n_correspondences) == (s.state, s.iterations, s.n_correspondences)
        assert max(pose_delta(synth_matrix(b), synth_matrix(s))) < 1e-6
        assert b.state == r.state and b.n_correspondences == r.n_correspondences, (h, b.state, r.state)
        rot, tr = pose_delta(synth_matrix(b), r.matrix())
        assert rot < ROT_TOL and tr < TRANS_TOL, (h, rot, tr)
    assert len(iters) > 1


def synth_matrix(r):
    return np.array(r.T, np.float32).reshape(4, 4).T


@pytest.mark.parametrize("H", [1, 16, 33, 300])
def test_launch_knobs_leave_records_unchanged(pcl, scene_small, H):
    p = scene_small
    G = _guesses(p, H, seed=H)
    chain = [(D, 0.006), (O2O,), (MED, 1.5), (TRIM, 0.9)]
    knobs = [dict(), dict(flag_deps=0), dict(batch_streams=1), dict(batch_streams=4), dict(split_moments=0),
             dict(split_min_hyp=2), dict(warm_bin=1), dict(cert_margin_x1000=250), dict(nn_cache_from=3),
             dict(warm_upfront=2), dict(warm_graph_queue=8), dict(nn_group=4), dict(profile=2)]
    base = None
    for k in knobs:
        with pcl.Context(0) as c:
            for key, v in k.items():
                c.set_int(key, v)
            icp = _icp(pcl, c, p.source, p.target, chain, **KW_STOP)
            res = icp.alignBatch(G)
            assert all(r.state != -1000 for r in res)
            rec = _records(res)
        if base is None:
            base = rec
        assert rec == base, k


def test_empty_chain_equals_plain_entry_points(pcl, ctx, scene_small):
    import ctypes as C

    from pose_estimation_b200 import _lib

    p = scene_small
    G = _guesses(p, 40)
    icp = _icp(pcl, ctx, p.source, p.target, [], **KW_STOP)
    plain = icp.alignBatch(G)
    g = np.ascontiguousarray(np.asarray(G, np.float32).transpose(0, 2, 1)).reshape(-1, 16)
    res = (_lib.IcpResult * len(G))()
    ctx.check(_lib.lib.peb_icp_align_batch_ex(ctx.handle, g.ctypes.data, len(G), C.byref(icp.params), None, 0, res))
    assert _records(res) == _records(plain)
    one = _lib.IcpResult()
    ctx.check(_lib.lib.peb_icp_align_ex(ctx.handle, g[:16].ctypes.data, C.byref(icp.params), None, 0, C.byref(one),
                                        None, None, None))
    icp.align(G[0], want_output=False)
    assert bytes(one) == bytes(icp.result)


def test_too_few_pairs_left(pcl, ctx, c1):
    icp = _icp(pcl, ctx, c1.source, c1.target, [(TRIM, 0.0, 2)], max_iterations=10)
    icp.align(c1.guess, want_output=False)
    assert icp.result.state == 5 and icp.result.n_correspondences == 2
    res = icp.alignBatch(np.stack([c1.guess] * 20))
    assert all(r.state == 5 and r.n_correspondences == 2 for r in res)


def test_multi_device_equals_one_context(pcl, scene_small):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    p = scene_small
    G = _guesses(p, 64)
    chain = [(O2O,), (MED, 1.0)]
    devs = list(range(torch.cuda.device_count()))
    with pcl.MultiContext(devs) as m:
        icp = _icp(pcl, m, p.source, p.target, chain, **KW_STOP)
        many = icp.alignBatch(G)
    for i in devs:
        with pcl.Context(i) as c:
            lo, hi = (len(G) + len(devs) - 1) // len(devs) * i, min(len(G), (len(G) + len(devs) - 1) // len(devs) * (i + 1))
            if lo >= hi:
                continue
            one = _icp(pcl, c, p.source, p.target, chain, **KW_STOP).alignBatch(G[lo:hi])
            assert _records(one) == _records(many[lo:hi])


def test_trimmed_rejection_recovers_the_pose_in_clutter(pcl, ctx, oracle):
    src, tgt, gt = clutter_problem()
    kw = dict(CLUTTER_KW)
    icp = _icp(pcl, ctx, src, tgt, [(TRIM, 0.7)], **kw)
    icp.align(None, want_output=False)
    ref = RO.ChainIcp(tgt, wide_accum=True).align(src, None, default_params(**kw), chain=[(TRIM, 0.7)])["result"]
    rot, tr = pose_delta(icp.getFinalTransformation(), ref.matrix())
    assert rot < ROT_TOL and tr < TRANS_TOL, (rot, tr)
    rot, tr = pose_delta(icp.getFinalTransformation(), gt)
    assert tr < 1e-3 and rot < np.deg2rad(0.2), (rot, tr)
    batch = icp.alignBatch(np.eye(4)[None])[0]
    assert max(pose_delta(synth_matrix(batch), icp.getFinalTransformation())) < 1e-6


def test_facade_chain_and_invalid_chains(tmp_path):
    exe = tmp_path / "rejector_check"
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "cpp" / "rejector_check.cpp"), "-o", str(exe), "-L", str(ROOT / "pose_estimation_b200"),
           "-lpe_b200", f"-Wl,-rpath,{ROOT / 'pose_estimation_b200'}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "facade chain ok" in r.stdout and "invalid chains refused" in r.stdout
