"""Batched ICP iterations split into a search launch and a moment launch (pose_estimation_b200/csrc/icp.cu :
icp_search_kernel, icp_moment_kernel; `split_moments`, default 1) against the fused iteration kernel (`split_moments` 0).

The moment launch recomputes every correspondence's squared distance from the working point and its match with the
expression every search path uses, and adds the moments with the fused kernel's blocks and query-to-thread mapping, so
the records must be byte-identical: both estimators, with and without per-hypothesis launch dependencies, one or several
chains of launches, hypotheses that stop at different iterations, non-finite points and guesses, sources shorter than a
block, and search launches whose block count differs from the moment launch's.  No record may report an internal error
(a per-hypothesis dependency wait that ran into its bound).
"""
import numpy as np
import pytest

from pose_estimation_b200.testing import synth

pytestmark = [pytest.mark.gpu]

INTERNAL_ERROR = -1000  # PEB_STATE_INTERNAL_ERROR


@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as m

    return m


@pytest.fixture(scope="module")
def scene_small(oracle):
    return synth.make_c2(scale=0.25, downsample=lambda p, leaf: oracle.voxel_grid(p, leaf)[0])


@pytest.fixture(scope="module")
def target_normals(pcl, scene_small):
    c = pcl.Context(0)
    ne = pcl.NormalEstimation(c)
    ne.setInputCloud(scene_small.target)
    ne.setKSearch(12)
    normals = ne.compute()
    c.close()
    return normals


def _run(pcl, source, target, guesses, split, opts=(), cls=None, normals=None, **params):
    from oracle import default_params

    c = pcl.Context(0)
    c.set_int("split_moments", split)
    c.set_int("split_min_hyp", 2)  # (split every batch here; by default batches below 256 hypotheses stay fused)
    for k, v in opts:
        c.set_int(k, v)
    icp = (cls or pcl.IterativeClosestPoint)(c)
    icp.setInputSource(source)
    icp.setInputTarget(target, normals)
    prm = default_params(**params)
    for name, _ in prm._fields_:
        if name != "estimator":
            setattr(icp.params, name, getattr(prm, name))
    res = icp.alignBatch(guesses)
    c.close()
    assert all(r.state != INTERNAL_ERROR for r in res)
    return [bytes(r) for r in res]


def _same(pcl, source, target, guesses, opts=(), **kw):
    a = _run(pcl, source, target, guesses, 0, opts, **kw)
    b = _run(pcl, source, target, guesses, 1, opts, **kw)
    assert a == b
    return a


def _guesses(p, seed, n, deg=5.0, m=0.006):
    rng = np.random.default_rng(seed)
    return np.stack([synth.perturb_pose(p.gt_pose, rng, deg, m) for _ in range(n)])


@pytest.mark.parametrize("deps,streams", [(1, 1), (1, 4), (0, 1), (0, 4)])
def test_split_point_to_point_dependencies_and_chains(pcl, scene_small, deps, streams):
    p = scene_small
    guesses = _guesses(p, 21, 200)
    a = _same(pcl, p.source, p.target, guesses, (("flag_deps", deps), ("batch_streams", streams)),
              max_iterations=25, max_corr_dist=0.02, abs_mse_threshold=-1.0)
    assert len({r[:64] for r in a}) > 1  # (the transforms differ between hypotheses: the comparison is not vacuous)


@pytest.mark.parametrize("H", [16, 32, 33])
def test_split_small_batches(pcl, scene_small, H):
    # 16: plain warm launches (below the k-NN graph's batch size), 32 / 33: over the graph, an odd share per chain
    p = scene_small
    _same(pcl, p.source, p.target, _guesses(p, 22, H), max_iterations=20, max_corr_dist=0.02, abs_mse_threshold=-1.0)


def test_split_per_launch_profile(pcl, scene_small):
    # profile level 2: one chain, whole-grid dependencies, both launches of an iteration between the same events
    p = scene_small
    _same(pcl, p.source, p.target, _guesses(p, 23, 64), (("profile", 2),), max_iterations=15, max_corr_dist=0.02,
          abs_mse_threshold=-1.0)


def test_split_point_to_plane_with_rejector(pcl, scene_small, target_normals):
    p = scene_small
    a = _same(pcl, p.source, p.target, _guesses(p, 24, 40, 4.0, 0.004), cls=pcl.IterativeClosestPointWithNormals,
              normals=target_normals, max_iterations=30, max_corr_dist=0.01, transformation_epsilon=1e-9,
              rejector_max_dist=0.008)
    assert len({r[-32:] for r in a}) > 1


def test_split_hypotheses_that_stop_at_different_iterations(pcl, scene_small):
    p = scene_small
    rng = np.random.default_rng(25)
    guesses = [synth.perturb_pose(p.gt_pose, rng, a, t) for a, t in [(0.2, 0.0003)] * 24 + [(2.0, 0.003)] * 24 + [(6.0, 0.008)] * 24]
    far = np.array(p.gt_pose, np.float64)
    far[:3, 3] += [0.5, 0.5, 0.5]  # no correspondence at iteration 0
    guesses = np.stack(guesses + [far] * 8)
    from pose_estimation_b200 import _lib

    kw = dict(max_iterations=40, max_corr_dist=0.01, transformation_epsilon=1e-9)
    # an absolute MSE threshold (on the change of the MSE between iterations, as in PCL) at a tenth of the median final MSE
    free = [_lib.IcpResult.from_buffer_copy(r) for r in _run(pcl, p.source, p.target, guesses, 0, abs_mse_threshold=-1.0, **kw)]
    thr = 0.1 * float(np.median([r.last_mse for r in free[:72]]))
    for deps in (1, 0):
        a = _same(pcl, p.source, p.target, guesses, (("flag_deps", deps),), abs_mse_threshold=thr, **kw)
    res = [_lib.IcpResult.from_buffer_copy(r) for r in a]
    its = np.array([r.iterations for r in res])
    states = np.array([r.state for r in res])
    assert len(set(its[:72].tolist())) > 1 and (states[72:] == 5).all()
    assert (states[:72] == 3).any()  # (the MSE threshold did fire)


def test_split_nonfinite_points_guesses_and_tiny_sources(pcl, scene_small):
    p = scene_small
    rng = np.random.default_rng(26)
    src = p.source.copy()
    src[rng.choice(len(src), 300, replace=False), rng.integers(0, 3, 300)] = np.nan
    src[rng.choice(len(src), 50, replace=False), 0] = np.inf
    guesses = _guesses(p, 27, 48)
    guesses[5, 0, 3] = np.nan  # non-finite guesses: every point of the hypothesis turns non-finite
    guesses[6, 1, 3] = np.inf
    guesses[7, 0, 0] = np.nan
    kw = dict(max_iterations=12, max_corr_dist=0.02, abs_mse_threshold=-1.0)
    _same(pcl, src, p.target, guesses, **kw)
    for n in (1, 31, 129, 700):  # less than a warp, a block, a few blocks
        _same(pcl, p.source[:n], p.target, guesses[:20], **kw)


@pytest.mark.parametrize("opts", [(("blocks_factor_search", 4),), (("blocks_factor_search", 96),),
                                  (("blocks_factor_search", 8), ("blocks_factor", 64), ("blocks_factor_cold", 8)),
                                  (("blocks_factor_search", 64), ("blocks_factor", 4))])
def test_split_search_and_moment_launches_with_different_block_counts(pcl, scene_small, opts):
    # the search launch's blocks are free (it writes no records); the moment launch's follow blocks_factor(_cold) as the
    # fused kernel's do
    p = scene_small
    _same(pcl, p.source, p.target, _guesses(p, 28, 200), opts, max_iterations=20, max_corr_dist=0.02,
          abs_mse_threshold=-1.0)


def test_split_applies_from_split_min_hyp_on(pcl, scene_small):
    # a split iteration is two launches: by default batches of 256 hypotheses and more split, smaller ones stay fused
    from oracle import default_params

    p = scene_small
    iters = 6
    extra = {}
    for H in (128, 256):
        counts = []
        for split in (0, 1):
            c = pcl.Context(0)
            c.set_int("split_moments", split)
            c.set_int("batch_streams", 1)
            icp = pcl.IterativeClosestPoint(c)
            icp.setInputSource(p.source)
            icp.setInputTarget(p.target)
            prm = default_params(max_iterations=iters, max_corr_dist=0.02, abs_mse_threshold=-1.0)
            for name, _ in prm._fields_:
                if name != "estimator":
                    setattr(icp.params, name, getattr(prm, name))
            icp.alignBatch(_guesses(p, 29, H))  # (the first call also builds the target's graph)
            n0 = c.launch_count
            icp.alignBatch(_guesses(p, 29, H))
            counts.append(c.launch_count - n0)
            c.close()
        extra[H] = counts[1] - counts[0]
    assert extra == {128: 0, 256: iters}
