"""The search launch of a split batched iteration over the target's k-NN graph (pose_estimation_b200/csrc/icp.cu :
icp_search_graph_queued) against the fused iteration kernel (`split_moments` 0).

In the split search every warp queues the queries the graph cannot prove and walks the grid for them 32 at a time, with
the moved point and the graph's best candidate kept in the queue.  The searches are exact and every working point is
written once with the bytes of the per-lane search, so the records must be byte-identical to the fused kernel's: both
estimators, with and without the flatness certificate, peeking or not, one chain without per-hypothesis dependencies,
few and many search blocks, sources shorter than a warp, tiny and degenerate targets, non-finite points and guesses,
far hypotheses that search cold, hypotheses stopped by an MSE threshold, the distance rejector and a rejector chain.
`split_min_hyp` and `warm_graph_min_hyp` are 2 so that small batches take the split path and search over the graph.
"""
import numpy as np
import pytest

from pose_estimation_b200.testing import synth

pytestmark = [pytest.mark.gpu]

INTERNAL_ERROR = -1000  # PEB_STATE_INTERNAL_ERROR
GRAPH = (("split_min_hyp", 2), ("warm_graph", 1), ("warm_graph_min_hyp", 2))
# every hypothesis over the graph from launch 1 on / only once its MSE says the certificate will hold
ALWAYS = GRAPH + (("warm_graph_kappa_x100", 0),)


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


def _run(pcl, source, target, guesses, opts, cls=None, normals=None, chain=(), **params):
    from oracle import default_params

    c = pcl.Context(0)
    for k, v in opts:
        c.set_int(k, v)
    icp = (cls or pcl.IterativeClosestPoint)(c)
    icp.setInputSource(source)
    icp.setInputTarget(target, normals)
    prm = default_params(**params)
    for name, _ in prm._fields_:
        if name != "estimator":
            setattr(icp.params, name, getattr(prm, name))
    for r in chain:
        getattr(icp, r[0])(*r[1:])
    res = icp.alignBatch(guesses)
    c.close()
    assert all(r.state != INTERNAL_ERROR for r in res)
    return [bytes(r) for r in res]


def _same(pcl, source, target, guesses, opts=ALWAYS, **kw):
    a = _run(pcl, source, target, guesses, opts + (("split_moments", 0),), **kw)
    b = _run(pcl, source, target, guesses, opts, **kw)
    assert a == b
    return a


def _guesses(p, seed, n, deg=5.0, m=0.006):
    rng = np.random.default_rng(seed)
    return np.stack([synth.perturb_pose(p.gt_pose, rng, deg, m) for _ in range(n)])


KW = dict(max_iterations=25, max_corr_dist=0.02, abs_mse_threshold=-1.0)
FLAT_ALL = (("warm_graph_flat", 1), ("warm_graph_flat_from", 1), ("warm_graph_flat_until", 1000))


@pytest.mark.parametrize("opts", [ALWAYS, GRAPH, ALWAYS + (("warm_graph_flat", 0),), ALWAYS + FLAT_ALL,
                                  ALWAYS + (("warm_graph_peek", 0),), ALWAYS + (("warm_graph_peek", 1000),),
                                  ALWAYS + FLAT_ALL + (("warm_graph_peek", 1000),),
                                  ALWAYS + (("batch_streams", 1), ("flag_deps", 0)),
                                  ALWAYS + (("blocks_factor_search", 4),), ALWAYS + (("blocks_factor_search", 96),)])
def test_queued_search_point_to_point(pcl, scene_small, opts):
    p = scene_small
    a = _same(pcl, p.source, p.target, _guesses(p, 41, 200), opts, **KW)
    assert len({r[:64] for r in a}) > 1  # (the transforms differ between hypotheses: the comparison is not vacuous)


@pytest.mark.parametrize("opts", [ALWAYS, GRAPH + FLAT_ALL])
def test_queued_search_point_to_plane_with_rejector(pcl, scene_small, target_normals, opts):
    p = scene_small
    a = _same(pcl, p.source, p.target, _guesses(p, 42, 40, 4.0, 0.004), opts, cls=pcl.IterativeClosestPointWithNormals,
              normals=target_normals, max_iterations=30, max_corr_dist=0.01, transformation_epsilon=1e-9,
              rejector_max_dist=0.008)
    assert len({r[-32:] for r in a}) > 1


def test_queued_search_nonfinite_far_tiny_sources_and_targets(pcl, scene_small):
    p = scene_small
    rng = np.random.default_rng(43)
    src = p.source.copy()
    src[rng.choice(len(src), 300, replace=False), rng.integers(0, 3, 300)] = np.nan
    src[rng.choice(len(src), 50, replace=False), 0] = np.inf
    guesses = _guesses(p, 44, 48)
    guesses[1::3, :3, 3] += (0.03 + 0.05 * rng.random((16, 1))) * np.array([1.0, -1.0, 0.5])  # far: cold searches
    # non-finite guesses: launch 0 stores -2 - j for every point of the hypothesis, and the queued search of launch 1
    # resets each such slot to -1
    guesses[5, 0, 3] = np.nan
    guesses[6, 1, 3] = np.inf
    guesses[8, 0, 0] = np.nan
    kw = dict(max_iterations=12, max_corr_dist=0.02, abs_mse_threshold=-1.0)
    for opts in (ALWAYS, ALWAYS + FLAT_ALL):
        _same(pcl, src, p.target, guesses, opts, **kw)
    # targets smaller than a row of the graph, and a target that is one point repeated
    for tgt in (p.target[:1], p.target[:7], p.target[:16], np.repeat(p.target[:1], 40, 0)):
        _same(pcl, src[:400], tgt, guesses, **kw)
    for n in (1, 31, 129, 700):  # less than a warp, a block, a few blocks
        _same(pcl, p.source[:n], p.target, guesses[:20], **kw)


def test_queued_search_hypotheses_stopped_by_mse_threshold(pcl, scene_small):
    p = scene_small
    rng = np.random.default_rng(45)
    guesses = np.stack([synth.perturb_pose(p.gt_pose, rng, a, t) for a, t in [(0.2, 0.0003)] * 24 + [(2.0, 0.003)] * 24 + [(6.0, 0.008)] * 24])
    from pose_estimation_b200 import _lib

    kw = dict(max_iterations=40, max_corr_dist=0.01, transformation_epsilon=1e-9)
    free = [_lib.IcpResult.from_buffer_copy(r) for r in _run(pcl, p.source, p.target, guesses, ALWAYS, abs_mse_threshold=-1.0, **kw)]
    thr = 0.1 * float(np.median([r.last_mse for r in free]))
    res = [_lib.IcpResult.from_buffer_copy(r) for r in _same(pcl, p.source, p.target, guesses, abs_mse_threshold=thr, **kw)]
    assert len({r.iterations for r in res}) > 1 and any(r.state == 3 for r in res)  # (the MSE threshold did fire)


def test_queued_search_rejector_chain(pcl, scene_small):
    # an align with a chain runs every iteration split (search, reject, moment launches), so the reference is the same
    # batch searching without the graph: the per-lane grid search, exact as well
    p = scene_small
    chain = [("addCorrespondenceRejectorDistance", 0.006), ("addCorrespondenceRejectorOneToOne",),
             ("addCorrespondenceRejectorMedianDistance", 1.5), ("addCorrespondenceRejectorTrimmed", 0.9)]
    guesses = _guesses(p, 46, 64, 2.0, 0.003)
    kw = dict(max_iterations=40, transformation_epsilon=1e-9, max_corr_dist=0.01, chain=chain)
    for opts in (ALWAYS, ALWAYS + FLAT_ALL):
        a = _run(pcl, p.source, p.target, guesses, opts, **kw)
        b = _run(pcl, p.source, p.target, guesses, (("warm_graph", 0),), **kw)
        assert a == b
    assert len({r[:64] for r in a}) > 1


def test_queued_search_default_thresholds(pcl, scene_small):
    # 256 hypotheses: split and over the graph with the library's defaults
    p = scene_small
    _same(pcl, p.source, p.target, _guesses(p, 47, 256), (), **KW)
