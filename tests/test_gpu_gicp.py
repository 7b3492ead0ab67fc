"""GeneralizedIterativeClosestPoint on the B200 (peb_gicp_align / peb_gicp_align_batch / peb_gicp_covariances) against the
CPU oracle (tests/gicp_oracle.cpp), batches against single aligns record for record, and the edges the header defines.
The C2-shaped case (12 500 source points) runs the BFGS on clusters of two blocks, the C1 case on one."""
import numpy as np
import pytest

import gicp_oracle as GO
from pose_estimation_b200.testing import synth

pytestmark = pytest.mark.gpu
STATE_NO_CORR = 5


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
    return synth.make_c1(3000, seed=11)


@pytest.fixture(scope="module")
def c2(pcl, ctx):
    def downsample(points, leaf):
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    prob = synth.make_c2(scale=0.5, downsample=downsample)
    assert len(prob.source) > 8192  # more than one block per cluster
    return prob


def _gicp(pcl, ctx, prob, max_corr_dist=0.05, **kw):
    g = pcl.GeneralizedIterativeClosestPoint(ctx)
    g.setInputSource(prob.source)
    g.setInputTarget(prob.target)
    g.setMaxCorrespondenceDistance(max_corr_dist)
    for name, v in kw.items():
        getattr(g, name)(v)
    return g


@pytest.mark.parametrize("case", ["c1", "c2"])
def test_covariances_match_the_oracle(pcl, ctx, case, request):
    prob = request.getfixturevalue(case)
    g = _gicp(pcl, ctx, prob)
    for which, cloud in (("source", prob.source), ("target", prob.target)):
        got = g.covariances(which).reshape(-1, 9)
        want = GO.covariances(cloud, 20).reshape(-1, 9)
        # svd3 (reciprocal square roots) against Eigen's JacobiSVD (divisions): last bits; rows whose neighbour list differs
        # (equidistant neighbours, FLANN's visiting order) may differ more
        ok = np.abs(got - want).max(1) <= 1e-12
        assert ok.mean() >= 0.999, (which, ok.mean())


@pytest.mark.parametrize("case,corr", [("c1", 0.05), ("c2", 0.02)])
def test_single_align_matches_the_oracle(pcl, ctx, case, corr, request):
    prob = request.getfixturevalue(case)
    rng = np.random.default_rng(3)
    g = _gicp(pcl, ctx, prob, max_corr_dist=corr)
    base = prob.gt_pose if prob.gt_pose is not None else np.eye(4)
    for _ in range(3):
        guess = synth.perturb_pose(base, rng, 1.0, 0.002)
        g.align(guess)
        ref = GO.align(prob.source, prob.target, guess, GO.params(max_corr_dist=corr))
        rot, tr = synth.pose_error(g.getFinalTransformation().astype(np.float64), GO.matrix(ref).astype(np.float64))
        # the device sums the pairs as a tree (the oracle in index order) and its cosf / atan2f differ from glibc's in the
        # last ulps; both change the float transforms' last bits
        assert rot < 5e-5 and tr < 5e-5, (rot, tr)
        assert (g.result.state, g.nr_iterations_, g.hasConverged()) == (ref.state, ref.iterations, bool(ref.converged))
        assert abs(g.result.n_correspondences - ref.n_correspondences) <= 1e-4 * ref.n_correspondences
        assert abs(g.getFitnessScore() - ref.fitness) <= 1e-6 * ref.fitness
        assert abs(g.result.last_mse - ref.last_mse) <= 1e-4 * ref.last_mse


def test_batch_records_equal_single_aligns(pcl, ctx, c2):
    rng = np.random.default_rng(5)
    base = c2.gt_pose if c2.gt_pose is not None else np.eye(4)
    guesses = np.stack([synth.perturb_pose(base, rng, 2.0, 0.003) for _ in range(256)])
    g = _gicp(pcl, ctx, c2, max_corr_dist=0.02)
    singles = []
    for h in range(256):
        g.align(guesses[h], want_output=False)
        singles.append(bytes(g.result))
    for H in (1, 7, 64, 256):
        batch = g.alignBatch(guesses[:H])
        assert [bytes(r) for r in batch] == singles[:H], H
    assert [bytes(r) for r in g.alignBatch(guesses)] == singles


def test_edges(pcl, c1):
    with pcl.Context(0) as c:
        g = pcl.GeneralizedIterativeClosestPoint(c)
        with pytest.raises(pcl.PebError):
            g.align()  # no target, no source
        g.setInputTarget(c1.target)
        with pytest.raises(pcl.PebError):
            g.align()  # no source
        g.setInputSource(c1.source)
        for k in (0, len(c1.source) + 1):
            g.setCorrespondenceRandomness(k)
            with pytest.raises(pcl.PebError):
                g.align()
        g.setCorrespondenceRandomness(193)
        with pytest.raises(pcl.PebError) as e:
            g.align()
        assert e.value.code == -6
        g.setCorrespondenceRandomness(20)
        g.setMaxCorrespondenceDistance(0.0)
        g.align()
        assert g.result.state == STATE_NO_CORR and not g.hasConverged() and g.result.n_correspondences == 0
        g.setMaxCorrespondenceDistance(0.05)
        g.setMaximumIterations(1)
        g.align()
        assert g.nr_iterations_ == 1 and g.hasConverged()
        assert g.alignBatch(np.zeros((0, 4, 4))) == []


def test_fewer_than_four_pairs_end_the_align(pcl):
    # PCL's estimator throws NotEnoughPointsException below 4 pairs: the align ends there, unconverged
    tgt = np.zeros((30, 4), np.float32)
    tgt[:, 0] = np.arange(30) * 0.01
    tgt[:, 1] = (np.arange(30) % 5) * 0.01
    tgt[:, 3] = 1
    for m in (1, 2, 3):
        src = tgt.copy()
        src[m:, 2] = 1.0  # all but the first m points a metre away
        with pcl.Context(0) as c:
            g = pcl.GeneralizedIterativeClosestPoint(c)
            g.setInputSource(src)
            g.setInputTarget(tgt)
            g.setMaxCorrespondenceDistance(0.005)
            g.align()
            assert (g.result.state, g.result.n_correspondences, g.nr_iterations_, g.hasConverged()) == (STATE_NO_CORR, m, 0, False)
            ref = GO.align(src, tgt, None, GO.params(max_corr_dist=0.005))
            assert (ref.state, ref.n_correspondences, ref.iterations) == (STATE_NO_CORR, m, 0)


def test_non_finite_points_change_nothing(pcl, ctx, c1):
    a = _gicp(pcl, ctx, c1)
    a.align()
    rec = bytes(a.result)
    nan = np.full((5, 4), np.nan, np.float32)
    src = np.concatenate([c1.source[:100], nan, c1.source[100:]])
    tgt = np.concatenate([c1.target[:700], nan, c1.target[700:], nan])
    b = pcl.GeneralizedIterativeClosestPoint(ctx)
    b.setInputSource(src)
    b.setInputTarget(tgt)
    b.setMaxCorrespondenceDistance(0.05)
    b.align()
    assert bytes(b.result) == rec


def test_icp_after_gicp_is_unchanged(pcl, c1):
    def icp_records(run_gicp_first):
        with pcl.Context(0) as c:
            if run_gicp_first:
                _gicp(pcl, c, c1).align()
            icp = pcl.IterativeClosestPoint(c)
            icp.setInputSource(c1.source)
            icp.setInputTarget(c1.target)
            icp.setMaximumIterations(20)
            icp.align()
            return bytes(icp.result)

    assert icp_records(True) == icp_records(False)


def test_new_target_recomputes_covariances(pcl, ctx, c1):
    g = _gicp(pcl, ctx, c1)
    before = g.covariances("target")
    moved = c1.target.copy()
    moved[:, 0] *= 2.0
    g.setInputTarget(moved)
    after = g.covariances("target")
    assert np.allclose(after, GO.covariances(moved, 20), atol=1e-9) and not np.allclose(before, after)
