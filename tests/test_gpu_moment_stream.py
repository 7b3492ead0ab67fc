"""The batched moment launch (pose_estimation_b200/csrc/icp.cu : icp_moment_kernel) streams each block's chunks of the
working clouds through a ring of kMomentRing (4) shared-memory slots of 128 points with bulk copies, and adds them in the
same order as the fused iteration kernel (`split_moments` 0): the records must be byte-identical.

The ring's edges come from the source size and the blocks per hypothesis: with 37 hypotheses and blocks_factor 1 every
hypothesis has 4 moment blocks (ceil(148 / 37)), so a block adds ceil((n - 128 blk) / 512) passes of 128 queries; with
150 hypotheses it has one block and n / 128 passes.  The sizes below give blocks with 1, 2, 3, 4, 5 and 6 passes (fewer
than, as many as and more than the ring's slots), a clipped last chunk (n not a multiple of 128) and blocks one query past
a full pass.  (Every moment block has at least one pass: the host never gives a hypothesis more blocks than 128-point
chunks.)  Hypotheses that stop at different iterations and ones without a correspondence at iteration 0 leave moment
blocks that return before any copy; non-finite points and guesses take the -2 - j slot path.  The rejector-chain instance
(CHAIN) is checked against records of the same chains written by the library before the ring
(tests/golden/moment_chain.npz, `python tests/test_gpu_moment_stream.py --write-golden PATH`).
"""
import sys
from pathlib import Path

import numpy as np
import pytest

from pose_estimation_b200.testing import synth

pytestmark = [pytest.mark.gpu]

INTERNAL_ERROR = -1000  # PEB_STATE_INTERNAL_ERROR
GOLDEN = Path(__file__).resolve().parent / "golden" / "moment_chain.npz"
MED, O2O = 1, 2  # PEB_REJECTOR_MEDIAN_DISTANCE, PEB_REJECTOR_ONE_TO_ONE
CHAINS = {"median": [(MED, 1.5)], "one_to_one_median": [(O2O,), (MED, 2.0)]}
CHAIN_SIZES = (129, 2561)
KW = dict(max_iterations=12, max_corr_dist=0.02, abs_mse_threshold=-1.0)


@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as m

    return m


def make_scene(oracle):
    return synth.make_c2(scale=0.25, downsample=lambda p, leaf: oracle.voxel_grid(p, leaf)[0])


@pytest.fixture(scope="module")
def scene(oracle):
    return make_scene(oracle)  # 3125 source points


@pytest.fixture(scope="module")
def target_normals(pcl, scene):
    with pcl.Context(0) as c:
        ne = pcl.NormalEstimation(c)
        ne.setInputCloud(scene.target)
        ne.setKSearch(12)
        return ne.compute()


def _guesses(p, seed, n, deg=5.0, m=0.006):
    rng = np.random.default_rng(seed)
    return np.stack([synth.perturb_pose(p.gt_pose, rng, deg, m) for _ in range(n)])


def _run(pcl, source, target, guesses, split, opts=(), cls=None, normals=None, chain=(), **params):
    from oracle import default_params

    with pcl.Context(0) as c:
        c.set_int("split_moments", split)
        c.set_int("split_min_hyp", 2)  # (split every batch here; by default batches below 256 hypotheses stay fused)
        c.set_int("blocks_factor", 1)
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
            if r[0] == MED:
                icp.addCorrespondenceRejectorMedianDistance(r[1])
            else:
                icp.addCorrespondenceRejectorOneToOne()
        res = icp.alignBatch(guesses)
    assert all(r.state != INTERNAL_ERROR for r in res)
    return [bytes(r) for r in res]


def _same(pcl, source, target, guesses, opts=(), **kw):
    a = _run(pcl, source, target, guesses, 0, opts, **kw)
    b = _run(pcl, source, target, guesses, 1, opts, **kw)
    assert a == b
    return a


@pytest.mark.parametrize("H,n", [(37, 1), (37, 127), (37, 128), (37, 129), (37, 511), (37, 513), (37, 1536), (37, 2048),
                                 (37, 2560), (37, 2561), (37, 3125), (150, 384), (150, 512), (150, 640), (150, 1025)])
def test_ring_edges(pcl, scene, H, n):
    p = scene
    a = _same(pcl, p.source[:n], p.target, _guesses(p, 40 + n, H), **KW)
    if n >= 128:
        assert len({r[:64] for r in a}) > 1  # (the transforms differ between hypotheses: the comparison is not vacuous)


@pytest.mark.parametrize("deps", [1, 0])
def test_hypotheses_that_stop_early_or_find_nothing(pcl, scene, deps):
    from pose_estimation_b200 import _lib

    p = scene
    rng = np.random.default_rng(41)
    guesses = [synth.perturb_pose(p.gt_pose, rng, a, t) for a, t in [(0.2, 0.0003)] * 12 + [(2.0, 0.003)] * 12 + [(6.0, 0.008)] * 9]
    far = np.array(p.gt_pose, np.float64)
    far[:3, 3] += [0.5, 0.5, 0.5]  # no correspondence at iteration 0
    guesses = np.stack(guesses + [far] * 4)
    a = _same(pcl, p.source[:2561], p.target, guesses, (("flag_deps", deps),), max_iterations=40, max_corr_dist=0.01,
              transformation_epsilon=1e-7)
    res = [_lib.IcpResult.from_buffer_copy(r) for r in a]
    its = np.array([r.iterations for r in res])
    assert len(set(its[:33].tolist())) > 1 and all(r.state == 5 for r in res[33:])


def test_nonfinite_points_and_guesses(pcl, scene):
    p = scene
    rng = np.random.default_rng(42)
    src = p.source[:2561].copy()
    src[rng.choice(len(src), 200, replace=False), rng.integers(0, 3, 200)] = np.nan
    src[rng.choice(len(src), 40, replace=False), 0] = np.inf
    guesses = _guesses(p, 43, 37)
    guesses[5, 0, 3] = np.nan  # every point of the hypothesis turns non-finite: its matches travel as -2 - j
    guesses[6, 1, 3] = np.inf
    guesses[7, 0, 0] = np.nan
    _same(pcl, src, p.target, guesses, **KW)


@pytest.mark.parametrize("n", [129, 2561])
def test_point_to_plane_with_rejector(pcl, scene, target_normals, n):
    p = scene
    a = _same(pcl, p.source[:n], p.target, _guesses(p, 44, 37, 4.0, 0.004), cls=pcl.IterativeClosestPointWithNormals,
              normals=target_normals, max_iterations=20, max_corr_dist=0.01, transformation_epsilon=1e-9,
              rejector_max_dist=0.008)
    assert len({r[-32:] for r in a}) > 1


@pytest.mark.parametrize("deps,streams", [(1, 1), (1, 4), (0, 1), (0, 4)])
def test_scheduling(pcl, scene, deps, streams):
    p = scene
    _same(pcl, p.source[:2561], p.target, _guesses(p, 45, 37), (("flag_deps", deps), ("batch_streams", streams)), **KW)


def chain_records(pcl, p, normals):
    """{case: uint8 records} of the rejector chains (every iteration runs the CHAIN moment instance) at two ring sizes"""
    out = {}
    for name, chain in CHAINS.items():
        for n in CHAIN_SIZES:
            g = _guesses(p, 46, 37, 4.0, 0.004)
            out[f"svd_{name}_{n}"] = _run(pcl, p.source[:n], p.target, g, 1, chain=chain, max_iterations=15,
                                          max_corr_dist=0.01, transformation_epsilon=1e-9)
            out[f"lls_{name}_{n}"] = _run(pcl, p.source[:n], p.target, g, 1, chain=chain,
                                          cls=pcl.IterativeClosestPointWithNormals, normals=normals, max_iterations=15,
                                          max_corr_dist=0.01, transformation_epsilon=1e-9)
    return {k: np.frombuffer(b"".join(v), np.uint8) for k, v in out.items()}


def test_rejector_chains_match_the_records_before_the_ring(pcl, scene, target_normals):
    golden = np.load(GOLDEN)
    got = chain_records(pcl, scene, target_normals)
    assert sorted(got) == sorted(golden.files)
    for k, v in got.items():
        assert np.array_equal(v, golden[k]), k


if __name__ == "__main__":
    # --write-golden PATH: the chain records of the library this process loads
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    from oracle import Oracle
    from pose_estimation_b200 import pcl as _pcl

    assert sys.argv[1] == "--write-golden"
    sc = make_scene(Oracle())
    with _pcl.Context(0) as c:
        ne = _pcl.NormalEstimation(c)
        ne.setInputCloud(sc.target)
        ne.setKSearch(12)
        nrm = ne.compute()
    np.savez(sys.argv[2], **chain_records(_pcl, sc, nrm))
