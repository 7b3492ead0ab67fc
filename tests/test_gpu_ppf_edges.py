"""PPF3DDetector on the device (csrc/ppf.cu) at its edges, against the oracle (oracle/ppf_oracle.cpp).

Every raw pose (one per scene reference point: num_votes, model_index, alpha) must equal the oracle's.  The device's
acos / atan2 / sin are within 2 ulp of glibc's, so a quotient that lies within rounding of an integer may quantise
differently; a disagreement is accepted only where `Quotients.explains` finds such a quotient among the ones that decide
the reference point's votes — the feature quotients of its scene pairs, their alpha-bin quotients against the model
pairs of their bucket, and the feature quotients of the model pairs that could fall into one of those buckets.  Any other
disagreement fails.  The clustered output must be what the oracle's clusterPoses makes of the device's own raw poses.

Cases: 1 to 30+ accumulator ranges (a range is the chunk = 12288 / num_angles model points the voting kernel keeps in
shared memory at a time); a planar model at the 4095-point limit, where every pair falls into a few buckets; sampled
scenes around the 256-pair voting tile; 1 and more than 4 x 148 reference points (the vote kernel's grid-stride loop);
reference points without any vote; box faces whose normals are exactly +-x, +-y, +-z (computeTransformRT's axis branch,
acos(+-1), dot products rounding past 1)."""
import math

import numpy as np
import pytest

import oracle

EPS = 1.192092896e-07
TOL = 1e-12


# ---- float64 restatement of the quotients that decide the votes (same evaluation order as ppf_oracle.cpp) -----------
def _dot(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]


def transform_rt(p1, n1):
    angle = math.acos(n1[0])
    if n1[1] == 0.0 and n1[2] == 0.0:
        ax = np.array([0.0, 1.0, 0.0])
    else:
        ax = np.array([0.0, n1[2], -n1[1]])
        nn = math.sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2])
        if nn > EPS:
            inv = 1.0 / nn
            ax = ax * inv
    c, s = math.cos(angle), math.sin(angle)
    o = 1.0 - c
    x, y, z = ax
    R = np.array([[c + o * x * x, o * x * y - s * z, o * x * z + s * y],
                  [o * y * x + s * z, c + o * y * y, o * y * z - s * x],
                  [o * z * x - s * y, o * z * y + s * x, c + o * z * z]])
    t = -(R[:, 0] * p1[0] + R[:, 1] * p1[1] + R[:, 2] * p1[2])
    return R, t


def pair_quotients(S, i, angle_step, distance_step):
    """Feature quotients (j, 4) and alpha (j,) of the ordered pairs (i, j) of the float cloud S (n x 6)."""
    P, N = S[:, :3].astype(np.float64), S[:, 3:].astype(np.float64)
    d = P - P[i]
    f3 = np.sqrt(_dot(d, d))
    far = ~(f3 <= EPS)
    with np.errstate(invalid="ignore", divide="ignore"):
        dn = d * (1.0 / f3)[:, None]
        f0 = np.where(far, np.arccos(_dot(N[i], dn)), 0.0)
        f1 = np.where(far, np.arccos(_dot(N, dn)), 0.0)
        f2 = np.where(far, np.arccos(_dot(N[i][None], N)), 0.0)
    q = np.stack([f0 / angle_step, f1 / angle_step, f2 / angle_step, f3 / distance_step], 1)
    R, t = transform_rt(P[i], N[i])
    my = t[1] + (R[1, 0] * P[:, 0] + R[1, 1] * P[:, 1] + R[1, 2] * P[:, 2])
    mz = t[2] + (R[2, 0] * P[:, 0] + R[2, 1] * P[:, 1] + R[2, 2] * P[:, 2])
    a = np.arctan2(-mz, my)
    a = np.where(np.isnan(a), 0.0, a)
    a = np.where(np.sin(a) * mz < 0.0, -a, a)
    return q, -a


def pack(k):
    return ((k[:, 0] * 32768 + k[:, 1]) * 32768 + k[:, 2]) * 32768 + k[:, 3]


def valid_keys(q):
    ok = np.isfinite(q).all(1) & (q < 32767.0).all(1)
    k = np.zeros(q.shape, np.int64)
    k[ok] = q[ok].astype(np.int64)
    return ok, k


def near_integer(q):
    """Quotients within TOL of an integer >= 1 (below 1 a quotient of an angle or a distance cannot change bin)."""
    with np.errstate(invalid="ignore"):
        r = np.rint(q)
        return (np.abs(q - r) <= TOL * np.maximum(1.0, np.abs(q))) & (r >= 1)


class Quotients:
    """The model's table (packed key, model reference, float alpha of every ordered model pair) and the scene's quotients,
    in float64 numpy."""

    def __init__(self, model_s, scene_s, num_angles_param, distance_step, step=1):
        self.angle_step = (360.0 / num_angles_param) * math.pi / 180.0
        self.num_angles = int(math.floor(2 * math.pi / self.angle_step))
        self.distance_step = float(distance_step)
        self.model, self.scene, self.step = model_s, scene_s, step
        self._table = None

    def table(self):
        """(sorted packed keys, model references, float alphas, packed keys a model pair near a bin edge may take);
        built on first use — n^2 pairs."""
        if self._table is None:
            keys, refs, alphas, fragile = [], [], [], set()
            for i in range(len(self.model)):
                q, a = pair_quotients(self.model, i, self.angle_step, self.distance_step)
                q[i] = np.nan
                ok, k = valid_keys(q)
                keys.append(pack(k[ok]))
                refs.append(np.full(int(ok.sum()), i, np.int32))
                alphas.append(a[ok].astype(np.float32))
                # a model pair near a bin edge may sit in either bucket: both count as touched
                near = near_integer(q) & np.isfinite(q)
                for j in np.flatnonzero(near.any(1) & ok):
                    cands = [k[j]]
                    for c in np.flatnonzero(near[j]):
                        r = int(np.rint(q[j, c]))
                        cands = [x for b in cands for x in (_with(b, c, r), _with(b, c, r - 1))]
                    fragile.update(int(pack(x[None])[0]) for x in cands)
            key = np.concatenate(keys)
            order = np.argsort(key, kind="stable")  # (i, j) order inside a bucket, like the oracle's insertion order
            self._table = key[order], np.concatenate(refs)[order], np.concatenate(alphas)[order], fragile
        return self._table

    def bucket(self, k):
        key, ref, alpha, _ = self.table()
        lo, hi = np.searchsorted(key, k, "left"), np.searchsorted(key, k, "right")
        return ref[lo:hi], alpha[lo:hi]

    def scene_pairs(self, ri):
        i = ri * self.step
        q, a = pair_quotients(self.scene, i, self.angle_step, self.distance_step)
        q[i] = np.nan
        return q, a

    def alpha_quotients(self, alpha_model32, alpha_scene):
        return self.num_angles * (alpha_model32.astype(np.float64) - alpha_scene + 2 * math.pi) / (4 * math.pi)

    def votes(self, ri):
        """The accumulator of reference point ri (model reference x alpha bin)."""
        q, a = self.scene_pairs(ri)
        ok, k = valid_keys(q)
        acc = np.zeros(len(self.model) * self.num_angles, np.int64)
        for j in np.flatnonzero(ok):
            refs, am = self.bucket(pack(k[j][None])[0])
            b = np.minimum(self.alpha_quotients(am, a[j]).astype(np.int64), self.num_angles - 1)
            np.add.at(acc, refs.astype(np.int64) * self.num_angles + b, 1)
        return acc

    def explains(self, ri):
        q, a = self.scene_pairs(ri)
        if near_integer(q).any():
            return True
        ok, k = valid_keys(q)
        for j in np.flatnonzero(ok):
            kk = int(pack(k[j][None])[0])
            if kk in self.table()[3]:
                return True
            _, am = self.bucket(kk)
            if near_integer(self.alpha_quotients(am, a[j])).any():
                return True
        return False


def _with(k, c, v):
    k = k.copy()
    k[c] = v
    return k


def same_raw(a, b):
    return (a.num_votes, a.model_index) == (b.num_votes, b.model_index) and abs(a.alpha - b.alpha) < 1e-12


def check_raw(raw, oraw, quot, matrix_tol=1e-9, max_explained=0):
    """Every raw pose equals the oracle's or its disagreement is explained; agreeing poses within matrix_tol.  Explained
    disagreements are bounded as well (max_explained; none occur in the committed cases), so that a kernel fault which
    happens to hit reference points near a bin edge cannot hide behind the explanation."""
    assert len(raw) == len(oraw)
    explained, unexplained = [], []
    for ri, (a, b) in enumerate(zip(raw, oraw)):
        if same_raw(a, b):
            assert np.allclose(a.matrix, b.matrix, atol=matrix_tol, rtol=0), ri
            assert np.allclose(a.q, b.q, atol=matrix_tol, rtol=0) and abs(a.angle - b.angle) < 1e-7, ri
        else:
            d = (ri, (a.num_votes, a.model_index, a.alpha), (b.num_votes, b.model_index, b.alpha))
            (explained if quot.explains(ri) else unexplained).append(d)
    assert not unexplained, f"{len(unexplained)} of {len(raw)} reference points disagree without a quotient at a bin edge: {unexplained[:4]}"
    assert len(explained) <= max_explained, f"{len(explained)} of {len(raw)} reference points disagree at a bin edge: {explained[:4]}"


def check_clusters(res, raw, odet):
    """The device's clustering equals the oracle's clusterPoses of the device's own raw poses."""
    want = odet.cluster([oracle.PpfPose.from_buffer_copy(p) for p in raw])
    assert len(res) == len(want)
    for a, b in zip(res, want):
        assert a.num_votes == b.num_votes
        assert np.allclose(a.matrix, b.matrix, atol=1e-12, rtol=0) and np.allclose(a.q, b.q, atol=1e-12, rtol=0)


# ---- clouds with an exact number of sampled points ----------------------------------------------------------------
def exact_prefix(orc, stream, step, target):
    """The shortest prefix of `stream` that samples (samplePCByQuantization at `step`) to exactly `target` points.  The
    stream's first two rows span its bounding box, so the box is fixed and every further row adds 0 or 1 cell."""
    lo, hi = 2, len(stream)
    assert len(orc.ppf_sample(stream, step)) >= target
    while lo < hi:
        mid = (lo + hi) // 2
        if len(orc.ppf_sample(stream[:mid], step)) >= target:
            hi = mid
        else:
            lo = mid + 1
    out = np.ascontiguousarray(stream[:lo])
    assert len(orc.ppf_sample(out, step)) == target
    return out


def unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def boxed_stream(rng, pts, nrm, lo, hi):
    """Rows (x y z nx ny nz) float32: the two corners lo / hi first, then the points in random order."""
    order = rng.permutation(len(pts))
    corners = np.concatenate([np.array([lo, hi]), unit(rng, 2)], 1)
    return np.concatenate([corners, np.concatenate([pts[order], nrm[order]], 1)]).astype(np.float32)


def volume_cloud(rng, n):
    """n points filling a 0.1 m cube with random normals (buckets of every feature are populated)."""
    return rng.uniform(0.0, 0.1, (n, 3)), unit(rng, n)


def moved(pts, nrm, seed):
    rng = np.random.default_rng(seed)
    from pose_estimation_b200.testing import synth

    R = synth.rotation_about(synth.random_unit(rng), rng.uniform(0.3, 1.2))
    return pts @ R.T + np.array([0.02, -0.01, 0.03]), nrm @ R.T


# ---- CPU: the helper against the oracle ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def orc():
    return oracle.Oracle()


def test_quotients_helper_reproduces_the_oracle_votes(orc):
    rng = np.random.default_rng(1)
    mp, mn = volume_cloud(rng, 400)
    model = exact_prefix(orc, boxed_stream(rng, mp, mn, [0, 0, 0], [0.1, 0.1, 0.1]), 0.1, 150)
    det = orc.ppf_train(model, oracle.ppf_params(0.1, 0.1, 21))
    sp, sn = moved(mp, mn, 2)
    scene = np.concatenate([sp, sn], 1).astype(np.float32)
    _, oraw, ss = det.match(scene, 1.0 / 7.0, 0.1)
    quot = Quotients(det.sampled(), ss, 21, det.distance_step, step=7)
    assert len(quot.table()[0]) == det.table_size
    num_angles = quot.num_angles
    assert sum(quot.explains(ri) for ri in range(len(oraw))) <= 0.05 * len(oraw)  # it does not explain everything
    for ri in range(len(oraw)):
        acc = quot.votes(ri)
        assert oraw[ri].num_votes == acc.max()
        flat = int(acc.argmax()) if acc.max() > 0 else 0
        assert (oraw[ri].model_index, round((oraw[ri].alpha + 2 * math.pi) * num_angles / (4 * math.pi))) == divmod(flat, num_angles)
    # the near-integer test: a quotient one ulp off an integer is flagged, one 1e-6 off or below 1 is not
    assert list(near_integer(np.array([3.0, np.nextafter(3.0, 0), 3.000001, 1e-13, 0.5]))) == [True, True, False, False, False]


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pcl():
    from pose_estimation_b200 import pcl as m

    return m


def run_both(pcl, orc, model, scene, num_angles, rel_step, rss, rsd):
    det = pcl.PPF3DDetector(rel_step, rel_step, num_angles)
    det.trainModel(model)
    odet = orc.ppf_train(model, oracle.ppf_params(rel_step, rel_step, num_angles))
    assert np.array_equal(det.sampled_model().view(np.uint32), odet.sampled().view(np.uint32))
    res, raw = det.match(scene, rss, rsd, return_raw=True)
    ores, oraw, ss = odet.match(scene, rss, rsd)
    det.close()
    quot = Quotients(odet.sampled(), ss, num_angles, odet.distance_step, step=int(1.0 / rss))
    return res, raw, ores, oraw, odet, quot, ss


def chunk_of(num_angles_param):
    num_angles = int(math.floor(2 * math.pi / ((360.0 / num_angles_param) * math.pi / 180.0)))
    return 12288 // num_angles


# (num_angles, relative sampling step, sampled model points); 30+ ranges need num_angles = 120: at 40 angles 30 ranges
# would be 9 000+ points (the limit is 4095), at 360 the direct table allows only a few ranges (na^3 nd x ranges <= 2^28)
RANGES = [(40, 0.05, "one"), (40, 0.05, "chunk"), (40, 0.05, "chunk+1"),
          (120, 0.05, "one"), (120, 0.05, "chunk"), (120, 0.05, "chunk+1"), (120, 0.05, "30 ranges"),
          (360, 0.125, "one"), (360, 0.125, "chunk"), (360, 0.125, "chunk+1")]


@pytest.mark.gpu
@pytest.mark.parametrize("num_angles,rel_step,size", RANGES)
def test_vote_ranges(pcl, orc, num_angles, rel_step, size):
    chunk = chunk_of(num_angles)
    n = {"one": chunk // 2 + 3, "chunk": chunk, "chunk+1": chunk + 1, "30 ranges": 29 * chunk + 1}[size]
    rng = np.random.default_rng(n + num_angles)
    mp, mn = volume_cloud(rng, 12 * n + 200)
    model = exact_prefix(orc, boxed_stream(rng, mp, mn, [0, 0, 0], [0.1, 0.1, 0.1]), rel_step, n)
    sp, sn = moved(model[:, :3].astype(np.float64), model[:, 3:].astype(np.float64), n)
    scene = np.concatenate([sp, sn], 1).astype(np.float32)
    rss = 1.0 / max(1, n // 150)
    res, raw, ores, oraw, odet, quot, _ = run_both(pcl, orc, model, scene, num_angles, rel_step, rss, rel_step)
    assert odet.n == n and math.ceil(n / chunk) == {"one": 1, "chunk": 1, "chunk+1": 2}.get(size, 30)
    assert max(p.num_votes for p in oraw) >= 3
    check_raw(raw, oraw, quot)
    check_clusters(res, raw, odet)


def planar_grid(rows, cols, h=0.002, slope=0.05):
    """Points of a rows x cols grid on the plane z = slope x, every normal exactly +z: f0 and f1 stay within 3 degrees of
    pi / 2 (bin 7 at 31 angles) and f2 = acos(1) = 0, so only the distance separates the pairs' buckets."""
    x, y = np.meshgrid(np.arange(cols) * h, np.arange(rows) * h, indexing="xy")
    x, y = x.ravel().astype(np.float32), y.ravel().astype(np.float32)
    z = (np.float32(slope) * x).astype(np.float32)
    out = np.zeros((len(x), 6), np.float32)
    out[:, 0], out[:, 1], out[:, 2], out[:, 5] = x, y, z, 1.0
    return out


@pytest.mark.gpu
def test_planar_model_at_the_4095_point_limit(pcl, orc):
    full = planar_grid(64, 64)                 # 4096 lattice cells at a sampling step of 1 / 64
    model = np.delete(full, 64 * 30 + 17, 0)   # one interior point less: 4095
    scene = planar_grid(64, 64)[(np.arange(4096) % 64 < 14) & (np.arange(4096) // 64 < 14)]
    rel = 1.0 / 64
    # 31 angles: on a grid many pairs have the same planar angle as their scene counterpart, and a difference of 0 is
    # num_angles / 2 alpha bins — an odd num_angles keeps that off a bin edge
    res, raw, ores, oraw, odet, quot, ss = run_both(pcl, orc, model, scene, 31, rel, 1.0 / 8, 1.0 / 14)
    assert odet.n == 4095
    # nearly every model pair is in one of the ~64 distance buckets of the (7, 7, 0) feature
    assert odet.table_size == 4095 * 4094
    assert min(p.num_votes for p in oraw) > 300
    check_raw(raw, oraw, quot)
    check_clusters(res, raw, odet)
    det = pcl.PPF3DDetector(rel, rel, 31)
    try:
        with pytest.raises(pcl.PebError) as e:
            det.trainModel(full)
        assert e.value.code == -6  # PEB_E_UNSUPPORTED: 4096 sampled points
    finally:
        det.close()
    assert len(orc.ppf_sample(full, rel)) == 4096


@pytest.fixture(scope="module")
def tile_model(orc):
    rng = np.random.default_rng(21)
    mp, mn = volume_cloud(rng, 3000)
    model = exact_prefix(orc, boxed_stream(rng, mp, mn, [0, 0, 0], [0.1, 0.1, 0.1]), 0.05, 600)
    return model, mp, mn


# (sampled scene points, relative scene sample step): the 256-pair tiles of the vote kernel, one reference point, and
# more reference points than the 4 x 148 blocks of the grid
TILES = [(2, 1.0), (255, 1.0 / 3), (256, 1.0), (257, 1.0 / 300), (513, 1.0 / 2), (800, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("ms,rss", TILES)
def test_scene_tiles_and_reference_strides(pcl, orc, tile_model, ms, rss):
    model, mp, mn = tile_model
    rng = np.random.default_rng(ms)
    sp, sn = moved(mp, mn, ms)
    scene = exact_prefix(orc, boxed_stream(rng, sp, sn, sp.min(0) - 0.001, sp.max(0) + 0.001), 0.05, ms)
    res, raw, ores, oraw, odet, quot, ss = run_both(pcl, orc, model, scene, 40, 0.05, rss, 0.05)
    assert len(ss) == ms and len(raw) == (ms + int(1.0 / rss) - 1) // int(1.0 / rss)
    check_raw(raw, oraw, quot)
    check_clusters(res, raw, odet)


@pytest.mark.gpu
def test_reference_points_without_votes(pcl, orc, tile_model):
    model, mp, mn = tile_model
    # the model's cloud blown up 1000 times: every scene pair is longer than the model's diameter, no bucket exists
    scene = np.concatenate([mp * 1000.0, mn], 1).astype(np.float32)
    res, raw, ores, oraw, odet, quot, ss = run_both(pcl, orc, model, scene, 40, 0.05, 1.0 / 4, 0.05)
    assert len(raw) > 100
    for a, b in zip(raw, oraw):
        assert a.num_votes == 0 and b.num_votes == 0
        assert (a.model_index, a.alpha) == (b.model_index, b.alpha) == (0, -2 * math.pi)
        assert np.allclose(a.matrix, b.matrix, atol=1e-9, rtol=0)
    check_clusters(res, raw, odet)


def box_faces(rng, size, n):
    """n points on the faces of an axis-aligned box, normals exactly +-x, +-y, +-z."""
    size = np.asarray(size, np.float64)
    face = rng.integers(0, 6, n)
    axis, side = face // 2, face % 2
    pts = rng.uniform(0, 1, (n, 3)) * size
    pts[np.arange(n), axis] = side * size[axis]
    nrm = np.zeros((n, 3))
    nrm[np.arange(n), axis] = np.where(side == 1, 1.0, -1.0)
    return np.concatenate([pts, nrm], 1).astype(np.float32)


@pytest.mark.gpu
def test_axis_aligned_normals(pcl, orc):
    rng = np.random.default_rng(31)
    model = box_faces(rng, [0.1, 0.07, 0.05], 6000)
    # the box turned by 90 degrees about z and moved: (x, y, z) -> (-y, x, z), normals stay exact axis vectors
    sc = box_faces(rng, [0.1, 0.07, 0.05], 5000)
    scene = np.stack([-sc[:, 1], sc[:, 0], sc[:, 2], -sc[:, 4], sc[:, 3], sc[:, 5]], 1) + np.float32([0.3, 0.1, 0.5, 0, 0, 0])
    scene = scene.astype(np.float32)
    # 31 angles: pi / 2 and pi are 7.75 and 15.5 bins, away from the bin edges
    res, raw, ores, oraw, odet, quot, ss = run_both(pcl, orc, model, scene, 31, 0.05, 1.0 / 2, 0.05)
    # the n1.y == 0 && n1.z == 0 branch is taken for model points and scene reference points whose normal is exactly
    # -x: there acos(-1) = pi and the axis decides the frame (for +x the angle is 0 and R = I either way)
    minus_x = np.array([-1.0, 0.0, 0.0], np.float32)
    assert (odet.sampled()[:, 3:] == minus_x).all(1).sum() > 20
    assert (ss[::2][:, 3:] == minus_x).all(1).sum() > 20  # (every second sampled scene point is a reference point)
    assert max(p.num_votes for p in oraw) >= 20
    check_raw(raw, oraw, quot)
    check_clusters(res, raw, odet)
