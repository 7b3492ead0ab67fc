"""block_select_nth (csrc/block_select.cuh), the exact order statistic behind the cv ICP's median / MAD threshold and the
median-distance and trimmed rejectors of the PCL ICP, through the development entry point peb_debug_select_nth (one
1024-thread block per rank).

The reference is exact: the value of rank nth is the nth entry of the values sorted by their uint32 bit pattern (for
non-negative floats that is their numeric order), compared bit for bit.  With SKIP_NEG every value whose sign bit is set
is left out first — -0.0f included, by design: a caller marks an entry as not taken by writing a negative value, and
-0.0f has the sign bit.  The precondition nth < (number of values taken) is checked by the entry point before any
launch; inside the kernel a rank outside would read a bin state that no pass wrote.

The distributions aim at where a three-pass radix select (11 + 11 + 10 bits) goes wrong: every value in one bin, ranks
on the edges between bins, values that only the third pass separates, values that share the first pass's bin, denormals,
+inf, a spread over every exponent and the squared nearest-neighbour distances the ICP actually selects over; m below,
at and above the block's 1024 threads."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 31, 32, 33, 1023, 1024, 1025, 2049, 50000, 200000]


@pytest.fixture(scope="module")
def dev():
    from pose_estimation_b200 import pcl
    from pose_estimation_b200.pcl import lib

    lib.peb_debug_select_nth.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    ctx = pcl.Context(0)
    yield ctx, lib, pcl
    ctx.close()


@pytest.fixture(scope="module")
def c1_d2():
    """Squared nearest-neighbour distances of the C1 clouds (source onto target), float32 like the ICP's."""
    from scipy.spatial import cKDTree

    from pose_estimation_b200.testing import synth

    prob = synth.make_c1(20000, seed=1)
    d, _ = cKDTree(prob.target[:, :3].astype(np.float64)).query(prob.source[:, :3].astype(np.float64))
    return (d * d).astype(np.float32)


def _bits(u):
    return np.asarray(u, np.uint32).view(np.float32)


def _values(kind, m, rng, c1_d2):
    if kind == "all_equal":
        return np.full(m, 0.37, np.float32)
    if kind == "all_plus_zero":
        return np.zeros(m, np.float32)
    if kind == "two_values":
        return np.where(rng.random(m) < 0.3, np.float32(2.5e-5), np.float32(7.0)).astype(np.float32)
    if kind == "low10":       # one bin in the first two passes: the third (low 10 bits) decides
        return _bits(0x3F2A5400 | rng.integers(0, 1 << 10, m))
    if kind == "top11":       # the first pass's bin is shared, the lower 21 bits are free
        return _bits(0x3FA00000 | rng.integers(0, 1 << 21, m))
    if kind == "denormal":
        u = rng.integers(1, 1 << 23, m)
        u[rng.random(m) < 0.1] = 0
        return _bits(u)
    if kind == "inf":
        v = rng.random(m).astype(np.float32)
        v[rng.random(m) < 0.4] = np.inf
        return v
    if kind == "every_exponent":  # uniform over the bit patterns of the non-negative finite floats and +inf
        return _bits(rng.integers(0, 0x7F800001, m))
    if kind == "c1_d2":
        return c1_d2[rng.integers(0, len(c1_d2), m)] if m > len(c1_d2) else c1_d2[rng.permutation(len(c1_d2))[:m]]
    raise ValueError(kind)


def _ranks(sorted_u, rng):
    """{0, m/2, m-1}, a few random ranks, and ranks on both sides of the edges between the bins of each pass."""
    m = len(sorted_u)
    r = {0, m // 2, m - 1}
    r.update(int(x) for x in rng.integers(0, m, 5))
    for shift in (21, 10, 0):
        edges = np.flatnonzero(np.diff(sorted_u >> shift)) + 1
        for k in edges[:: max(1, len(edges) // 3)][:3]:
            r.update((int(k) - 1, int(k)))
    return np.array(sorted(r), np.int32)


def _select(dev, v, nths, skip_neg):
    ctx, lib, _ = dev
    v = np.ascontiguousarray(v, np.float32)
    nths = np.ascontiguousarray(nths, np.int32)
    out = np.full(len(nths), np.nan, np.float32)
    ctx.check(lib.peb_debug_select_nth(ctx.handle, v.ctypes.data, len(v), nths.ctypes.data, len(nths), int(skip_neg), out.ctypes.data))
    return out


@pytest.mark.parametrize("m", SIZES)
@pytest.mark.parametrize("kind", ["all_equal", "all_plus_zero", "two_values", "low10", "top11", "denormal", "inf",
                                  "every_exponent", "c1_d2"])
def test_select_nth_is_the_exact_order_statistic(dev, c1_d2, m, kind):
    rng = np.random.default_rng(m * 7 + len(kind))
    v = _values(kind, m, rng, c1_d2)
    su = np.sort(v.view(np.uint32))
    nths = _ranks(su, rng)
    got = _select(dev, v, nths, False)
    assert np.array_equal(got.view(np.uint32), su[nths]), [(int(k), float(a), float(b)) for k, a, b in
                                                           zip(nths, got, su[nths].view(np.float32)) if a != b][:5]


@pytest.mark.parametrize("m", SIZES)
@pytest.mark.parametrize("kind", ["minus_one_markers", "minus_zero"])
def test_select_nth_skips_values_with_the_sign_bit(dev, c1_d2, m, kind):
    rng = np.random.default_rng(m * 13 + len(kind))
    if kind == "minus_one_markers":  # how the rejectors leave entries out: -1.0f on about half of them
        v = _values("c1_d2", m, rng, c1_d2)
        v[rng.random(m) < 0.5] = -1.0
    else:  # -0.0f has the sign bit: skipped like any negative value, while +0.0f is taken
        v = _values("two_values", m, rng, c1_d2)
        r = rng.random(m)
        v[r < 0.35] = -0.0
        v[(r >= 0.35) & (r < 0.5)] = 0.0
    v[rng.integers(0, m)] = 0.125  # at least one value taken
    taken = v[~np.signbit(v)]
    su = np.sort(taken.view(np.uint32))
    nths = _ranks(su, rng)
    got = _select(dev, v, nths, True)
    assert np.array_equal(got.view(np.uint32), su[nths])
    assert not np.signbit(got).any()


def test_rank_outside_the_taken_values_is_refused_before_the_launch(dev):
    _, _, pcl = dev
    v = np.array([1.0, -1.0, -0.0, 2.0], np.float32)
    with pytest.raises(pcl.PebError):
        _select(dev, v, [2], True)   # two values taken: ranks 0 and 1 only
    with pytest.raises(pcl.PebError):
        _select(dev, v, [4], False)
    assert _select(dev, v, [1], True)[0] == 2.0
