"""GeneralizedIterativeClosestPoint without a GPU: the CPU oracle (tests/gicp_oracle.cpp, an independent sequential
restatement of gicp.hpp / bfgs.h on oracle/pcl_oracle.cpp) against numpy witnesses, central differences and scipy's BFGS,
and the library's scalar code compiled for the CPU (tests/host/gicp_host.cu) against the oracle bit for bit."""
import numpy as np
import pytest
from scipy.optimize import minimize

import gicp_oracle as GO


def _rot(x):
    cx, sx, cy, sy, cz, sz = np.cos(x[3]), np.sin(x[3]), np.cos(x[4]), np.sin(x[4]), np.cos(x[5]), np.sin(x[5])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    dRz = np.array([[-sz, -cz, 0], [cz, -sz, 0], [0, 0, 0]])
    dRy = np.array([[-sy, 0, cy], [0, 0, 0], [-cy, 0, -sy]])
    dRx = np.array([[0, 0, 0], [0, -sx, -cx], [0, cx, -sx]])
    return Rz @ Ry @ Rx, [Rz @ Ry @ dRx, Rz @ dRy @ Rx, dRz @ Ry @ Rx]


def _f_double(p, t, M, x):
    R, _ = _rot(x)
    res = p.astype(np.float64) @ R.T + x[:3] - t.astype(np.float64)
    return float(np.einsum("ni,nij,nj->", res, M, res) / len(p))


def _g_double(p, t, M, x):
    R, dR = _rot(x)
    pd = p.astype(np.float64)
    res = pd @ R.T + x[:3] - t.astype(np.float64)
    temp = np.einsum("nij,nj->ni", M, res)
    return np.concatenate([2.0 / len(p) * temp.sum(0), [2.0 / len(p) * np.sum(temp * (pd @ D.T)) for D in dR]])


@pytest.fixture(scope="module")
def pairs():
    rng = np.random.default_rng(7)
    m = 400
    p = rng.uniform(-0.05, 0.05, (m, 3)).astype(np.float32)
    t = (p + rng.normal(0, 0.02, (m, 3))).astype(np.float32)
    A = rng.normal(0, 1, (m, 3, 3))
    M = np.einsum("nij,nkj->nik", A, A) + 0.1 * np.eye(3)
    return p, t, M


def test_covariances_match_the_numpy_witness():
    rng = np.random.default_rng(1)
    cloud = rng.normal(0, 0.01, (300, 3)).astype(np.float32)
    cloud[::50] = np.nan
    k = 20
    got = GO.covariances(cloud, k)
    fin = np.nonzero(np.isfinite(cloud).all(1))[0]
    assert np.isnan(got[~np.isfinite(cloud).all(1)]).all()
    pts = cloud[fin]
    d = pts[:, None, :] - pts[None, :, :]
    d2 = ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).astype(np.float32)
    for r, i in enumerate(fin):
        nb = pts[np.lexsort((np.arange(len(pts)), d2[r]))[:k]]
        prod = np.einsum("ni,nj->nij", nb, nb).astype(np.float32).astype(np.float64)  # float products, double sums
        mean = nb.astype(np.float64).sum(0) / k
        cov = prod.sum(0) / k - np.outer(mean, mean)
        U, _, _ = np.linalg.svd(cov)
        want = U @ np.diag([1.0, 1.0, 1e-3]) @ U.T
        assert np.allclose(got[i], want, rtol=0, atol=1e-12), (i, np.abs(got[i] - want).max())
        # the library's covariance tail (svd3: reciprocal square roots where Eigen divides) agrees to the last bits
        assert np.allclose(GO.host_cov(nb), got[i], rtol=0, atol=1e-12)


def test_cost_and_gradient_match_the_witness_and_central_differences(pairs):
    p, t, M = pairs
    rng = np.random.default_rng(4)
    for _ in range(10):
        x = np.concatenate([rng.uniform(-0.01, 0.01, 3), rng.uniform(-0.3, 0.3, 3)])
        f, g = GO.fg(p, t, M, x)
        # witness with the oracle's own float transform: only the order of the double sums differs
        T = GO.apply_state(x)
        pp = (((T[None, :3, 0] * p[:, :1] + T[None, :3, 1] * p[:, 1:2]) + T[None, :3, 2] * p[:, 2:]) + T[None, :3, 3]).astype(np.float32)
        res = (pp - t).astype(np.float64)
        temp = np.einsum("nij,nj->ni", M, res)
        fw = float(np.sum(res * temp)) / len(p)
        Racc = 2.0 / len(p) * np.einsum("ni,nj->ij", p.astype(np.float64), temp)
        _, dR = _rot(x)
        gw = np.concatenate([2.0 / len(p) * temp.sum(0), [np.trace(D @ Racc) for D in dR]])
        assert abs(f - fw) <= 1e-12 * abs(f)
        assert np.abs(g - gw).max() <= 1e-12 * np.abs(g).max()
        num = np.array([(_f_double(p, t, M, x + e) - _f_double(p, t, M, x - e)) / 2e-7 for e in 1e-7 * np.eye(6)])
        assert np.abs(g - num).max() <= 1e-6 * np.abs(num).max(), (g, num)


def test_library_scalar_code_reproduces_the_oracle_bit_for_bit(pairs):
    p, t, M = pairs
    rng = np.random.default_rng(6)
    for _ in range(5):
        x = np.concatenate([rng.uniform(-0.01, 0.01, 3), rng.uniform(-0.5, 0.5, 3)])
        assert np.array_equal(GO.apply_state(x), GO.apply_state(x, "host"))
        fo, go = GO.fg(p, t, M, x)
        fh, gh = GO.fg(p, t, M, x, "host")
        assert fo == fh and np.array_equal(go, gh)
    for scale in (1.0, 1e4):
        xo, io, eo = GO.bfgs(p, t, M * scale, np.zeros(6), 50)
        xh, ih, eh = GO.bfgs(p, t, M * scale, np.zeros(6), 50, "host")
        assert np.array_equal(xo, xh) and (io, eo) == (ih, eh)


def test_oracle_bfgs_minimises_a_quadratic_and_rosenbrock():
    rng = np.random.default_rng(5)
    A = rng.normal(size=(6, 6))
    Q = A @ A.T + 6 * np.eye(6)
    b = rng.normal(size=6)
    x, _, _ = GO.bfgs_fn(lambda x: (0.5 * x @ Q @ x - b @ x, Q @ x - b), np.zeros(6), 200)
    assert np.allclose(x, np.linalg.solve(Q, b), atol=1e-3)  # |g| < 0.01 stops it

    def rosen(x):
        f = sum(100 * (x[i + 1] - x[i] ** 2) ** 2 + (1 - x[i]) ** 2 for i in range(5))
        g = np.zeros(6)
        for i in range(5):
            g[i] += -400 * x[i] * (x[i + 1] - x[i] ** 2) - 2 * (1 - x[i])
            g[i + 1] += 200 * (x[i + 1] - x[i] ** 2)
        return f, g

    x, _, _ = GO.bfgs_fn(rosen, np.full(6, -0.5), 2000)
    assert np.allclose(x, 1.0, atol=1e-2), x


def test_oracle_bfgs_on_a_gicp_cost_reaches_scipys_minimum():
    # a well-conditioned cost (points spread over a metre); PCL's inner loop stops at |g| < 0.01, an absolute bound, so
    # the weights are scaled to put it far below the cost
    rng = np.random.default_rng(8)
    p = rng.uniform(-1, 1, (400, 3)).astype(np.float32)
    t = (p + rng.normal(0, 0.05, (400, 3))).astype(np.float32)
    A = rng.normal(0, 1, (400, 3, 3))
    M = (np.einsum("nij,nkj->nik", A, A) + 0.1 * np.eye(3)) * 1e6
    x, _, _ = GO.bfgs(p, t, M, np.zeros(6), 200)
    ref = minimize(lambda v: _f_double(p, t, M, v), np.zeros(6), jac=lambda v: _g_double(p, t, M, v), method="BFGS",
                   options={"gtol": 1e-12})
    f = _f_double(p, t, M, x)
    # PCL's cost moves the points with float transforms: f is resolved to ~1e-7 relative (float eps x coordinate / residual), not 1e-9
    assert abs(f - ref.fun) <= 1e-6 * abs(ref.fun), (f, ref.fun)
    # ... and its line search stops (NoProgress) once f's float noise hides the descent: x within 1e-4 of the minimum
    assert np.allclose(x, ref.x, atol=1e-4), (x - ref.x)
