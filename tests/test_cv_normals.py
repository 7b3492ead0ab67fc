"""cv::ppf_match_3d::computeNormalsPC3d (DESIGN.md §13) without a GPU.

- The device's eigen solver (core_math.cuh : cv_eigen_sym3, compiled for the host by tests/host/cv_normals_host.cu) and
  the oracle's general-n restatement agree with the real cv2.eigen bit for bit.  The image's cv2 is built without Eigen,
  so cv2.eigen runs OpenCV's own JacobiImpl_.
- The oracle (tests/cv_normals_oracle.cpp : orc_cv_normals) agrees with an independent witness: real cv2.flann_Index
  (KDTREE_SINGLE, leaf 8, as indexPCFlann builds it), numpy float32 products summed in float64 in list order, real
  cv2.eigen and the float flip.  Bitwise wherever the two neighbour lists agree.
- The formula is accurate: on a wavy patch at 0.72 m the normals are within 0.1 deg (median) of a double PCA of the
  same neighbours.
- The header's prototypes compile from C and through the C++ facade (tests/cpp/cv_normals_check.cpp)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cv_normals_oracle as cvo
from util import tie_ok

ROOT = Path(__file__).resolve().parents[1]
NVCC = "/usr/local/cuda/bin/nvcc" if Path("/usr/local/cuda/bin/nvcc").exists() else "nvcc"


# ---- inputs shared with test_gpu_cv_normals.py ---------------------------------------------------------------------
def wavy_patch(n: int = 40000, seed: int = 0, z0: float = 0.72, noise: float = 1e-4, side: float = 0.2) -> np.ndarray:
    """n points on a tilted, wavy surface around z = z0 with Gaussian noise, (n, 3) float32."""
    rng = np.random.default_rng(seed)
    u = rng.uniform(-side / 2, side / 2, n)
    v = rng.uniform(-side / 2, side / 2, n)
    h = 0.004 * np.sin(40.0 * u) * np.cos(30.0 * v) + 0.25 * u - 0.15 * v
    p = np.stack([u, v, z0 + h], 1) + rng.normal(0.0, noise, (n, 3))
    return p.astype(np.float32)


def symmetric_matrices(rng, per_scale: int = 400) -> np.ndarray:
    """Random, rank-deficient (rank 2 and 1), diagonal and zero symmetric 3 x 3 doubles at scales 1e-16 .. 1e4."""
    out = [np.zeros((3, 3))]
    for scale in (1e-16, 1e-12, 1e-8, 1e-4, 1e-2, 1.0, 1e2, 1e4):
        B = rng.normal(size=(per_scale, 3, 3))
        out += list((B + B.transpose(0, 2, 1)) * scale)
        U = rng.normal(size=(per_scale, 3, 2))
        out += list(np.einsum("nik,nk,njk->nij", U, rng.uniform(0, 1, (per_scale, 2)), U) * scale)
        u = rng.normal(size=(per_scale // 2, 3))
        out += list(np.einsum("ni,nj->nij", u, u) * scale)
        out += [np.diag(d) * scale for d in rng.normal(size=(per_scale // 2, 3))]
        out += [np.diag(np.repeat(d, 3)) * scale for d in rng.normal(size=per_scale // 8)]
    return np.ascontiguousarray(np.array(out, np.float64))


def cv_covariances(P: np.ndarray, idx: np.ndarray) -> np.ndarray:
    """meanCovLocalPCInd over the lists idx (n, k): float32 products, float64 sums in list order."""
    k = idx.shape[1]
    nb = P[idx][:, :, :3].astype(np.float32)
    Cs = np.zeros((len(idx), 3, 3))
    mu = np.zeros((len(idx), 3))
    for i in range(k):  # one neighbour after the other, like the loop upstream
        c = nb[:, i]
        Cs += (c[:, :, None] * c[:, None, :]).astype(np.float64)  # product in float32, then widened
        mu += c.astype(np.float64)
    inv = 1.0 / k
    mu = mu * inv
    Cs = Cs * inv
    return Cs - mu[:, :, None] * mu[:, None, :]


def witness_normals(P: np.ndarray, k: int, flip: bool = True, viewpoint=(0.0, 0.0, 0.0)):
    """The independent witness: real FLANN, numpy arithmetic, real cv2.eigen.  Finite clouds only.
    -> ((n, 6) float32, (n, k) int32 lists)."""
    import cv2

    P = np.ascontiguousarray(np.asarray(P, np.float32)[:, :3])
    index = cv2.flann_Index(P, {"algorithm": 4, "leaf_max_size": 8})  # KDTreeSingleIndexParams(8)
    idx, _ = index.knnSearch(P, k, params={"checks": 32})
    idx = idx.astype(np.int32).reshape(len(P), k)
    Cs = cv_covariances(P, idx)
    n = np.empty((len(P), 3), np.float32)
    for i in range(len(P)):
        _, _, V = cv2.eigen(Cs[i])
        n[i] = V[2].astype(np.float32)
    if flip:
        d = np.asarray(viewpoint, np.float32)[None, :] - P
        cos = np.float32(0) + d[:, 0] * n[:, 0]
        cos = cos + d[:, 1] * n[:, 1]
        cos = cos + d[:, 2] * n[:, 2]
        n[cos < 0] *= np.float32(-1)
    return np.concatenate([P, n], 1), idx


def same_bits(a, b) -> np.ndarray:
    return np.asarray(a, np.float32).view(np.uint32) == np.asarray(b, np.float32).view(np.uint32)


# ---- the host build of the device tail -------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    so = tmp_path_factory.mktemp("cv_normals_host") / "libcv_normals_host.so"
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-fmad=false", "-Xcompiler",
           "-fPIC,-fvisibility=hidden,-ffp-contract=off", "--expt-relaxed-constexpr", "-shared", "-cudart", "static",
           "-o", str(so), str(ROOT / "tests" / "host" / "cv_normals_host.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(so))
    L.hc_cv_eigen_sym3.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    L.hc_cv_normal.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return L


def host_eigen(L, A):
    A = np.ascontiguousarray(A, np.float64).reshape(-1, 9)
    W = np.empty((len(A), 3))
    V = np.empty((len(A), 9))
    L.hc_cv_eigen_sym3(A.ctypes.data, len(A), W.ctypes.data, V.ctypes.data)
    return W, V.reshape(-1, 3, 3)


def cv2_eigen(A):
    import cv2

    W = np.empty((len(A), 3))
    V = np.empty((len(A), 3, 3))
    for i, M in enumerate(A):
        ok, w, v = cv2.eigen(np.ascontiguousarray(M))
        assert ok
        W[i] = w.ravel()
        V[i] = v
    return W, V


def test_image_cv2_runs_opencvs_own_jacobi():
    import cv2

    info = cv2.getBuildInformation()
    line = next(ln for ln in info.splitlines() if ln.strip().startswith("Eigen:"))
    assert "NO" in line, line  # with Eigen, cv::eigen would be Eigen::SelfAdjointEigenSolver: nothing to pin against


def test_device_and_oracle_eigen_match_cv2_bitwise(hostlib, oracle):
    rng = np.random.default_rng(2026)
    A = symmetric_matrices(rng)
    # real neighbourhood covariances of the accuracy patch, k = 20
    P = wavy_patch(4000, seed=3)
    idx, _ = oracle.knn(P, P, 20)
    A = np.concatenate([A, cv_covariances(P, idx)])
    assert len(A) >= 10000
    Wc, Vc = cv2_eigen(A)
    Wh, Vh = host_eigen(hostlib, A)
    Wo, Vo = cvo.cv_eigen3(A)
    for W, V in ((Wh, Vh), (Wo, Vo)):
        assert np.array_equal(W.view(np.uint64), Wc.view(np.uint64))
        assert np.array_equal(V.view(np.uint64), Vc.view(np.uint64))


def test_device_tail_matches_oracle_bitwise(hostlib):
    """cv_moments_add + cv_normal_from_moments (host build) on the oracle's own lists give the oracle's normals."""
    P = wavy_patch(3000, seed=5)
    for k, flip, vp in ((20, True, (0.0, 0.0, 0.0)), (7, False, (0.0, 0.0, 0.0)), (33, True, (0.05, -0.3, 1.5))):
        ref, nn = cvo.cv_normals(P, k, flip=flip, viewpoint=vp, want_nn=True)
        vpa = np.asarray(vp, np.float32)
        got = np.empty((len(P), 3), np.float32)
        for i in range(len(P)):
            nb = np.ascontiguousarray(P[nn[i]])
            hostlib.hc_cv_normal(nb.ctypes.data, k, P[i].ctypes.data, int(flip), vpa.ctypes.data, got[i].ctypes.data)
        assert same_bits(got, ref[:, 3:]).all()


@pytest.mark.parametrize("k,flip,vp", [(20, True, (0.0, 0.0, 0.0)), (5, True, (0.0, 0.0, 0.0)), (20, False, (0.0, 0.0, 0.0)),
                                       (40, True, (0.1, 0.2, 2.0))])
def test_oracle_matches_independent_witness(k, flip, vp):
    P = wavy_patch(6000, seed=7)
    ref, rnn = cvo.cv_normals(P, k, flip=flip, viewpoint=vp, want_nn=True)
    wit, wnn = witness_normals(P, k, flip, vp)
    assert tie_ok(P, P, rnn.reshape(-1), wnn.reshape(-1))
    same = (rnn == wnn).all(1)
    assert same.mean() > 0.99
    assert same_bits(ref[same], wit[same]).all()
    assert same_bits(ref[:, :3], P).all()


def test_accuracy_against_double_pca_of_the_same_neighbours():
    P = wavy_patch(40000, seed=0)
    out, nn = cvo.cv_normals(P, 20, want_nn=True)
    nb = P[nn].astype(np.float64)
    d = nb - nb.mean(1, keepdims=True)
    _, vecs = np.linalg.eigh(np.einsum("nki,nkj->nij", d, d))
    ref = vecs[:, :, 0]
    cos = np.abs((out[:, 3:].astype(np.float64) * ref).sum(1)) / np.linalg.norm(out[:, 3:], axis=1)
    ang = np.degrees(np.arccos(np.clip(cos, -1.0, 1.0)))
    assert np.median(ang) < 0.1 and ang.max() < 1.0, (np.median(ang), np.percentile(ang, 99), ang.max())
    assert (out[:, 5] <= 0).all()  # flipped towards the origin, which lies below the patch's normals


def test_oracle_edge_cases():
    rng = np.random.default_rng(11)
    P = rng.normal(0, 0.01, (60, 3)).astype(np.float32) + np.float32([0, 0, 0.7])
    P[7] = np.nan
    P[9, 1] = np.inf
    out, nn = cvo.cv_normals(P, 10, want_nn=True)
    bad = np.array([7, 9])
    assert np.isnan(out[bad, 3:]).all() and (nn[bad] == -1).all()
    assert np.isnan(out[7, :3]).all() and out[9, 1] == np.inf  # xyz copied as they are
    good = np.setdiff1d(np.arange(60), bad)
    assert np.isfinite(out[good]).all() and not np.isin(nn[good], bad).any()
    with pytest.raises(ValueError):
        cvo.cv_normals(P, 0)
    with pytest.raises(ValueError):
        cvo.cv_normals(P, 59)  # 58 finite points
    assert cvo.cv_normals(P, 58).shape == (60, 6)
    # duplicates whose float products are exact: zero covariance, cv::eigen keeps the identity, row 2 = (0, 0, 1),
    # flipped towards the viewpoint.  (For other values the float-rounded products against the double mean leave a
    # covariance of rounding noise, and the normal is whatever that noise gives — in OpenCV as here.)
    D = np.repeat(np.float32([[0.5, 0.25, 0.75]]), 12, 0)
    assert (cvo.cv_normals(D, 5, viewpoint=(0, 0, 0))[:, 3:] == np.float32([0, 0, -1])).all()
    assert (cvo.cv_normals(D, 5, viewpoint=(0, 0, 2))[:, 3:] == np.float32([0, 0, 1])).all()
    assert (cvo.cv_normals(D, 5, flip=False)[:, 3:] == np.float32([0, 0, 1])).all()
    # collinear points: a unit normal perpendicular to the line
    L = np.zeros((30, 3), np.float32)
    L[:, 0] = np.linspace(0, 0.03, 30)
    L[:, 2] = 0.7
    n = cvo.cv_normals(L, 6)[:, 3:]
    assert np.allclose(np.linalg.norm(n, axis=1), 1, atol=1e-6) and np.abs(n[:, 0]).max() < 1e-3
    assert cvo.cv_normals(np.empty((0, 3), np.float32), 20).shape == (0, 6)


def test_header_prototypes_compile_from_c_and_the_facade(tmp_path):
    lib_dir = ROOT / "pose_estimation_b200"
    src = ROOT / "tests" / "cpp" / "cv_normals_check.cpp"
    builds = {"c": ["gcc", "-x", "c", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror"],
              "cpp": ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra"]}
    P = wavy_patch(500, seed=1)
    (tmp_path / "in.f32").write_bytes(P.tobytes())
    for name, cc in builds.items():
        exe = tmp_path / f"cv_normals_check_{name}"
        r = subprocess.run(cc + ["-I", str(ROOT / "include"), str(src), "-o", str(exe), "-L", str(lib_dir), "-lpe_b200",
                                 "-lm", f"-Wl,-rpath,{lib_dir}"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        import torch

        if torch.cuda.is_available():
            continue  # the run is checked in test_gpu_cv_normals.py
        r = subprocess.run([str(exe), str(tmp_path / "in.f32"), "500", "20", "1", str(tmp_path / "out.f32")],
                           capture_output=True, text=True)
        assert r.returncode == 3 and "no CPU fallback" in r.stderr, (r.returncode, r.stderr)
        assert not (tmp_path / "out.f32").exists()

