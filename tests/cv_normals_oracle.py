"""ctypes face of tests/cv_normals_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle of
cv::ppf_match_3d::computeNormalsPC3d (the unchanged oracle/pcl_oracle.cpp kd-tree plus OpenCV's tail, DESIGN.md §13).
Each build of the shared object is compiled once per process into a temporary directory, so the repository tree is never
written: `parity` with the flags of oracle/Makefile's parity build (-O2 -ffp-contract=off), `timing` with those of its
timing build (-O3 -march=x86-64-v3) for tools/bench_cv_normals.py."""
from __future__ import annotations

import atexit
import ctypes as C
import functools
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_vp, _sz = C.c_void_p, C.c_size_t
_FLAGS = {"parity": ["-O2", "-ffp-contract=off"], "timing": ["-O3", "-march=x86-64-v3"]}


@functools.lru_cache(maxsize=2)
def _lib(build: str = "parity") -> C.CDLL:
    tmp = Path(tempfile.mkdtemp(prefix="cv_normals_oracle_"))
    atexit.register(shutil.rmtree, tmp, True)
    so = tmp / f"libcv_normals_oracle_{build}.so"
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    cmd = [cxx, "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-fopenmp", *_FLAGS[build], "-o", str(so),
           str(_HERE / "cv_normals_oracle.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building the computeNormalsPC3d oracle failed:\n{r.stderr}")
    L = C.CDLL(str(so))
    L.orc_cv_normals.restype = C.c_int
    L.orc_cv_normals.argtypes = [_vp, _sz, _sz, C.c_int, C.c_int, _vp, _vp, _vp, C.c_int]
    L.orc_cv_eigen3.argtypes = [_vp, _sz, _vp, _vp]
    return L


def cv_normals(pts: np.ndarray, k: int = 20, flip: bool = True, viewpoint=(0.0, 0.0, 0.0), threads: int = 1,
               want_nn: bool = False, build: str = "parity"):
    """(N, 6) float32 rows x y z nx ny nz (and the (N, k) neighbour lists, -1 on non-finite rows); ValueError where the
    library returns PEB_E_INVALID_ARG (k < 1, k > the number of finite points).  threads <= 0: all cores."""
    p = np.ascontiguousarray(pts, np.float32)
    vp = np.ascontiguousarray(np.asarray(viewpoint, np.float32).reshape(3))
    out = np.empty((p.shape[0], 6), np.float32)
    nn = np.empty((p.shape[0], max(k, 0)), np.int32) if want_nn else None
    rc = _lib(build).orc_cv_normals(p.ctypes.data, p.shape[0], p.strides[0], k, int(bool(flip)), vp.ctypes.data,
                                    out.ctypes.data, nn.ctypes.data if want_nn else None, threads)
    if rc != 0:
        raise ValueError(f"cv_normals: k = {k} is not in [1, finite points]")
    return (out, nn) if want_nn else out


def cv_eigen3(A: np.ndarray):
    """cv::eigen of (m, 3, 3) symmetric doubles -> (eigenvalues (m, 3) descending, eigenvectors (m, 3, 3) as rows)."""
    a = np.ascontiguousarray(np.asarray(A, np.float64).reshape(-1, 9))
    W = np.empty((a.shape[0], 3), np.float64)
    V = np.empty((a.shape[0], 9), np.float64)
    _lib().orc_cv_eigen3(a.ctypes.data, a.shape[0], W.ctypes.data, V.ctypes.data)
    return W, V.reshape(-1, 3, 3)
