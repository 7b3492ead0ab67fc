"""ctypes face of tests/gicp_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle of pcl::GeneralizedIterativeClosestPoint (the
unchanged oracle/pcl_oracle.cpp plus an independent sequential restatement of gicp.hpp and bfgs.h), and of
tests/host/gicp_host.cu (the library's scalar GICP code, csrc/gicp_math.cuh, compiled for the CPU) so that the two can be
compared bit for bit.  Both shared objects are compiled once per process into a temporary directory, with the parity
flags of oracle/Makefile, so the repository tree is never written."""
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
_vp, _i, _sz = C.c_void_p, C.c_int, C.c_size_t
FDF = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double))


class GicpParams(C.Structure):
    """peb_gicp_params (include/pe_b200.h)."""

    _fields_ = [("max_iterations", C.c_int32), ("k_correspondences", C.c_int32), ("max_inner_iterations", C.c_int32),
                ("reserved", C.c_int32), ("max_corr_dist", C.c_double), ("transformation_epsilon", C.c_double),
                ("rotation_epsilon", C.c_double), ("fitness_max_range", C.c_double)]


def params(**kw) -> GicpParams:
    p = GicpParams(200, 20, 20, 0, 5.0, 5e-4, 2e-3, float(np.finfo(np.float64).max))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _tmp(prefix):
    tmp = Path(tempfile.mkdtemp(prefix=prefix))
    atexit.register(shutil.rmtree, tmp, True)
    return tmp


@functools.lru_cache(maxsize=1)
def oracle() -> C.CDLL:
    so = _tmp("gicp_oracle_") / "libgicp_oracle.so"
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    r = subprocess.run([cxx, "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-O2", "-ffp-contract=off", "-o", str(so),
                        str(_HERE / "gicp_oracle.cpp")], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building the GICP oracle failed:\n{r.stderr}")
    L = C.CDLL(str(so))
    L.orc_gicp_covariances.argtypes = [_vp, _sz, _sz, _i, _vp]
    L.orc_gicp_fg.argtypes = [_vp, _vp, _vp, _i, _vp, _vp, _vp]
    L.orc_gicp_apply_state.argtypes = [_vp, _vp]
    L.orc_gicp_bfgs.argtypes = [_vp, _vp, _vp, _i, FDF, _vp, _i, _vp]
    L.orc_gicp_bfgs.restype = _i
    L.orc_gicp_align.argtypes = [_vp, _sz, _sz, _vp, _sz, _sz, _vp, C.POINTER(GicpParams), _vp]
    return L


@functools.lru_cache(maxsize=1)
def host() -> C.CDLL:
    so = _tmp("gicp_host_") / "libgicp_host.so"
    nvcc = "/usr/local/cuda/bin/nvcc" if Path("/usr/local/cuda/bin/nvcc").exists() else "nvcc"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-fmad=false", "-Xcompiler",
                        "-fPIC,-fvisibility=hidden,-ffp-contract=off", "--expt-relaxed-constexpr", "-shared", "-cudart", "static",
                        "-o", str(so), str(_HERE / "host" / "gicp_host.cu")], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building the GICP host shim failed:\n{r.stderr}")
    L = C.CDLL(str(so))
    L.gh_fg.argtypes = [_vp, _vp, _vp, _i, _vp, _vp, _vp]
    L.gh_bfgs.argtypes = [_vp, _vp, _vp, _i, _vp, _i, _vp]
    L.gh_bfgs.restype = _i
    L.gh_cov.argtypes = [_vp, _i, _vp]
    L.gh_apply_state.argtypes = [_vp, _vp]
    return L


def _p(a):
    return a.ctypes.data


def _pairs(p, t, M):
    return (np.ascontiguousarray(p, np.float32), np.ascontiguousarray(t, np.float32), np.ascontiguousarray(M, np.float64))


def fg(p, t, M, x, lib="oracle"):
    """f and g of fixed pairs (p = output[i], t = target point: (m, 3); M: (m, 3, 3)) at x."""
    p, t, M = _pairs(p, t, M)
    x = np.ascontiguousarray(x, np.float64)
    f, g = np.zeros(1), np.zeros(6)
    fn = oracle().orc_gicp_fg if lib == "oracle" else host().gh_fg
    fn(_p(p), _p(t), _p(M), len(p), _p(x), _p(f), _p(g))
    return f[0], g


def bfgs(p, t, M, x, max_inner=20, lib="oracle"):
    """estimateRigidTransformationBFGS's minimisation over fixed pairs -> (x, inner iterations, evaluations)."""
    p, t, M = _pairs(p, t, M)
    x = np.array(x, np.float64)
    ev = C.c_int(0)
    if lib == "oracle":
        inner = oracle().orc_gicp_bfgs(_p(p), _p(t), _p(M), len(p), FDF(), _p(x), max_inner, C.byref(ev))
    else:
        inner = host().gh_bfgs(_p(p), _p(t), _p(M), len(p), _p(x), max_inner, C.byref(ev))
    return x, inner, ev.value


def bfgs_fn(fn, x, max_inner=200):
    """The oracle's minimiser over a Python objective fn(x) -> (f, g)."""
    def cb(xp, fp, gp):
        f, g = fn(np.ctypeslib.as_array(xp, (6,)).copy())
        fp[0] = float(f)
        for i in range(6):
            gp[i] = float(g[i])

    x = np.array(x, np.float64)
    ev = C.c_int(0)
    inner = oracle().orc_gicp_bfgs(None, None, None, 0, FDF(cb), _p(x), max_inner, C.byref(ev))
    return x, inner, ev.value


def apply_state(x, lib="oracle"):
    T = np.zeros(16, np.float32)
    x = np.ascontiguousarray(x, np.float64)
    (oracle().orc_gicp_apply_state if lib == "oracle" else host().gh_apply_state)(_p(x), _p(T))
    return T.reshape(4, 4).T.copy()


def host_cov(neighbours):
    nb = np.ascontiguousarray(neighbours, np.float32)
    out = np.zeros(9)
    host().gh_cov(_p(nb), len(nb), _p(out))
    return out.reshape(3, 3)


def covariances(cloud, k=20):
    c = np.ascontiguousarray(np.asarray(cloud, np.float32)[:, :3])
    out = np.zeros((len(c), 9))
    oracle().orc_gicp_covariances(_p(c), len(c), 12, k, _p(out))
    return out.reshape(-1, 3, 3)


def align(source, target, guess=None, prm: GicpParams | None = None):
    """The oracle's computeTransformation + getFitnessScore -> peb_icp_result-shaped record (oracle.IcpResult)."""
    from oracle import IcpResult

    s = np.ascontiguousarray(np.asarray(source, np.float32)[:, :3])
    t = np.ascontiguousarray(np.asarray(target, np.float32)[:, :3])
    g = np.ascontiguousarray(np.asarray(guess, np.float32).T) if guess is not None else None
    res = IcpResult()
    oracle().orc_gicp_align(_p(s), len(s), 12, _p(t), len(t), 12, _p(g) if g is not None else None, C.byref(prm or params()),
                            C.byref(res))
    return res


def matrix(rec):
    return np.array(rec.T, np.float32).reshape(4, 4).T.copy()
