"""ctypes face of tests/rejector_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's ICP with a correspondence rejector
chain (the unchanged oracle/pcl_oracle.cpp plus the chain).  The shared object is compiled once per process into a
temporary directory, with the parity flags of oracle/Makefile, so the repository tree is never written."""
from __future__ import annotations

import atexit
import ctypes as C
import functools
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import IcpParams, IcpResult, default_params

_HERE = Path(__file__).resolve().parent
_vp, _sz = C.c_void_p, C.c_size_t

REJECTOR_DISTANCE, REJECTOR_MEDIAN_DISTANCE, REJECTOR_ONE_TO_ONE, REJECTOR_TRIMMED = range(4)


class Rejector(C.Structure):
    """peb_rejector (include/pe_b200.h)."""

    _fields_ = [("kind", C.c_int32), ("min_correspondences", C.c_int32), ("value", C.c_double)]


def rejector_chain(chain):
    """chain: (kind, value[, min_correspondences]) tuples, in the order the rejectors are added -> (array, count)."""
    arr = (Rejector * max(len(chain), 1))()
    for k, r in enumerate(chain):
        arr[k].kind = int(r[0])
        arr[k].value = float(r[1]) if len(r) > 1 else 0.0
        arr[k].min_correspondences = int(r[2]) if len(r) > 2 else 0
    return arr, len(chain)


@functools.lru_cache(maxsize=1)
def _lib() -> C.CDLL:
    tmp = Path(tempfile.mkdtemp(prefix="rejector_oracle_"))
    atexit.register(shutil.rmtree, tmp, True)
    so = tmp / "librejector_oracle.so"
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    cmd = [cxx, "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-fopenmp", "-O2", "-ffp-contract=off",
           "-o", str(so), str(_HERE / "rejector_oracle.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building the rejector oracle failed:\n{r.stderr}")
    L = C.CDLL(str(so))
    L.orc_icp_chain_create.restype = _vp
    L.orc_icp_chain_destroy.argtypes = [_vp]
    L.orc_icp_chain_as_icp.restype = _vp
    L.orc_icp_chain_as_icp.argtypes = [_vp]
    L.orc_icp_set_wide_accum.argtypes = [_vp, C.c_int]
    L.orc_icp_set_target.argtypes = [_vp, _vp, _sz, _sz, _vp, _sz]
    L.orc_icp_align_ex.argtypes = [_vp, _vp, _sz, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]
    L.orc_icp_align_batch_ex.argtypes = [_vp, _vp, _sz, _sz, _vp, _sz, _vp, _vp, _sz, _vp, C.c_int]
    L.orc_reject_pairs.restype = _sz
    L.orc_reject_pairs.argtypes = [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]
    return L


def reject_pairs(q, m, d2, score, chain) -> np.ndarray:
    """The rejector chain over a scripted pair set (q unique): positions of the pairs left, in the chain's order."""
    L = _lib()
    q, m = np.ascontiguousarray(q, np.int32), np.ascontiguousarray(m, np.int32)
    d2, score = np.ascontiguousarray(d2, np.float32), np.ascontiguousarray(score, np.float32)
    arr, n_chain = rejector_chain(chain)
    out = np.empty(max(len(q), 1), np.int32)
    k = L.orc_reject_pairs(q.ctypes.data, m.ctypes.data, d2.ctypes.data, score.ctypes.data, len(q), arr, n_chain,
                           out.ctypes.data)
    return out[:k].copy()


class ChainIcp:
    """oracle.OracleIcp's align / align_batch with a rejector chain."""

    def __init__(self, target: np.ndarray, normals=None, wide_accum: bool = False):
        self.L = _lib()
        self.t = np.ascontiguousarray(target, np.float32)
        self.n = np.ascontiguousarray(normals, np.float32) if normals is not None else None
        self.h = self.L.orc_icp_chain_create()
        icp = self.L.orc_icp_chain_as_icp(self.h)
        self.L.orc_icp_set_wide_accum(icp, int(wide_accum))
        self.L.orc_icp_set_target(icp, self.t.ctypes.data, self.t.shape[0], self.t.strides[0],
                                  self.n.ctypes.data if self.n is not None else None,
                                  self.n.strides[0] if self.n is not None else 0)

    def __del__(self):
        try:
            self.L.orc_icp_chain_destroy(self.h)
        except Exception:
            pass

    def align(self, source: np.ndarray, guess=None, params: IcpParams | None = None, trace_cap: int = 0, chain=()):
        s = np.ascontiguousarray(source, np.float32)
        prm = params or default_params()
        g = np.ascontiguousarray(np.asarray(guess, np.float32).T) if guess is not None else None  # -> column-major
        res = IcpResult()
        aligned = np.empty((s.shape[0], 4), np.float32)
        idx = np.empty(s.shape[0], np.int32)
        d2 = np.empty(s.shape[0], np.float32)
        tT = np.zeros((max(trace_cap, 1), 16), np.float32)
        tm = np.zeros(max(trace_cap, 1), np.float64)
        tn = C.c_size_t(0)
        arr, n_chain = rejector_chain(chain)
        self.L.orc_icp_align_ex(self.h, s.ctypes.data, s.shape[0], s.strides[0], g.ctypes.data if g is not None else None,
                                C.byref(prm), arr, n_chain, C.byref(res), aligned.ctypes.data, idx.ctypes.data,
                                d2.ctypes.data, tT.ctypes.data if trace_cap else None,
                                tm.ctypes.data if trace_cap else None, trace_cap, C.byref(tn))
        out = {"result": res, "aligned": aligned, "corr_idx": idx, "corr_d2": d2}
        if trace_cap:
            k = tn.value
            out["trace_T"] = tT[:k].reshape(k, 4, 4).transpose(0, 2, 1).copy()
            out["trace_mse"] = tm[:k].copy()
        return out

    def align_batch(self, source: np.ndarray, guesses: np.ndarray, params: IcpParams | None = None, threads: int = 0,
                    chain=()):
        s = np.ascontiguousarray(source, np.float32)
        prm = params or default_params()
        g = np.ascontiguousarray(np.asarray(guesses, np.float32).transpose(0, 2, 1)).reshape(-1, 16)
        H = g.shape[0]
        res = (IcpResult * H)()
        arr, n_chain = rejector_chain(chain)
        self.L.orc_icp_align_batch_ex(self.h, s.ctypes.data, s.shape[0], s.strides[0], g.ctypes.data, H, C.byref(prm),
                                      arr, n_chain, res, threads)
        return list(res)
