"""The GeneralizedIterativeClosestPoint interfaces outside Python: the C part of include/pe_b200.h compiles as pedantic C99
and links from C (tests/c/gicp_abi_check.c), the C++ facade class compiles with plain g++, and on the B200 the facade
gives the records of the Python class (tests/cpp/gicp_facade_check.cpp).  Executables are built into a temporary directory."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from pose_estimation_b200.testing import synth

ROOT = Path(__file__).resolve().parents[1]
LIB_DIR = ROOT / "pose_estimation_b200"


def _gpu():
    import torch

    return torch.cuda.is_available()


def test_gicp_header_is_plain_c99(tmp_path):
    exe = tmp_path / "gicp_abi_check"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", str(ROOT / "include"),
                        str(ROOT / "tests" / "c" / "gicp_abi_check.c"), "-o", str(exe), "-L", str(LIB_DIR), "-lpe_b200", "-lm",
                        f"-Wl,-rpath,{LIB_DIR}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    if _gpu():
        assert r.returncode == 0 and "ctx ok" in r.stdout, r.stdout
    else:
        assert r.returncode == 10 and "no CPU fallback" in r.stdout, r.stdout


@pytest.fixture(scope="module")
def facade_exe(tmp_path_factory):
    exe = tmp_path_factory.mktemp("gicp_facade") / "gicp_facade_check"
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "cpp" / "gicp_facade_check.cpp"), "-o", str(exe), "-L", str(LIB_DIR), "-lpe_b200",
           f"-Wl,-rpath,{LIB_DIR}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def _case(tmp_path):
    prob = synth.make_c1(3000, seed=5)
    rng = np.random.default_rng(9)
    guesses = np.stack([synth.perturb_pose(prob.gt_pose, rng, 1.0, 0.002) for _ in range(5)]).astype(np.float32)
    paths = [tmp_path / n for n in ("src.bin", "tgt.bin", "guesses.bin", "out.bin")]
    paths[0].write_bytes(np.ascontiguousarray(prob.source, np.float32).tobytes())
    paths[1].write_bytes(np.ascontiguousarray(prob.target, np.float32).tobytes())
    paths[2].write_bytes(np.ascontiguousarray(guesses.transpose(0, 2, 1)).tobytes())  # column-major
    return prob, guesses, paths


def test_gicp_facade_builds_and_fails_loudly_without_gpu(facade_exe, tmp_path):
    if _gpu():
        pytest.skip("GPU present: covered by the gpu test")
    _, _, paths = _case(tmp_path)
    r = subprocess.run([str(facade_exe), *map(str, paths)], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stdout, r.stdout


@pytest.mark.gpu
def test_gicp_facade_gives_the_python_records(facade_exe, tmp_path):
    from pose_estimation_b200 import pcl

    prob, guesses, paths = _case(tmp_path)
    r = subprocess.run([str(facade_exe), *map(str, paths)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = paths[3].read_bytes()
    rec = 96
    assert len(raw) == rec * (1 + len(guesses))
    with pcl.Context(0) as ctx:
        g = pcl.GeneralizedIterativeClosestPoint(ctx)
        g.setInputSource(prob.source)
        g.setInputTarget(prob.target)
        g.setMaxCorrespondenceDistance(0.05)
        g.setMaximumIterations(30)
        g.align(guesses[0])
        assert raw[:rec] == bytes(g.result)
        batch = g.alignBatch(guesses)
        assert raw[rec:] == b"".join(bytes(x) for x in batch)
