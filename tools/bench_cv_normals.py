"""Time computeNormalsPC3d (peb_cv_normals, DESIGN.md §13) against PCL's NormalEstimation (peb_normals_knn) at k = 20 on
the C2 scene and write one JSON line to OUT/bench_cv_normals.json.

- device: peb_cv_normals_dev and peb_normals_knn_dev on the same device-resident scene, alternated in rounds (one round =
  --reps calls of one entry point between two CUDA events on the context's stream; both entry points build their grid
  in every call, as a user's call does).  Median and spread of the per-call time over the rounds.
- end to end: peb_cv_normals from host buffers (upload, grid, normals, download), host clock around the blocking call.
- CPU: the oracle's restatement (tests/cv_normals_oracle.cpp : orc_cv_normals, timing build) on 1 thread and on all cores.
The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_cv_normals.py --out OUT_DIR [--rounds 10] [--reps 50]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.dont_write_bytecode = True

K = 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the timing does not depend on it
        return f"unknown ({e})"


def spread(ms):
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "samples": len(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--e2e-runs", type=int, default=20)
    ap.add_argument("--cpu-runs", type=int, default=3)
    args = ap.parse_args()
    import torch

    import cv_normals_oracle as cvo
    from pose_estimation_b200 import pcl
    from pose_estimation_b200.testing import synth

    info = card()
    ctx = pcl.Context(0)

    def downsample(points, leaf):
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    scene = np.ascontiguousarray(synth.make_c2(downsample=downsample).target[:, :3], np.float32)
    n = len(scene)
    vp = np.zeros(3, np.float32)
    d_in = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
    d_in[:, :3] = torch.from_numpy(scene).cuda()
    d_cv = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    d_pcl = torch.empty((n, 8), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(ctx.stream, device=0)
    calls = {
        "cv_normals_dev": lambda: ctx.check(pcl.lib.peb_cv_normals_dev(ctx.handle, d_in.data_ptr(), n, K, 1, vp.ctypes.data,
                                                                       d_cv.data_ptr())),
        "normals_knn_dev": lambda: ctx.check(pcl.lib.peb_normals_knn_dev(ctx.handle, d_in.data_ptr(), n, K, vp.ctypes.data,
                                                                         d_pcl.data_ptr())),
    }
    for fn in calls.values():  # warm-up: module load, grid buffers
        for _ in range(5):
            fn()
    ctx.sync()
    per_call = {name: [] for name in calls}
    for _ in range(args.rounds):
        for name, fn in calls.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(args.reps):
                fn()
            b.record(stream)
            b.synchronize()
            per_call[name].append(a.elapsed_time(b) / args.reps)
    device = {name: spread(ms) for name, ms in per_call.items()}
    ratio = device["cv_normals_dev"]["ms_median"] / device["normals_knn_dev"]["ms_median"]

    # the device entry and the host entry give the same bytes
    host_out = pcl.compute_normals_pc3d(scene, K, True, vp, ctx=ctx)
    same_bytes = bool(np.array_equal(host_out.view(np.uint32), d_cv.cpu().numpy().view(np.uint32)))
    e2e = []
    for _ in range(3):
        pcl.compute_normals_pc3d(scene, K, True, vp, ctx=ctx)
    for _ in range(args.e2e_runs):
        t = time.perf_counter()
        pcl.compute_normals_pc3d(scene, K, True, vp, ctx=ctx)
        e2e.append((time.perf_counter() - t) * 1e3)

    cvo._lib("timing")  # compiled before the clock starts
    cores = os.cpu_count() or 1
    cpu = {}
    for label, threads in (("1_thread", 1), ("all_cores", cores)):
        ms = []
        for _ in range(args.cpu_runs):
            t = time.perf_counter()
            cvo.cv_normals(scene, K, threads=threads, build="timing")
            ms.append((time.perf_counter() - t) * 1e3)
        cpu[label] = spread(ms)
    cpu["cores"] = cores
    cpu["oracle_build"] = "timing (-O3 -march=x86-64-v3)"

    out = {"card": info, "k": K, "scene": "C2 (synth.make_c2, CUDA VoxelGrid)", "n_points": n,
           "device_per_call": device, "cv_over_pcl_device": ratio, "rounds": args.rounds, "reps_per_round": args.reps,
           "host_buffer_end_to_end": spread(e2e), "dev_equals_host_bytes": same_bytes, "cpu_oracle": cpu,
           "card_after": card()}
    Path(args.out).mkdir(parents=True, exist_ok=True)
    line = json.dumps(out)
    (Path(args.out) / "bench_cv_normals.json").write_text(line + "\n")
    print(line)
    ctx.close()


if __name__ == "__main__":
    main()
