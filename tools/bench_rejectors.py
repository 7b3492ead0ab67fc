"""Time ICP with correspondence rejector chains on one GPU and write one JSON line to OUT/bench_rejectors.json.

C2 single align and C4 1024-hypothesis batch (bench.py's workloads and ICP settings), for: no chain, OneToOne,
Median(1.0), Trimmed(0.8), Distance -> OneToOne -> Median.  Every case is warmed up, then timed N times (CUDA events
on the context's stream around the blocking call); the median is reported.  The card's name and power limit are read
in the same run.  With --per-launch, one more C4 run per case with profile level 2 gives the device time of every
iteration (search + reject + moment launches between the same events).

    python tools/bench_rejectors.py --out OUT_DIR [--runs 20] [--hyp 1024]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

import bench  # noqa: E402  (the workloads and the ICP settings of the flagship benchmark)

CHAINS = {
    "none": [],
    "one_to_one": [(2,)],
    "median_1.0": [(1, 1.0)],
    "trimmed_0.8": [(3, 0.8)],
    "distance_one_to_one_median": [(0, 0.005), (2,), (1, 1.0)],
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the timing does not depend on it
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--hyp", type=int, default=1024)
    ap.add_argument("--per-launch", action="store_true")
    args = ap.parse_args()
    import torch

    from pose_estimation_b200 import _lib, pcl

    info = card()
    ctx = pcl.Context(0)

    def downsample(points, leaf):
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    c4, c2 = bench.make_workloads(downsample, True, args.hyp, 1.0)
    params = pcl.IcpParams()
    _lib.lib.peb_icp_params_default(C.byref(params))
    params.max_iterations = bench.ITERATIONS
    params.abs_mse_threshold = -1.0
    params.max_corr_dist = bench.MAX_CORR_DIST
    stream = torch.cuda.ExternalStream(ctx.stream, device=0)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        ms = []
        for _ in range(args.runs):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            ms.append(a.elapsed_time(b))
        return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "runs": len(ms)}

    def align_fn(prob, chain, batch):
        ctx.target_set(prob.target)
        ctx.source_set(prob.source)
        arr, n = _lib.rejector_array(chain)
        if batch:
            g = bench.col_major(prob.guess)
            res = (_lib.IcpResult * len(prob.guess))()

            def run():
                ctx.check(_lib.lib.peb_icp_align_batch_ex(ctx.handle, g.ctypes.data, len(prob.guess), C.byref(params),
                                                          arr, n, res))
        else:
            g = bench.col_major(prob.guess[None] if prob.guess.ndim == 2 else prob.guess[:1])
            res = _lib.IcpResult()

            def run():
                ctx.check(_lib.lib.peb_icp_align_ex(ctx.handle, g.ctypes.data, C.byref(params), arr, n, C.byref(res),
                                                    None, None, None))
        return run

    out = {"card": info, "iterations": bench.ITERATIONS, "max_corr_dist_m": bench.MAX_CORR_DIST,
           "c2_target_pts": len(c2.target), "c4_target_pts": len(c4.target), "c4_hypotheses": len(c4.guess), "cases": {}}
    for name, chain in CHAINS.items():
        c2r = timed(align_fn(c2, chain, False))
        c4r = timed(align_fn(c4, chain, True))
        c4r["hypotheses_per_s"] = len(c4.guess) / (c4r["ms_median"] / 1e3)
        out["cases"][name] = {"c2_single_align": c2r, "c4_batch": c4r}
        print(name, json.dumps(out["cases"][name]), flush=True)
        if args.per_launch:
            ctx.set_int("profile", 2)
            align_fn(c4, chain, True)()
            n_ms = C.c_size_t(0)
            buf = (C.c_float * 256)()
            ctx.check(_lib.lib.peb_profile_read(ctx.handle, buf, 256, C.byref(n_ms)))
            out["cases"][name]["c4_per_iteration_ms_profile2"] = [round(buf[i], 4) for i in range(n_ms.value)]
            ctx.set_int("profile", 0)
    out["card_after"] = card()
    Path(args.out).mkdir(parents=True, exist_ok=True)
    line = json.dumps(out)
    (Path(args.out) / "bench_rejectors.json").write_text(line + "\n")
    print(line)
    ctx.close()


if __name__ == "__main__":
    main()
