"""GeneralizedIterativeClosestPoint on one GPU: C2 single align, C4 batches, covariance time, and the pose errors of GICP,
point-to-point and point-to-plane ICP from the same C4 guesses.  Writes profiles/gicp_<tag>.json (or --out) and prints it.
The card's name, power limit and SM clock are read in the same run and stored beside the numbers."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from pose_estimation_b200 import pcl  # noqa: E402
from pose_estimation_b200.testing import synth  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, reps):
    fn()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()  # every entry point ends in a stream synchronise
        t.append(time.perf_counter() - t0)
    return float(np.median(t)), [float(v) for v in t]


def errors(records_T, gt):
    e = [synth.pose_error(np.asarray(T, np.float64), gt) for T in records_T]
    rot = np.array([a for a, _ in e])
    tr = np.array([b for _, b in e])
    return {"rot_median_rad": float(np.median(rot)), "trans_median_m": float(np.median(tr)),
            "rot_p90_rad": float(np.percentile(rot, 90)), "trans_p90_m": float(np.percentile(tr, 90))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--max-corr-dist", type=float, default=0.02)  # bench.py's
    ap.add_argument("--out", default=str(ROOT / "profiles" / "gicp_bench.json"))
    a = ap.parse_args()
    out = {"card": card(), "reps": a.reps, "max_corr_dist": a.max_corr_dist}
    ctx = pcl.Context(0)

    def downsample(points, leaf):  # the scenes are voxel-filtered on the device, as bench.py does
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    c2 = synth.make_c2(downsample=downsample)
    g = pcl.GeneralizedIterativeClosestPoint(ctx)
    g.setMaxCorrespondenceDistance(a.max_corr_dist)
    g.setInputSource(c2.source)
    g.setInputTarget(c2.target)

    def cov():
        g.setInputSource(c2.source)  # clears the cached covariances of both clouds
        g.setInputTarget(c2.target)
        g.covariances("source")

    out["covariances_s"], _ = timed(cov, a.reps)
    guess = c2.guess if c2.guess.ndim == 2 else c2.guess[0]
    out["c2_single_s"], out["c2_single_all_s"] = timed(lambda: g.align(guess, want_output=False), a.reps)
    out["c2_single_iterations"] = g.nr_iterations_
    out["c2_sizes"] = [len(c2.source), len(c2.target)]
    c4 = synth.make_c4(downsample=downsample)
    g.setInputSource(c4.source)
    g.setInputTarget(c4.target)
    for H in (128, 1024):
        t, _ = timed(lambda: g.alignBatch(c4.guess[:H]), max(1, a.reps // 2))
        out[f"c4_batch{H}_s"] = t
        out[f"c4_batch{H}_hyp_per_s"] = H / t
    recs = g.alignBatch(c4.guess[:128])
    out["gicp_errors"] = errors([pcl.result_matrix(r) for r in recs], c4.gt_pose)
    out["gicp_iterations_median"] = float(np.median([r.iterations for r in recs]))
    icp = pcl.IterativeClosestPoint(ctx)
    icp.setInputSource(c4.source)
    icp.setInputTarget(c4.target)
    icp.setMaxCorrespondenceDistance(a.max_corr_dist)
    icp.setMaximumIterations(30)
    out["point_to_point_errors"] = errors([pcl.result_matrix(r) for r in icp.alignBatch(c4.guess[:128])], c4.gt_pose)
    icpn = pcl.IterativeClosestPointWithNormals(ctx)
    icpn.setInputSource(c4.source)
    nrm = pcl.NormalEstimation(ctx)
    nrm.setInputCloud(c4.target)
    nrm.setKSearch(30)
    icpn.setInputTarget(c4.target, nrm.compute()[:, :3])
    icpn.setMaxCorrespondenceDistance(a.max_corr_dist)
    icpn.setMaximumIterations(30)
    out["point_to_plane_errors"] = errors([pcl.result_matrix(r) for r in icpn.alignBatch(c4.guess[:128])], c4.gt_pose)
    out["guess_errors"] = errors(c4.guess[:128], c4.gt_pose)
    ctx.close()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(out, indent=1))
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
