"""Time OpenCVSurfaceMatch::find_object_in_scene as one call (peb_surface_match) against the same request made of the step
entry points (peb_scene_prepare, peb_cv_normals, peb_ppf_match, peb_cvicp_register; selection and packing on the host), and
write one JSON line to OUT/bench_surface_match.json.

Workloads, both from the organised 1944 x 1200 C2 cloud (synth.render_scene as synth.make_c2 renders it) with NaN removal
and one plane removal, then find_object_in_scene with the reference's parameters (peb_surface_match_params_default):
  - "reference": no VoxelGrid, as the reference runs it;
  - "c2_leaf":   VoxelGrid with the bench's C2 leaf.
In each workload the two forms run alternately in the same process, wall clock around each blocking request (the one call
does not ask for the scene back).  Recorded: the card's name, power limit and maximum SM clock (read in the same run), the
scene sizes, whether both forms give the same bytes, and the bytes of the cloud-sized transfers over PCIe of each form,
computed from the shapes (the small transfers both forms share — the PPF raw poses, the cv ICP's per-iteration pose
tables and sums — are left out).

    python tools/bench_surface_match.py --out OUT_DIR [--runs 7]
"""
from __future__ import annotations

import argparse
import ctypes
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the timing does not depend on it
        return f"unknown ({e})"


def spread(ms):
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "samples": len(ms)}


def same(one, ref) -> bool:
    refined, best, pose7, n_results, scene = one
    s_scene, s_refined, s_best, s_pose7, s_n = ref
    return (scene.tobytes() == s_scene.tobytes() and (best, n_results, len(refined)) == (s_best, s_n, len(s_refined))
            and all(bytes(a) == bytes(b) for a, b in zip(refined, s_refined)) and pose7.tobytes() == s_pose7.tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=7)
    args = ap.parse_args()
    from pose_estimation_b200 import pcl
    from pose_estimation_b200._lib import PpfPose
    from pose_estimation_b200.testing import surface_match, synth

    info = card()
    ctx = pcl.Context(0)
    prob = synth.make_c2()  # the organised cloud and the bench's C2 leaf (no down-sampling here)
    cloud = np.ascontiguousarray(prob.organized, np.float32)
    rng = np.random.default_rng(2)
    mp, mn = synth.Surface(2).sample(50000, rng)  # the C2 object with its normals
    model6 = np.concatenate([mp, mn], 1).astype(np.float32)
    det = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=ctx)
    det.trainModel(model6)
    params = pcl.surface_match_params()
    out = {"card": info, "scene": "C2 organised 1944 x 1200 (synth.make_c2), NaN removal + 1 plane removal",
           "model_rows": len(model6), "params": "peb_surface_match_params_default (k 20, match 1.0 / 0.03, 6 x ICP(250, 0.005, 2.5, 8))",
           "runs": args.runs, "workloads": {}}
    for name, leaf in (("reference", 0.0), ("c2_leaf", float(prob.leaf))):
        prep = dict(prepare=True, num_planes=1, leaf=leaf)
        one = pcl.find_object_in_scene(det, cloud, params, return_scene=True, **prep)
        ref = surface_match.steps(ctx, det, model6, cloud, params, **prep)
        t_one, t_steps = [], []
        for _ in range(args.runs):
            t0 = time.perf_counter()
            pcl.find_object_in_scene(det, cloud, params, **prep)
            t1 = time.perf_counter()
            surface_match.steps(ctx, det, model6, cloud, params, **prep)
            t2 = time.perf_counter()
            t_one.append((t1 - t0) * 1e3)
            t_steps.append((t2 - t1) * 1e3)
        n, m = len(cloud), len(ref[0])
        n_ref = len(ref[1])
        pose_bytes = n_ref * ctypes.sizeof(PpfPose)
        out["workloads"][name] = {
            "leaf": leaf, "n_input": n, "n_prepared": m, "n_results": ref[4], "n_refined": n_ref, "best": ref[2],
            "one_call": spread(t_one), "steps": spread(t_steps),
            "steps_over_one_call": statistics.median(t_steps) / statistics.median(t_one),
            "equal_bytes": same(one, ref),
            "pcie_bytes": {
                # input up once; the result record and the refined poses down
                "one_call": {"up": n * 16, "down": 48 + pose_bytes},
                # prepare: cloud up, prepared down; normals: up, scene rows down; match: rows up (pageable); cv ICP: model and
                # scene rows up (pageable); refined poses stay on the host
                "steps": {"up": n * 16 + m * 16 + m * 24 + len(model6) * 24 + m * 24, "down": m * 16 + m * 24},
            },
        }
    out["card_after"] = card()
    line = json.dumps(out)
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "bench_surface_match.json").write_text(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
