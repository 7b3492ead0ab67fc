"""Time the search and the moment launch of every split ICP iteration of the C4 batch separately.

Profile level 2 of the library puts both launches of an iteration between the same pair of events, so its per-iteration
times are their sum.  This script runs bench.py's C4 workload (synth.make_c4, VoxelGrid downsampling on the device, 30
iterations, the 2 cm correspondence threshold, `--hyp` hypotheses) at profile level 2 under torch.profiler with CUDA
activities and reads every icp_search_kernel<...> and icp_moment_kernel<...> from the trace.  Profile level 2 runs one
chain of launches, so launch k of each kind belongs to iteration k.  The moment launch is issued with programmatic
dependent launch and its blocks may wait while the search drains, so it is reported twice: `moment_ms` counts from the
end of its search launch (or its own start, if later) and `moment_span_ms` is the kernel's whole duration.

The card's name, power limit and SM clocks are read with nvidia-smi in the same run.  Writes OUT/split_launches.json
and prints a table.

    python tools/profile_split_launches.py --out OUT_DIR [--hyp 1024] [--warmup 2] [--steps 3]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import re
import statistics
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

import bench  # noqa: E402  (the workloads and the ICP settings of the flagship benchmark)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the timing does not depend on it
        return f"unknown ({e})"


def kernels(trace_path):
    """-> [(start_us, end_us, "search" | "moment", kernel name)] of one trace, in launch order"""
    events = json.loads(Path(trace_path).read_text())["traceEvents"]
    out = []
    for e in events:
        if e.get("cat") != "kernel":
            continue
        name = e["name"]
        kind = "search" if "icp_search_kernel<" in name else "moment" if "icp_moment_kernel<" in name else None
        if kind:
            out.append((float(e["ts"]), float(e["ts"]) + float(e["dur"]), kind, name))
    out.sort()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--hyp", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    from pose_estimation_b200 import _lib, pcl

    info = card()
    ctx = pcl.Context(0)

    def downsample(points, leaf):
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    c4, _ = bench.make_workloads(downsample, False, args.hyp, 1.0)
    params = pcl.IcpParams()
    _lib.lib.peb_icp_params_default(C.byref(params))
    params.max_iterations = bench.ITERATIONS
    params.abs_mse_threshold = -1.0
    params.max_corr_dist = bench.MAX_CORR_DIST
    ctx.target_set(c4.target)
    ctx.source_set(c4.source)
    g = bench.col_major(c4.guess)
    res = (_lib.IcpResult * len(c4.guess))()
    ctx.set_int("profile", 2)

    def step():
        ctx.check(_lib.lib.peb_icp_align_batch(ctx.handle, g.ctypes.data, len(c4.guess), C.byref(params), res))

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    steps = []
    with tempfile.TemporaryDirectory() as tmp:
        for s in range(args.steps):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step()
                torch.cuda.synchronize()
            path = Path(tmp) / f"step{s}.json"
            prof.export_chrome_trace(str(path))
            steps.append(kernels(path))
    ctx.close()

    rows = []
    for it in range(bench.ITERATIONS):
        search, moment, span, names = [], [], [], set()
        for ks in steps:
            se = [k for k in ks if k[2] == "search"]
            mo = [k for k in ks if k[2] == "moment"]
            if it >= len(se) or it >= len(mo):
                continue
            s0, s1, _, sn = se[it]
            m0, m1, _, _ = mo[it]
            search.append((s1 - s0) / 1e3)
            moment.append((m1 - max(m0, s1)) / 1e3)
            span.append((m1 - m0) / 1e3)
            names.add(re.search(r"icp_search_kernel<[^>]*>", sn).group(0))
        if search:
            rows.append({"iteration": it, "search_ms": round(statistics.median(search), 4),
                         "moment_ms": round(statistics.median(moment), 4),
                         "moment_span_ms": round(statistics.median(span), 4), "search_kernel": sorted(names)})
    out = {"card": info, "card_after": card(), "workload": "C4", "hypotheses": len(c4.guess), "n_src": len(c4.source),
           "iterations": bench.ITERATIONS, "steps": args.steps, "statistic": "median over steps",
           "profile_level": 2, "per_iteration": rows,
           "search_ms_total": round(sum(r["search_ms"] for r in rows), 3),
           "moment_ms_total": round(sum(r["moment_ms"] for r in rows), 3)}
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "split_launches.json").write_text(json.dumps(out) + "\n")
    print(f"# {info}")
    print(f"{'it':>3} {'search_ms':>10} {'moment_ms':>10} {'span_ms':>9}  search kernel")
    for r in rows:
        print(f"{r['iteration']:>3} {r['search_ms']:>10.4f} {r['moment_ms']:>10.4f} {r['moment_span_ms']:>9.4f}  {r['search_kernel'][0]}")
    print(f"total search {out['search_ms_total']} ms, moment {out['moment_ms_total']} ms")


if __name__ == "__main__":
    main()
