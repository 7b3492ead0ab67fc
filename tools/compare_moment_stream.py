"""Compare two builds of the library on the flagship workload in one run: the moment launch, the step, the records.

For each build (a PEB_LIB_VARIANT name; "" is libpe_b200.so), alternated `--rounds` times, this runs
  - tools/profile_split_launches.py (C4 at profile level 2: per-iteration search_ms and moment_ms), and
  - bench.py --gpus 1 --no-cpu-baseline --no-inproc --dump-outputs (the C4 value, C2 align_ms and the C4 records),
then compares every --dump-outputs field of every run with the first build's first run and reports the moment launch's
algorithmic stream rate: 16 bytes per query (the working point, read once) x hypotheses x source points / moment_ms,
against the 6 545 GB/s HBM peak bench.py uses.  Builds listed with --profile-only get the profile run only (sweeps).
The card's name, power limit and SM clock are read with nvidia-smi before and after.  Writes OUT/moment_stream.json.

    python tools/compare_moment_stream.py --out OUT --builds parent "" [--profile-only r2 r8] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
PEAK_GBS = 6545.0


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active",
                        "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    return r.stdout.strip().splitlines()[0] if r.stdout.strip() else f"unknown ({r.stderr.strip()})"


def run(cmd, variant, log):
    env = dict(os.environ, PEB_LIB_VARIANT=variant)
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    log.write(f"$ PEB_LIB_VARIANT={variant} {' '.join(cmd)}\n{r.stdout}\n{r.stderr[-4000:]}\n")
    if r.returncode != 0:
        raise RuntimeError(f"{cmd} ({variant!r}) exited {r.returncode}:\n{r.stderr[-4000:]}")
    return r.stdout


def profile(variant, out, log):
    run([sys.executable, "tools/profile_split_launches.py", "--out", str(out)], variant, log)
    return json.loads((out / "split_launches.json").read_text())


def bench(variant, out, steps, warmup, log):
    text = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                "--no-cpu-baseline", "--no-inproc", "--dump-outputs", str(out)], variant, log)
    line = [ln for ln in text.splitlines() if ln.startswith("{")][-1]
    return json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--builds", nargs="+", required=True, help="PEB_LIB_VARIANT names, the reference first ('' = default)")
    ap.add_argument("--profile-only", nargs="*", default=[])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    log = open(out / "moment_stream.log", "w")
    report = {"card_before": card(), "peak_gbs": PEAK_GBS, "rounds": []}
    ref_dump = None
    for rnd in range(args.rounds):
        entry = {}
        for b in args.builds + (args.profile_only if rnd == 0 else []):
            name = b or "default"
            prof = profile(b, out / f"prof_{name}_{rnd}", log)
            queries = prof["hypotheses"] * prof.get("n_src", 0)
            rows = prof["per_iteration"]
            warm = [r["moment_ms"] for r in rows[2:]]
            e = {"moment_ms_total": prof["moment_ms_total"], "search_ms_total": prof["search_ms_total"],
                 "moment_ms_warm_median": statistics.median(warm) if warm else None,
                 "moment_ms": [r["moment_ms"] for r in rows], "search_ms": [r["search_ms"] for r in rows]}
            if queries and warm:
                e["moment_stream_gbs"] = round(16.0 * queries / (e["moment_ms_warm_median"] * 1e-3) / 1e9, 1)
                e["moment_share_of_peak"] = round(e["moment_stream_gbs"] / PEAK_GBS, 3)
            if b in args.builds:
                dump = out / f"dump_{name}_{rnd}"
                res = bench(b, dump, args.steps, args.warmup, log)
                e["bench"] = res
                e["value"] = res.get("value")
                e["align_ms"] = res.get("align_ms")
                fields = {p.stem: np.load(p) for p in sorted(dump.glob("*.npy"))}
                if ref_dump is None:
                    ref_dump = fields
                e["records_equal_reference"] = bool(fields) and sorted(fields) == sorted(ref_dump) and all(
                    np.array_equal(fields[k].view(np.uint8), ref_dump[k].view(np.uint8)) for k in fields)
                e["fields_differing"] = [k for k in fields if k not in ref_dump or
                                         not np.array_equal(fields[k].view(np.uint8), ref_dump[k].view(np.uint8))]
            entry[name] = e
            print(f"round {rnd} {name:>8}: moment {e['moment_ms_total']:.3f} ms/step (warm median "
                  f"{e['moment_ms_warm_median']}, {e.get('moment_stream_gbs')} GB/s), search {e['search_ms_total']:.3f}"
                  + (f", value {e['value']}, align_ms {e['align_ms']}, records equal: {e['records_equal_reference']}"
                     if "bench" in e else ""), flush=True)
        report["rounds"].append(entry)
    report["card_after"] = card()
    (out / "moment_stream.json").write_text(json.dumps(report, indent=1) + "\n")
    print(f"# {report['card_before']}\n# {report['card_after']}")


if __name__ == "__main__":
    main()
