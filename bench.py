#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on synthetic clouds of BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on rank 0.  metric = ICP hypotheses/s (whole job) on configs[3] — 1024 initial
poses x 50k-pt model vs ~500k-pt scene, 30 point-to-point iterations, hypotheses sharded over
the ranks — and, at N = 1, the single-align latency of configs[1] (200k scene / 50k model,
30 iterations) beside it as `align_ms`.  A "step" is one pass of the hot path over the whole
batch of hypotheses.  See DESIGN.md ("Measurement") for every key.

--dump-outputs DIR writes the result records of the last timed step, one DIR/<field>.npy per field of
peb_icp_result in hypothesis order (float32 / float64), so that two builds can be compared output for
output: the inputs are seeded and identical from run to run.

The benchmark writes nothing into the repository tree (which may be read-only): it expects the
native libraries that build() compiled and writes no bytecode cache.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # no __pycache__ of the project's modules in the tree

ITERATIONS = 30
MAX_CORR_DIST = 0.02
N_HYP = 1024
ALG_BYTES_PER_QUERY = 40  # SURVEY.md 8d: 16 read source + 16 gather matched target + 8 write correspondence
DUMP_BYTES_MAX = 64 << 20
HBM_PEAK_GBS = 6544.7  # measured HBM bandwidth of one B200 (power limit not recorded): the roofline denominator of BASELINE.md


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------
def make_workloads(downsample, want_c2: bool, n_hyp: int, scale: float):
    from pose_estimation_b200.testing import synth

    t0 = time.perf_counter()
    # PEB_HYP_OFFSET (development): the block of n_hyp hypotheses that starts at this index of the full sequence — the
    # share of one rank of an N-GPU run, alone on one GPU
    off = int(os.environ.get("PEB_HYP_OFFSET", "0"))
    c4 = synth.make_c4(scale=scale, n_guesses=off + n_hyp, downsample=downsample)
    if off:
        c4.guess = c4.guess[off:]
    c2 = synth.make_c2(scale=scale, downsample=downsample) if want_c2 else None
    log(f"[bench] workloads generated in {time.perf_counter() - t0:.1f} s: C4 target {len(c4.target)} pts, "
        f"model {len(c4.source)} pts, {len(c4.guess)} poses" + (f"; C2 target {len(c2.target)} pts" if c2 else ""))
    return c4, c2


def col_major(guesses: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(guesses, np.float32).reshape(-1, 4, 4).transpose(0, 2, 1)).reshape(-1, 16)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU, sampled DURING the timed region: NVML in a thread (a sample
    every ~5 ms, so that even an 80 ms 8-GPU run is covered); `nvidia-smi -lms` if NVML is not importable."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines: list[str] = []
        self.nvml = None
        self.samples: list[tuple[int, int]] = []
        self.max_mhz = None
        self.stop_flag = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            try:  # CUDA_VISIBLE_DEVICES re-numbers CUDA devices, not NVML's: go by UUID
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    why = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    why = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((int(mhz), int(why)))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            sm = [m for m, _ in self.samples]
            reasons = set()
            for _, why in self.samples:
                for bit, nm in self.NVML_REASONS.items():
                    if why & bit:
                        reasons.add(nm)
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons),
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ---------------------------------------------------------------------------------------------
# the CPU arm: the oracle's timing build (PCL 1.10 restatement, single kd-tree, exact search),
# OpenMP over hypotheses like cv::ppf_match_3d::ICP::registerModelToScene
# ---------------------------------------------------------------------------------------------
def cpu_params():
    from oracle import default_params

    return default_params(max_iterations=ITERATIONS, abs_mse_threshold=-1.0, max_corr_dist=MAX_CORR_DIST)


def host_threads() -> int:
    """Host cores this process may use (torchrun pins OMP_NUM_THREADS to 1; the oracle takes an explicit count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_batch_rate(orc_icp, source, guesses, threads: int, n: int) -> tuple[float, float]:
    g = guesses[:n]
    t0 = time.perf_counter()
    orc_icp.align_batch(source, g, cpu_params(), threads=threads)
    dt = time.perf_counter() - t0
    return n / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import Oracle

    orc = Oracle(fast=True)
    slow = Oracle()
    cores = host_threads()
    c4, _ = make_workloads(lambda p, leaf: slow.voxel_grid(p, leaf)[0], False, N_HYP, args.scale)
    icp = orc.icp(c4.target)
    # calibrate the per-step sample so that the whole run stays within ~150 s
    rate0, dt0 = cpu_batch_rate(icp, c4.source, c4.guess, cores, cores)
    budget = 150.0 / max(args.steps + args.warmup, 1)
    sample = int(max(cores, min(N_HYP, (budget * rate0) // cores * cores)))
    log(f"[bench] reference arm: {cores} threads, calibration {cores} hypotheses in {dt0:.1f} s, sample {sample}/step")
    for _ in range(args.warmup):
        cpu_batch_rate(icp, c4.source, c4.guess, cores, sample)
    t_total = 0.0
    for _ in range(args.steps):
        _, dt = cpu_batch_rate(icp, c4.source, c4.guess, cores, sample)
        t_total += dt
    value = sample * args.steps / t_total
    line = {
        "impl": "reference", "metric": "icp_hypotheses_per_s", "value": value, "unit": "hypotheses/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the SAME config as the CUDA arm's line (the workload); a step of this arm is a bounded sample of it, named in
        # cpu_baseline.sample, and `value` is a rate, so the two lines compare directly
        "config": workload_config(c4, N_HYP),
        "cpu_baseline": {"value": value, "unit": "hypotheses/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} of the {N_HYP} hypotheses per step ({cores} host threads; the ratio to the CUDA arm "
                                   f"depends on the host: round 1 saw 354x on a 16-core and 188x on a 32-core box), OpenMP over hypotheses, "
                                   f"oracle timing build (-O3 AVX2/FMA), PCL 1.10 restatement: real PCL is not installable here"},
        "e2e": {"value": value, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(c4, hyp_per_step):
    return {
        "workload": "C4 (BASELINE.json configs[3]): multi-hypothesis refinement, one 50k-pt model vs one voxel-down-sampled "
                    "1944x1200 organized scene, point-to-point ICP",
        "hypotheses": int(hyp_per_step), "n_source": int(len(c4.source)), "n_target": int(len(c4.target)),
        "iterations": ITERATIONS, "max_corr_dist_m": MAX_CORR_DIST, "leaf_m": float(c4.leaf),
        "sharding": "contiguous blocks of hypotheses per rank, replicated scene grid, all_gather of 96-byte result records",
        "l2": "flushed (256 MiB write) before every timed step",
    }


# ---------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from pose_estimation_b200 import pcl
    from pose_estimation_b200.pcl import lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    park = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        park = dist.new_group(backend="gloo")  # host-side barrier: ranks parked on it leave their GPU idle
    ctx = pcl.Context(local)
    for kv in filter(None, os.environ.get("PEB_OPTS", "").split(",")):  # development: library tuning knobs
        k, v = kv.split("=")
        ctx.set_int(k, int(v))
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def downsample(points, leaf):
        vg = pcl.VoxelGrid(ctx)
        vg.setInputCloud(points)
        vg.setLeafSize(leaf)
        return vg.filter()

    c4, c2 = make_workloads(downsample, world == 1 and not args.no_single, args.hyp, args.scale)
    from pose_estimation_b200 import multi

    H = len(c4.guess)
    per = multi.shard_size(H, world)
    lo, hi = multi.shard_range(H, world, rank)
    h_local = hi - lo
    params = pcl.IcpParams()
    lib.peb_icp_params_default(C.byref(params))
    params.max_iterations = ITERATIONS
    params.abs_mse_threshold = -1.0  # fixed iteration count (icp.getConvergeCriteria()->setAbsoluteMSE(-1))
    params.max_corr_dist = MAX_CORR_DIST

    guesses_cm = col_major(c4.guess)
    h_scene = torch.from_numpy(np.ascontiguousarray(c4.target)).pin_memory()
    h_model = torch.from_numpy(np.ascontiguousarray(c4.source)).pin_memory()
    h_guess = torch.from_numpy(guesses_cm[lo:hi].copy()).pin_memory()
    rec = C.sizeof(pcl.IcpResult)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def chk(rc):
        ctx.check(rc)

    with torch.cuda.stream(stream):
        d_guess = h_guess.to(dev, non_blocking=True)
        d_res = torch.zeros(max(h_local, 1) * rec, dtype=torch.uint8, device=dev)
        d_all = torch.zeros(world * per * rec, dtype=torch.uint8, device=dev)
        d_pad = torch.zeros(per * rec, dtype=torch.uint8, device=dev)
    chk(lib.peb_target_set(ctx.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
    chk(lib.peb_source_set(ctx.handle, h_model.data_ptr(), h_model.shape[0], 16))
    ctx.sync()

    def gather():
        multi.gather_results(d_res, H, world, rank, out=d_all, pad=d_pad)

    def step_device():
        chk(lib.peb_icp_align_batch_dev(ctx.handle, d_guess.data_ptr(), h_local, C.byref(params), d_res.data_ptr()))
        gather()

    h_out = torch.empty(world * per * rec, dtype=torch.uint8).pin_memory()
    host_results = (pcl.IcpResult * max(h_local, 1))()

    def step_e2e():
        chk(lib.peb_target_set(ctx.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
        chk(lib.peb_source_set(ctx.handle, h_model.data_ptr(), h_model.shape[0], 16))
        if world == 1:
            chk(lib.peb_icp_align_batch(ctx.handle, h_guess.data_ptr(), h_local, C.byref(params), host_results))
        else:
            d_guess.copy_(h_guess, non_blocking=True)
            step_device()
            h_out.copy_(d_all, non_blocking=True)
            stream.synchronize()

    def timed(fn, steps, profile=0):
        """-> (total ms of `steps` steps, per-launch iteration-kernel ms)"""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kernel_ms: list[float] = []
        buf = np.zeros(ITERATIONS + 8, np.float32)
        cnt = C.c_size_t(0)
        for a, b in ev:
            flush.zero_()
            a.record(stream)
            fn()
            b.record(stream)
            if profile == 1:    # one value: the span of this step's ITERATIONS iteration launches
                chk(lib.peb_profile_read(ctx.handle, buf.ctypes.data, len(buf), C.byref(cnt)))
                kernel_ms.extend(float(x) for x in buf[: cnt.value])
            elif profile == 2:  # per launch (last entry = fitness launch)
                chk(lib.peb_profile_read(ctx.handle, buf.ctypes.data, len(buf), C.byref(cnt)))
                kernel_ms.extend(float(x) for x in buf[: max(cnt.value - 1, 0)])
        stream.synchronize()
        return sum(a.elapsed_time(b) for a, b in ev), kernel_ms

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    with torch.cuda.stream(stream):
        # ---- device-resident leg: `value` ---------------------------------------------------
        ctx.set_int("profile", 1)
        timed(step_device, args.warmup)
        barrier()
        launches0 = ctx.launch_count
        if rank == 0:
            sampler.start()
        total_ms, span_ms = timed(step_device, args.steps, profile=1)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        launches = ctx.launch_count - launches0
        last_step_records = (d_all if world > 1 else d_res).cpu().numpy().tobytes() if args.dump_outputs else None
        # per-iteration detail from one extra, untimed step (events between the launches serialise them)
        ctx.set_int("profile", 2)
        _, kernel_ms = timed(step_device, 1, profile=2)
        ctx.set_int("profile", 0)
        ms_per_step_local = total_ms / args.steps
        per_rank_ms = [ms_per_step_local]
        if world > 1:  # diagnostics: how uneven the ranks are (the all_gather of every step waits for the slowest)
            t = torch.tensor([ms_per_step_local], dtype=torch.float64, device=dev)
            allt = torch.zeros(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(allt, t)
            per_rank_ms = [round(float(x), 3) for x in allt.cpu()]
        total_ms = max_over_ranks(total_ms)
        # ---- end-to-end leg through the host-buffer C ABI ---------------------------------
        timed(step_e2e, max(1, min(args.warmup, 3)))
        barrier()
        e2e_ms, _ = timed(step_e2e, args.steps)
        barrier()
        e2e_ms = max_over_ranks(e2e_ms)

    # ---- the product's multi-GPU path: ONE process, peb_multi_* over all N devices ---------------------------
    # (the reference node is a single process, launch/pose_estimation.launch.py:17-35).  Rank 0 drives every GPU
    # of the box through one peb_multi handle while the other ranks are parked on a HOST barrier (gloo), their
    # contexts idle; its records must equal the NCCL-gathered records of the one-rank-per-GPU legs byte for byte.
    inproc = None
    if not args.no_inproc:
        ranks_records = (d_all if world > 1 else d_res).cpu().numpy().tobytes()
        torch.cuda.synchronize()
        if rank == 0:
            inproc = inproc_leg(args, torch, pcl, lib, c4, guesses_cm, params, world, H, rec, ranks_records)
        if park is not None:
            dist.barrier(group=park)

    ms_per_step = total_ms / args.steps
    value = H / (ms_per_step * 1e-3)
    e2e_value = H / (e2e_ms / args.steps * 1e-3)
    results_bytes = (d_all if world > 1 else d_res).cpu().numpy().tobytes()

    # ---- roofline of the dominant kernel (icp_iteration_kernel) -------------------------------
    peak, peak_src = HBM_PEAK_GBS, "measured HBM bandwidth of one B200, BASELINE.md (of measured)"
    kernel_name = "icp_iteration_kernel (batched, one launch = one ICP iteration of this rank's hypotheses)"
    alg_bytes = h_local * len(c4.source) * ALG_BYTES_PER_QUERY
    avg_kernel_ms = sum(span_ms) / max(len(span_ms) * ITERATIONS, 1)
    launches_timed = len(span_ms) * ITERATIONS
    achieved = alg_bytes / (avg_kernel_ms * 1e-3) / 1e9 if avg_kernel_ms > 0 else 0.0
    # traffic: dram__bytes_read + dram__bytes_write of one launch from an `ncu --set full` capture of THIS configuration
    # (profiles/roofline_traffic.json names the launch size it was captured at); any other launch size -> null
    traffic = None
    tf = ROOT / "profiles" / "roofline_traffic.json"
    if tf.exists():
        try:
            t = json.loads(tf.read_text())
            if int(t.get("hypotheses_per_launch", -1)) == h_local and int(t.get("n_source", -1)) == len(c4.source):
                traffic = t.get("icp_iteration_kernel_batch_bytes_per_launch")
        except (ValueError, OSError):
            traffic = None
    roofline = {"bound": "hbm", "kernel": kernel_name,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_kernel_ms,
                "launches_timed": launches_timed,
                "peak_source": peak_src,
                "launch_ms_by_iteration": [round(float(x), 3) for x in kernel_ms] if len(kernel_ms) == ITERATIONS else None,
                "share_of_step": (sum(span_ms) / args.steps) / ms_per_step_local if ms_per_step_local > 0 else None}

    line = {
        "metric": "icp_hypotheses_per_s", "value": value, "unit": "hypotheses/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(c4, H),
        "e2e": {"value": e2e_value, "unit": "hypotheses/s", "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": int(world * (h_scene.numel() + h_model.numel()) * 4 + H * 64),
                "d2h_bytes_per_step": int(H * rec if world == 1 else world * world * per * rec),
                "what": "peb_target_set + peb_source_set + peb_icp_align_batch from pinned host buffers, results back on the host"},
        "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks,
        "per_rank_ms_per_step": per_rank_ms,
        "nn_queries_per_s": H * len(c4.source) * ITERATIONS / (ms_per_step * 1e-3),
    }
    if inproc is not None:
        line["inproc"] = inproc

    if rank == 0 and world == 1:
        if c2 is not None:
            with torch.cuda.stream(stream):
                line["align_ms"] = single_align(ctx, c2, torch, stream, flush, pcl, lib)
                line["align_ms"]["c1"] = c1_leg(ctx, torch, stream, flush, pcl, lib)
                line["align_ms"]["cvicp_reference_call"] = cvicp_leg(ctx, c2, pcl, not args.no_cpu_baseline)
                line["align_ms"]["ppf_reference_call"] = ppf_leg(ctx, c2, pcl, not args.no_cpu_baseline)
            stage_fractions(line["align_ms"], peak)
            if not args.no_cpu_baseline:
                # SURVEY.md 8d / BASELINE.md section 4: the CPU port beside EVERY GPU number, same run, same host
                line["align_ms"]["cpu_baseline"] = cpu_stage_baselines(c2)
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(c4)
    if rank == 0:
        # sanity: every hypothesis ran all its iterations
        recs = multi.unpack_results(results_bytes, H, world)
        line["check"] = {"iterations_all": bool((recs["iterations"] == ITERATIONS).all()),
                         "fitness_median": float(np.median(recs["fitness"])),
                         "best_hypothesis": multi.best_hypothesis(recs)}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, multi.unpack_results(last_step_records, H, world))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, records: np.ndarray) -> None:
    """One <out_dir>/<field>.npy per field of the peb_icp_result records: T as (H, 16) float32, column-major as in the
    struct, fitness and last_mse float64, the integer fields widened to float64 (exact), and hypothesis.npy, the index of
    every row.  Above DUMP_BYTES_MAX in all, the rows are a fixed, seeded sample of the hypotheses, in hypothesis order."""
    cols = {f: records[f] if records[f].dtype.kind == "f" else records[f].astype(np.float64) for f in records.dtype.names}
    cols["hypothesis"] = np.arange(len(records), dtype=np.float64)
    total = sum(a.nbytes for a in cols.values())
    budget = DUMP_BYTES_MAX - 4096 * len(cols)  # room for the .npy headers
    if total > budget:
        keep = np.sort(np.random.default_rng(0).choice(len(records), len(records) * budget // total, replace=False))
        cols = {f: a[keep] for f, a in cols.items()}
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for f, a in cols.items():
        np.save(out / f"{f}.npy", a)


def inproc_leg(args, torch, pcl, lib, c4, guesses_cm, params, n_dev, H, rec, ranks_records):
    """peb_multi_create(N) + peb_multi_target_set / _source_set / _icp_align_batch from HOST buffers, results on the
    host: what the reference's single process would call.  Timed with the host clock around the blocking calls (the
    caller's view; there is no asynchronous multi-device entry point), L2 of every device flushed before every step."""
    from pose_estimation_b200 import multi

    m = pcl.MultiContext(list(range(n_dev)))
    for kv in filter(None, os.environ.get("PEB_OPTS", "").split(",")):
        k, v = kv.split("=")
        m.check(lib.peb_multi_set_int(m.handle, k.encode(), int(v)))
    h_scene = torch.from_numpy(np.ascontiguousarray(c4.target)).pin_memory()
    h_model = torch.from_numpy(np.ascontiguousarray(c4.source)).pin_memory()
    h_guess = torch.from_numpy(np.ascontiguousarray(guesses_cm)).pin_memory()
    results = (pcl.IcpResult * H)()
    flushes = [torch.empty(256 << 20, dtype=torch.uint8, device=torch.device("cuda", d)) for d in range(n_dev)]

    def flush_all():
        for f in flushes:
            f.zero_()
        for d in range(n_dev):
            torch.cuda.synchronize(d)

    def setup():
        m.check(lib.peb_multi_target_set(m.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
        m.check(lib.peb_multi_source_set(m.handle, h_model.data_ptr(), h_model.shape[0], 16))

    def align():
        m.check(lib.peb_multi_icp_align_batch(m.handle, h_guess.data_ptr(), H, C.byref(params), results))

    def timed(fn, steps):
        total = 0.0
        for _ in range(steps):
            flush_all()
            t0 = time.perf_counter()
            fn()
            total += time.perf_counter() - t0
        return 1e3 * total / max(steps, 1)

    setup()
    timed(align, max(args.warmup, 1))
    launches0 = m.launch_count
    ms = timed(align, args.steps)
    launches = m.launch_count - launches0
    same = bytes(results) == multi.unpack_results(ranks_records, H, n_dev).tobytes()

    def both():
        setup()
        align()

    timed(both, max(1, min(args.warmup, 3)))
    ms_e2e = timed(both, args.steps)
    # the device's own view of one step: the span of the iteration launches of every device (CUDA events of the library)
    m.check(lib.peb_multi_set_int(m.handle, b"profile", 1))
    align()
    spans = []
    buf = np.zeros(4, np.float32)
    cnt = C.c_size_t(0)
    for d in range(n_dev):
        lib.peb_profile_read(lib.peb_multi_ctx(m.handle, d), buf.ctypes.data, len(buf), C.byref(cnt))
        spans.append(round(float(buf[0]), 3) if cnt.value else None)
    m.close()
    return {
        "what": "ONE process, peb_multi_* over all devices (the single-process node's multi-GPU path): "
                "peb_multi_icp_align_batch from host buffers to host records, scene + model resident",
        "n_devices": n_dev, "value": H / (ms * 1e-3), "unit": "hypotheses/s", "ms_per_step": ms,
        "e2e": {"value": H / (ms_e2e * 1e-3), "unit": "hypotheses/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int((h_scene.numel() + h_model.numel()) * 4 + H * 64), "d2h_bytes_per_step": int(H * rec),
                "what": "peb_multi_target_set + peb_multi_source_set (one upload, device-to-device replicas) + "
                        "peb_multi_icp_align_batch"},
        "records_identical_to_ranks": bool(same), "gpu_launches": int(launches),
        "iteration_span_ms_per_device": spans,
        "timing": "host clock around the blocking calls, 256 MiB L2 flush of every device before every step",
    }


def single_align(ctx, c2, torch, stream, flush, pcl, lib):
    """configs[1]: 200k-pt scene / 50k-pt model, 30 iterations, one align on one GPU."""
    params = pcl.IcpParams()
    lib.peb_icp_params_default(C.byref(params))
    params.max_iterations = ITERATIONS
    params.abs_mse_threshold = -1.0
    h_scene = torch.from_numpy(np.ascontiguousarray(c2.target)).pin_memory()
    h_model = torch.from_numpy(np.ascontiguousarray(c2.source)).pin_memory()
    guess = col_major(c2.guess)
    ctx.check(lib.peb_target_set(ctx.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
    ctx.check(lib.peb_source_set(ctx.handle, h_model.data_ptr(), h_model.shape[0], 16))
    d_res = torch.zeros(C.sizeof(pcl.IcpResult), dtype=torch.uint8, device=flush.device)
    res = pcl.IcpResult()

    def run(cold: bool, host: bool, reps: int = 30):
        out = []
        for _ in range(reps):
            if cold:
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            if host:
                ctx.check(lib.peb_target_set(ctx.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
                ctx.check(lib.peb_source_set(ctx.handle, h_model.data_ptr(), h_model.shape[0], 16))
                ctx.check(lib.peb_icp_align(ctx.handle, guess.ctypes.data, C.byref(params), C.byref(res), None, None, None))
            else:
                ctx.check(lib.peb_icp_align_dev(ctx.handle, guess.ctypes.data, C.byref(params), d_res.data_ptr()))
            b.record(stream)
            stream.synchronize()
            out.append(a.elapsed_time(b))
        return out

    stages = preprocessing_stages(ctx, c2, torch, stream, flush, pcl, lib)
    ctx.check(lib.peb_target_set(ctx.handle, h_scene.data_ptr(), h_scene.shape[0], 16, None, 0))
    run(False, False, 5)
    warm = run(False, False)
    cold = run(True, False)
    e2e = run(True, True, 10)
    return {"workload": "C2 (BASELINE.json configs[1]): one align, 30 point-to-point iterations",
            "n_source": int(len(c2.source)), "n_target": int(len(c2.target)),
            "device_resident_warm_l2": {"median": statistics.median(warm), "min": min(warm)},
            "device_resident_cold_l2": {"median": statistics.median(cold), "min": min(cold)},
            "e2e_host_buffers": {"median": statistics.median(e2e), "min": min(e2e),
                                 "what": "peb_target_set + peb_source_set + peb_icp_align, L2 flushed"},
            "unit": "ms", "target_ms": 2.0, "stages": stages}


def c1_leg(ctx, torch, stream, flush, pcl, lib):
    """configs[0] (C1): 20k-pt model vs its rigidly moved, 1 mm-noise copy, 30 point-to-point iterations — the
    reference's CPU-runnable case, here on the GPU (device-resident and from host buffers)."""
    from pose_estimation_b200.testing import synth

    c1 = synth.make_c1(20000, seed=1)
    params = pcl.IcpParams()
    lib.peb_icp_params_default(C.byref(params))
    params.max_iterations = ITERATIONS
    params.abs_mse_threshold = -1.0
    h_t = torch.from_numpy(np.ascontiguousarray(c1.target)).pin_memory()
    h_s = torch.from_numpy(np.ascontiguousarray(c1.source)).pin_memory()
    d_res = torch.zeros(C.sizeof(pcl.IcpResult), dtype=torch.uint8, device=flush.device)
    res = pcl.IcpResult()

    def setup():
        ctx.check(lib.peb_target_set(ctx.handle, h_t.data_ptr(), h_t.shape[0], 16, None, 0))
        ctx.check(lib.peb_source_set(ctx.handle, h_s.data_ptr(), h_s.shape[0], 16))

    def run(host: bool, reps: int):
        out = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            if host:
                setup()
                ctx.check(lib.peb_icp_align(ctx.handle, None, C.byref(params), C.byref(res), None, None, None))
            else:
                ctx.check(lib.peb_icp_align_dev(ctx.handle, None, C.byref(params), d_res.data_ptr()))
            b.record(stream)
            stream.synchronize()
            out.append(a.elapsed_time(b))
        return out

    setup()
    run(False, 5)
    dev = run(False, 20)
    e2e = run(True, 10)
    alg = ALG_BYTES_PER_QUERY * len(c1.source) * ITERATIONS
    return {"workload": "C1 (BASELINE.json configs[0]): 20k-pt model vs its moved 1 mm-noise copy, 30 point-to-point iterations",
            "device_resident_cold_l2": {"median": statistics.median(dev), "min": min(dev)},
            "e2e_host_buffers": {"median": statistics.median(e2e), "min": min(e2e)},
            "iterations": int(res.iterations), "fitness": float(res.fitness), "algorithmic_bytes": alg,
            "achieved_gbs": alg / (statistics.median(dev) * 1e-3) / 1e9, "unit": "ms"}


def stage_fractions(align, peak):
    """achieved GB/s and fraction of the measured HBM peak for every stage that has algorithmic bytes (SURVEY.md 8d)."""
    n_src = align["n_source"]
    align["algorithmic_bytes"] = ALG_BYTES_PER_QUERY * n_src * ITERATIONS
    align["achieved_gbs"] = align["algorithmic_bytes"] / (align["device_resident_cold_l2"]["median"] * 1e-3) / 1e9
    align["frac"] = align["achieved_gbs"] / peak
    st = align["stages"]
    n_t = align["n_target"]
    st["c3_point_to_plane_align"]["algorithmic_bytes"] = 56 * n_src * ITERATIONS
    st["c5_end_to_end"]["algorithmic_bytes"] = (st["voxel_grid"]["algorithmic_bytes"] + st["normals_k30"]["algorithmic_bytes"]
                                                + 36 * n_t + 56 * n_src * 50)
    for k in ("c3_point_to_plane_align", "c5_end_to_end"):
        st[k]["achieved_gbs"] = st[k]["algorithmic_bytes"] / (st[k]["ms_median"] * 1e-3) / 1e9
    for v in list(st.values()) + [align["c1"]]:
        if isinstance(v, dict) and "achieved_gbs" in v:
            v["frac"] = v["achieved_gbs"] / peak


def cpu_stage_baselines(c2):
    """The CPU port (oracle timing build, the PCL 1.10 restatement: single kd-tree, leaf 15, exact search) on this box's
    host cores for every stage bench.py times on the GPU.  PCL 1.10's ICP loop, VoxelGrid and NormalEstimation are serial
    (1 thread); NormalEstimationOMP is the all-cores figure."""
    from oracle import Oracle, default_params
    from pose_estimation_b200.testing import synth

    orc = Oracle(fast=True)
    cores = host_threads()

    def timed(fn):
        t0 = time.perf_counter()
        out = fn()
        return 1e3 * (time.perf_counter() - t0), out

    out = {"kind": "port", "cores": cores, "unit": "ms",
           "what": "oracle timing build (-O3 AVX2/FMA) of the PCL 1.10 restatement, wall clock, kd-tree build included"}
    c1 = synth.make_c1(20000, seed=1)
    prm = default_params(max_iterations=ITERATIONS, abs_mse_threshold=-1.0)
    out["c1_align_1_thread"], _ = timed(lambda: orc.icp(c1.target).align(c1.source, None, prm))
    out["c2_align_1_thread"], _ = timed(lambda: orc.icp(c2.target).align(c2.source, c2.guess, prm))
    out["voxel_grid_1_thread"], (ds, _u) = timed(lambda: orc.voxel_grid(c2.organized, c2.leaf))
    out["normals_k30_1_thread"], nrm = timed(lambda: orc.normals(ds, 30, threads=1))
    out["normals_k30_all_cores"], _ = timed(lambda: orc.normals(ds, 30, threads=cores))
    p3 = default_params(max_iterations=ITERATIONS, abs_mse_threshold=-1.0, estimator=1)
    out["c3_point_to_plane_align_1_thread"], _ = timed(lambda: orc.icp(ds, nrm[:, :3].copy()).align(c2.source, c2.guess, p3))
    p5 = default_params(max_iterations=50, abs_mse_threshold=-1.0, estimator=1)

    def c5():
        d, _ = orc.voxel_grid(c2.organized, c2.leaf)
        n = orc.normals(d, 30, threads=1)
        return orc.icp(d, n[:, :3].copy()).align(c2.source, c2.guess, p5)

    out["c5_end_to_end_1_thread"], _ = timed(c5)
    return out


def cvicp_leg(ctx, c2, pcl, with_cpu: bool):
    """The reference's own call in the refinement slot (opencv_surface_match.cpp:85-94): cv::ppf_match_3d::ICP(250, 0.005f,
    2.5f, 8).registerModelToScene(model, scene with normals, 6 poses), on the C2 clouds, through the host-buffer C ABI
    (uploads, 8 level grids, read-backs included), wall clock."""
    import time

    from pose_estimation_b200.testing import synth

    def with_normals(cloud):
        ne = pcl.NormalEstimation(ctx)
        ne.setInputCloud(cloud)
        ne.setKSearch(20)  # computeNormalsPC3d(scene, out, 20, true, viewpoint) in the reference
        nrm = ne.compute()
        ok = np.isfinite(nrm[:, :3]).all(1) & np.isfinite(cloud[:, :3]).all(1)
        return np.ascontiguousarray(np.concatenate([cloud[ok, :3], nrm[ok, :3]], 1), np.float32)

    scene6 = with_normals(c2.target)
    model6 = with_normals(c2.source)
    rng = np.random.default_rng(7)
    poses = np.stack([synth.perturb_pose(c2.gt_pose, rng, 4.0, 0.006) for _ in range(6)])
    icp = pcl.CvIcp(250, 0.005, 2.5, 8, ctx=ctx)
    icp.registerModelToScene(model6, scene6, poses)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        got, res = icp.registerModelToScene(model6, scene6, poses)
        ts.append(1e3 * (time.perf_counter() - t0))
    out = {"workload": "cv::ppf_match_3d::ICP(250, 0.005, 2.5, 8).registerModelToScene, 6 poses, C2 clouds with k = 20 normals",
           "n_model": int(len(model6)), "n_scene": int(len(scene6)), "ms_median": statistics.median(ts), "ms_min": min(ts),
           "residual_median": float(np.median(res)),
           "pose_error_vs_truth_rad_max": float(max(synth.pose_error(P, c2.gt_pose)[0] for P in got))}
    if with_cpu:
        from oracle import Oracle, cvicp_params
        orc = Oracle(fast=True)
        t0 = time.perf_counter()
        ref, _ = orc.cvicp_register(model6, scene6, poses, cvicp_params())
        out["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
        out["cpu_port_threads"] = min(6, host_threads())
        out["vs_cpu_port_rad_max"] = float(max(synth.pose_error(a, b)[0] for a, b in zip(got, ref)))
    return out


def ppf_leg(ctx, c2, pcl, with_cpu: bool):
    """The reference's coarse matcher in front of the refinement slot (opencv_surface_match.cpp:45-46, :65):
    PPF3DDetector(0.03, 0.03, 40).trainModel(model) once, then match(scene with normals, results, 1.0, 0.03) per frame, on
    the C2 clouds (background plane cut off like remove_planes does), through the host-buffer C ABI, wall clock."""
    import time

    from pose_estimation_b200.testing import synth

    def with_normals(cloud, viewpoint):
        ne = pcl.NormalEstimation(ctx)
        ne.setInputCloud(cloud)
        ne.setKSearch(20)
        ne.setViewPoint(*viewpoint)
        nrm = ne.compute()
        ok = np.isfinite(nrm[:, :3]).all(1) & np.isfinite(cloud[:, :3]).all(1)
        return np.ascontiguousarray(np.concatenate([cloud[ok, :3], nrm[ok, :3]], 1), np.float32)

    scene = c2.target[c2.target[:, 2] < 0.735]
    scene6 = with_normals(scene, (0.0, 0.0, 0.0))
    model6 = with_normals(c2.source, (0.0, 0.0, 1.0))  # the model's outward side (object frame), consistently
    det = pcl.PPF3DDetector(0.03, 0.03, 40, ctx=ctx)

    def timed(fn, reps):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            ts.append(1e3 * (time.perf_counter() - t0))
        return statistics.median(ts), min(ts), r

    t_train, t_train_min, _ = timed(lambda: det.trainModel(model6), 3)
    t_match, t_match_min, clustered = timed(lambda: det.match(scene6, 1.0, 0.03), 5)
    _, raw = det.match(scene6, 1.0, 0.03, return_raw=True)
    rot, trans = synth.pose_error(clustered[0].matrix, c2.gt_pose)
    out = {"workload": "cv::ppf_match_3d::PPF3DDetector(0.03, 0.03, 40): trainModel(model) and match(scene, 1.0, 0.03), C2 clouds "
                       "with k = 20 normals, plane cut off",
           "n_model": int(len(model6)), "n_scene": int(len(scene6)), "n_model_sampled": int(len(det.sampled_model())),
           "n_scene_reference_points": int(len(raw)), "n_clusters": int(len(clustered)),
           "train_ms_median": t_train, "train_ms_min": t_train_min, "match_ms_median": t_match, "match_ms_min": t_match_min,
           "top_votes": int(clustered[0].num_votes), "top_pose_error_rad": rot, "top_pose_error_m": trans}
    if with_cpu:
        from oracle import Oracle
        orc = Oracle(fast=True)
        t0 = time.perf_counter()
        ref = orc.ppf_train(model6)
        out["cpu_port_train_ms"] = 1e3 * (time.perf_counter() - t0)
        t0 = time.perf_counter()
        ores, oraw, _ = ref.match(scene6, 1.0, 0.03)
        out["cpu_port_match_ms"] = 1e3 * (time.perf_counter() - t0)
        out["cpu_port_threads"] = host_threads()
        out["raw_poses_identical_to_cpu_port"] = float(np.mean([(a.num_votes, a.model_index) == (b.num_votes, b.model_index)
                                                                for a, b in zip(raw, oraw)]))
    det.close()
    return out


def preprocessing_stages(ctx, c2, torch, stream, flush, pcl, lib):
    """configs[4] stages that feed the align: VoxelGrid of the 2.33M-pt organized scene and k = 30 normals of
    the ~200k-pt result, device-resident, CUDA events, L2 flushed; algorithmic bytes per SURVEY.md 8d."""
    dev = flush.device
    d_scene = torch.from_numpy(np.ascontiguousarray(c2.organized)).to(dev)
    n_in = d_scene.shape[0]
    d_out = torch.empty((n_in, 4), dtype=torch.float32, device=dev)
    m = C.c_size_t(0)
    leaf = float(c2.leaf)

    def timed(fn, reps=10):
        out = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            stream.synchronize()
            out.append(a.elapsed_time(b))
        return out

    def vox():
        ctx.check(lib.peb_voxel_grid_dev(ctx.handle, d_scene.data_ptr(), n_in, leaf, leaf, leaf, 0, d_out.data_ptr(), C.byref(m)))

    vox()
    t_vox = timed(vox)
    n_ds = m.value
    d_nrm = torch.empty((n_ds, 8), dtype=torch.float32, device=dev)
    vp = np.zeros(3, np.float32)

    def nrm():
        ctx.check(lib.peb_normals_knn_dev(ctx.handle, d_out.data_ptr(), n_ds, 30, vp.ctypes.data, d_nrm.data_ptr()))

    nrm()
    t_nrm = timed(nrm)
    h_ds = torch.empty((n_ds, 4), dtype=torch.float32).pin_memory()
    h_ds.copy_(d_out[:n_ds])

    def tset():
        ctx.check(lib.peb_target_set_dev(ctx.handle, d_out.data_ptr(), n_ds, None))

    tset()
    t_set = timed(tset)

    # ---- the brute-force FP32 validator (north star (2)) and the grid search on the same queries (C2: the model under
    # the initial guess against the down-sampled scene), through the host-buffer C ABI (uploads / downloads inside)
    g4 = np.asarray(c2.guess, np.float64)
    q_host = np.ascontiguousarray(c2.source, np.float32).copy()
    q_host[:, :3] = (c2.source[:, :3].astype(np.float64) @ g4[:3, :3].T + g4[:3, 3]).astype(np.float32)
    h_q = torch.from_numpy(q_host).pin_memory()
    nq = h_q.shape[0]
    h_idx = [torch.empty(nq, dtype=torch.int32).pin_memory() for _ in range(2)]
    h_d2 = [torch.empty(nq, dtype=torch.float32).pin_memory() for _ in range(2)]

    def nn_brute():
        ctx.check(lib.peb_nn_search_bruteforce(ctx.handle, h_q.data_ptr(), nq, 16, h_idx[0].data_ptr(), h_d2[0].data_ptr()))

    def nn_grid():
        ctx.check(lib.peb_nn_search(ctx.handle, h_q.data_ptr(), nq, 16, h_idx[1].data_ptr(), h_d2[1].data_ptr()))

    nn_brute()
    nn_grid()
    t_brute = timed(nn_brute, 5)
    t_grid = timed(nn_grid, 5)
    nn_same = bool(torch.equal(h_d2[0], h_d2[1]) and torch.equal(h_idx[0], h_idx[1]))
    pairs = float(nq) * float(n_ds)
    fp32_instr_peak = 148 * 128 * 1.965e9  # one FADD / FMUL per lane and clock (no FMA: the distance is PCL's unfused expression)
    brute_stage = {
        "what": "nn_bruteforce_kernel, every query against every target point (8 FP32 instructions per pair: 3 FADD + 3 FMUL + "
                "2 FADD, unfused, + 1 FMNMX), host buffers in and out",
        "n_queries": int(nq), "n_target": int(n_ds), "ms_median": statistics.median(t_brute), "ms_min": min(t_brute),
        "fp32_instr_per_s": 8.0 * pairs / (statistics.median(t_brute) * 1e-3),
        "fp32_pipe_frac": 8.0 * pairs / (statistics.median(t_brute) * 1e-3) / fp32_instr_peak,
        "fp32_pipe_peak": "148 SMs x 128 lanes x 1.965 GHz = 3.72e13 FADD|FMUL per s",
        "grid_search_same_queries_ms": statistics.median(t_grid), "identical_to_grid_search": nn_same}

    # ---- configs[2] (C3) and configs[4] (C5): point-to-plane aligns with the normals estimated on the device ----
    d_nrm4 = torch.zeros((n_ds, 4), dtype=torch.float32, device=dev)
    d_model = torch.from_numpy(np.ascontiguousarray(c2.source)).to(dev)
    d_res = torch.zeros(C.sizeof(pcl.IcpResult), dtype=torch.uint8, device=dev)
    guess = col_major(c2.guess)
    prm = pcl.IcpParams()
    lib.peb_icp_params_default(C.byref(prm))
    prm.estimator = 1  # PEB_ESTIMATOR_POINT_TO_PLANE_LLS
    prm.abs_mse_threshold = -1.0
    ctx.check(lib.peb_source_set_dev(ctx.handle, d_model.data_ptr(), d_model.shape[0]))

    def target_with_normals():
        d_nrm4.copy_(d_nrm[:, :4])  # pcl::Normal (8 floats) -> normal_x normal_y normal_z 0
        ctx.check(lib.peb_target_set_dev(ctx.handle, d_out.data_ptr(), n_ds, d_nrm4.data_ptr()))

    def p2plane(iters):
        prm.max_iterations = iters
        ctx.check(lib.peb_icp_align_dev(ctx.handle, guess.ctypes.data, C.byref(prm), d_res.data_ptr()))

    with torch.cuda.stream(stream):
        target_with_normals()
        p2plane(30)
        t_c3 = timed(lambda: p2plane(30), 20)

        def c5():
            vox()
            nrm()
            target_with_normals()
            p2plane(50)

        c5()
        t_c5 = timed(c5)
        res_c5 = pcl.IcpResult.from_buffer_copy(d_res.cpu().numpy().tobytes())
    # scene preparation in front of VoxelGrid (SURVEY.md 8f rank 1): NaN removal, then the reference's plane fit
    # (threshold 0.0001, 100 iterations, optimised coefficients) and its 5 mm band removal
    from pose_estimation_b200._lib import PrefilterParams, SacParams
    pf = PrefilterParams()
    pf.plane_band = 0.005
    d_clean = torch.empty((n_in, 4), dtype=torch.float32, device=dev)
    d_kept = torch.empty((n_in, 4), dtype=torch.float32, device=dev)
    mc = C.c_size_t(0)

    def clean():
        ctx.check(lib.peb_scene_prefilter_dev(ctx.handle, d_scene.data_ptr(), n_in, C.byref(pf), d_clean.data_ptr(), C.byref(mc)))

    clean()
    t_clean = timed(clean)
    n_clean = mc.value
    sp = SacParams()
    lib.peb_sac_params_default(C.byref(sp))
    sp.distance_threshold, sp.max_iterations = 1e-4, 100
    coeff = np.zeros(4, np.float32)
    n_inl = C.c_size_t(0)
    its = C.c_int32(0)

    def sac():
        ctx.check(lib.peb_sac_plane_dev(ctx.handle, d_clean.data_ptr(), n_clean, C.byref(sp), coeff.ctypes.data, None,
                                        C.byref(n_inl), C.byref(its)))

    sac()
    t_sac = timed(sac)
    pf2 = PrefilterParams()
    pf2.plane_band = 0.005
    pf2.n_planes = 1
    for j in range(4):
        pf2.planes[j] = float(coeff[j])
    mk = C.c_size_t(0)

    def band():
        ctx.check(lib.peb_scene_prefilter_dev(ctx.handle, d_clean.data_ptr(), n_clean, C.byref(pf2), d_kept.data_ptr(), C.byref(mk)))

    band()
    t_band = timed(band)
    vb = 16 * n_in + 16 * n_ds
    nb = n_ds * (16 + 16 * 30 + 32)
    gb = n_ds * 36
    return {
        "voxel_grid": {"n_in": int(n_in), "n_out": int(n_ds), "ms_median": statistics.median(t_vox), "ms_min": min(t_vox),
                       "algorithmic_bytes": vb, "achieved_gbs": vb / (statistics.median(t_vox) * 1e-3) / 1e9},
        "normals_k30": {"n": int(n_ds), "ms_median": statistics.median(t_nrm), "ms_min": min(t_nrm),
                        "algorithmic_bytes": nb, "achieved_gbs": nb / (statistics.median(t_nrm) * 1e-3) / 1e9},
        "target_grid_build": {"n": int(n_ds), "ms_median": statistics.median(t_set), "ms_min": min(t_set),
                              "algorithmic_bytes": gb, "achieved_gbs": gb / (statistics.median(t_set) * 1e-3) / 1e9},
        "nn_validator_bruteforce": brute_stage,
        "nan_removal": {"n_in": int(n_in), "n_out": int(n_clean), "ms_median": statistics.median(t_clean), "ms_min": min(t_clean),
                        "algorithmic_bytes": 16 * (n_in + n_clean),
                        "achieved_gbs": 16 * (n_in + n_clean) / (statistics.median(t_clean) * 1e-3) / 1e9},
        "plane_ransac": {"n": int(n_clean), "iterations": int(its.value), "inliers": int(n_inl.value),
                         "coefficients": [float(v) for v in coeff], "ms_median": statistics.median(t_sac), "ms_min": min(t_sac),
                         "what": "pcl::SACSegmentation plane fit of remove_planes (threshold 1e-4, 100 iterations, optimised): "
                                 "one counting pass over the cloud for all candidate planes + two inlier selections + moments",
                         "algorithmic_bytes": 16 * n_clean * 4,
                         "achieved_gbs": 16 * n_clean * 4 / (statistics.median(t_sac) * 1e-3) / 1e9},
        "plane_band_removal": {"n_in": int(n_clean), "n_out": int(mk.value), "ms_median": statistics.median(t_band),
                               "ms_min": min(t_band)},
        "c3_point_to_plane_align": {"workload": "C3 (BASELINE.json configs[2]): one align, 30 point-to-plane iterations, normals k = 30 "
                                                "from the device, target grid resident", "ms_median": statistics.median(t_c3), "ms_min": min(t_c3)},
        "c5_end_to_end": {"workload": "C5 (BASELINE.json configs[4]): 2.33 M-point organized scene resident in HBM -> VoxelGrid -> normals "
                                      "k = 30 -> target grid -> 50 point-to-plane iterations", "ms_median": statistics.median(t_c5),
                          "ms_min": min(t_c5), "iterations": int(res_c5.iterations), "fitness": float(res_c5.fitness)},
        "note": "device-resident inputs, CUDA events on the library stream, includes the host syncs each stage needs "
                "(bounding box, run counts)",
    }


def cpu_baseline(c4):
    """The oracle's timing build on this box's host cores, bounded sample of the same workload."""
    from oracle import Oracle

    orc = Oracle(fast=True)
    cores = host_threads()
    icp = orc.icp(c4.target)
    n = max(cores, 8)
    rate, dt = cpu_batch_rate(icp, c4.source, c4.guess, cores, n)
    if dt < 8.0:  # scale the sample up to ~10-20 s of wall time
        n2 = int(min(N_HYP, max(n, (15.0 / dt) * n) // cores * cores))
        if n2 > n:
            rate, dt = cpu_batch_rate(icp, c4.source, c4.guess, cores, n2)
            n = n2
    return {"value": rate, "unit": "hypotheses/s", "cores": cores, "kind": "port",
            "sample": f"{n} of the {len(c4.guess)} hypotheses in {dt:.1f} s, OpenMP over hypotheses ({cores} threads), "
                      "oracle timing build (-O3 AVX2/FMA) of the PCL 1.10 restatement"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--hyp", type=int, default=N_HYP, help="total hypotheses (default: the 1024 of configs[3])")
    ap.add_argument("--scale", type=float, default=1.0, help="linear scene scale (1.0 = the 1944x1200 configuration)")
    ap.add_argument("--no-single", action="store_true", help="skip the configs[1] single-align leg")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-inproc", action="store_true", help="skip the single-process peb_multi_* leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA arm (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        log("[bench] note: the timing rules ask for >= 3 warm-up steps")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
