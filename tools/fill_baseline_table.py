"""Rewrites the result table of BASELINE.md section 5 from a bench.py line (the N = 1 default run).

usage: python tools/fill_baseline_table.py <bench line .json> [--write]

Every figure of the table is read from the JSON line: GPU times are CUDA-event medians of the run, CPU times are the
oracle's timing build measured in the SAME run on the GPU box's host cores (bench.py : cpu_baseline legs).
"""
import json
import pathlib
import re
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
PEAK = 6544.7


def gbs(nbytes, ms):
    return nbytes / (ms * 1e-3) / 1e9


def row(config, stage, ms, nbytes, cpu, parity):
    g = gbs(nbytes, ms)
    return f"| {config} | {stage} | {ms:.3f} | {nbytes / 1e6:.1f} MB | {g:.0f} | {100 * g / PEAK:.2f} % | {cpu} | {parity} |"


def main():
    src = pathlib.Path(sys.argv[1])
    d = json.loads(src.read_text().strip().splitlines()[-1])
    a = d["align_ms"]
    st = a["stages"]
    cb = a["cpu_baseline"]
    cores = cb["cores"]
    rl = d["roofline"]
    c4_bytes = rl["algorithmic_bytes_per_launch"] * d["config"]["iterations"]
    traffic = rl.get("traffic")  # ncu DRAM bytes per launch (profiles/roofline_traffic.json), null when none is recorded
    traffic_note = (f"DRAM traffic per launch measured by ncu: {traffic / 1e9:.2f} GB, `profiles/roofline_traffic.json`"
                    if traffic else "DRAM traffic per launch: not measured for this launch structure")
    rows = [
        "| config | stage | GPU ms (median, cold L2) | algorithmic bytes | achieved GB/s | % of measured HBM (6 544.7 GB/s) | CPU oracle ms (threads) | parity (test) |",
        "|---|---|---|---|---|---|---|---|",
        row("C1 20 k/20 k p2p 30 it", "align", a["c1"]["device_resident_cold_l2"]["median"], a["c1"]["algorithmic_bytes"],
            f"{cb['c1_align_1_thread']:.0f} (1)", "bit-exact indices, 1e-5 rad / m vs the oracle (`test_icp_c1_*`)"),
        row("C2 200 k/50 k p2p 30 it", "align (grid resident)", a["device_resident_cold_l2"]["median"], a["algorithmic_bytes"],
            f"{cb['c2_align_1_thread']:.0f} (1)", "`test_c2_single_align_full_size_vs_oracle`"),
        row("C2", "align from host buffers (upload + grid build + align)", a["e2e_host_buffers"]["median"], a["algorithmic_bytes"],
            f"{cb['c2_align_1_thread']:.0f} (1)", "same records"),
        row("C2", "target grid build", st["target_grid_build"]["ms_median"], st["target_grid_build"]["algorithmic_bytes"],
            "(kd-tree build is inside the align figures)", "every NN test"),
        row("C3 200 k/50 k p2plane 30 it", "normals k = 30", st["normals_k30"]["ms_median"], st["normals_k30"]["algorithmic_bytes"],
            f"{cb['normals_k30_1_thread']:.0f} (1) / {cb['normals_k30_all_cores']:.0f} ({cores})",
            "lists identical up to ties, <= 0.05 deg (`test_normals_match_oracle`)"),
        row("C3", "align", st["c3_point_to_plane_align"]["ms_median"], st["c3_point_to_plane_align"]["algorithmic_bytes"],
            f"{cb['c3_point_to_plane_align_1_thread']:.0f} (1)", "`test_c3_point_to_plane_with_gpu_normals_full_size_vs_oracle`"),
        row(f"C4 {d['config']['hypotheses']} x 50 k vs 507 k, 30 it, 1 GPU", f"batch align: {d['value']:.0f} hypotheses/s",
            d["ms_per_step"], c4_bytes,
            f"{d['cpu_baseline']['value']:.1f} hypotheses/s ({d['cpu_baseline']['cores']}) = "
            f"{1e3 * d['config']['hypotheses'] / d['cpu_baseline']['value']:.0f} ms",
            "`test_c4_batch_sample_full_size_vs_oracle` (96 of 1024 vs the oracle), batch == singles"),
        row("C5 2.33 M end-to-end", "VoxelGrid", st["voxel_grid"]["ms_median"], st["voxel_grid"]["algorithmic_bytes"],
            f"{cb['voxel_grid_1_thread']:.0f} (1)", "bit-exact (`test_c5_voxel_grid_2m3_points_bit_exact`)"),
        row("C5", "VoxelGrid + normals + grid + 50-it p2plane", st["c5_end_to_end"]["ms_median"],
            st["c5_end_to_end"]["algorithmic_bytes"], f"{cb['c5_end_to_end_1_thread']:.0f} (1)",
            "`test_c5_end_to_end_50_iterations`"),
        row("C5 scene preparation", "NaN removal", st["nan_removal"]["ms_median"], st["nan_removal"]["algorithmic_bytes"], "—",
            "bit-exact (`test_scene_prefilter_bit_exact`)"),
        row("C5 scene preparation", f"plane RANSAC ({st['plane_ransac']['iterations']} it)", st["plane_ransac"]["ms_median"],
            st["plane_ransac"]["algorithmic_bytes"], "—", "bit-exact vs the sequential loop (`test_sac.py`)"),
    ]
    v = st["nn_validator_bruteforce"]
    extra = [
        "",
        f"Validator (north star (2)): `nn_bruteforce_kernel`, {v['n_queries']} x {v['n_target']} pairs in {v['ms_median']:.2f} ms = "
        f"{100 * v['fp32_pipe_frac']:.0f} % of the FP32 pipe ({v['fp32_pipe_peak']}); identical to the grid search "
        f"({v['grid_search_same_queries_ms']:.3f} ms for the same queries): {v['identical_to_grid_search']}.",
        "",
        f"C4 roofline of the dominant kernel: {rl['achieved']:.0f} GB/s = {rl['frac']:.3f} of {rl['peak']} GB/s "
        f"(algorithmic {rl['algorithmic_bytes_per_launch'] / 1e9:.3f} GB per launch = 40 B per query; average launch "
        f"{rl['avg_launch_ms']:.2f} ms; {traffic_note}).  End to end from host buffers: {d['e2e']['value']:.0f} hypotheses/s.",
        "",
        f"Source: `{src.name}` (B200, SM clock {d['clocks']['sm_mhz']} MHz, throttle reasons {d['clocks']['reasons']}); CPU = "
        f"{cb['what']}; the GPU box had {cores} host cores.",
    ]
    table = "\n".join(rows + extra)
    print(table)
    if "--write" in sys.argv:
        p = ROOT / "BASELINE.md"
        text = p.read_text()
        head, sep, tail = text.partition("## 5. Result table")
        m = re.search(r"\nAlgorithmic-byte definitions", tail)
        new_tail = " (filled from the bench line named below by `tools/fill_baseline_table.py`)\n\n" + table + "\n" + tail[m.start():]
        p.write_text(head + "## 5. Result table" + new_tail)


if __name__ == "__main__":
    main()
