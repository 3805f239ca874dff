#!/usr/bin/env python3
"""Turn the scratch captures under gpurun_out/ into the tracked summaries under profiles/.

    python tools/make_profiles.py TAG [ncu-rep] [launch-list-csv]

Writes profiles/<TAG>_metrics.csv (selected `ncu --set full` metrics per captured kernel),
profiles/<TAG>_launches.csv (kernel, grid, block, gpu__time_duration per launch), and
profiles/sass/<kernel>.sass (cuobjdump of the shipped libsmplgpu.so, one file per kernel).
"""
import csv
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROF = os.path.join(ROOT, "profiles")

METRICS = [
    "gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread",
    "launch__shared_mem_per_block_dynamic", "launch__occupancy_limit_shared_mem", "launch__occupancy_limit_registers",
    "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
    "smsp__inst_executed.sum", "smsp__thread_inst_executed_per_inst_executed.ratio",
    "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active",
    "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active",
    "dram__bytes_read.sum", "dram__bytes_write.sum", "dram__throughput.avg.pct_of_peak_sustained_elapsed",
    "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "lts__t_bytes.sum", "lts__t_bytes.sum.per_second", "lts__t_sector_hit_rate.pct", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
    "l1tex__t_sector_hit_rate.pct", "l1tex__t_bytes.sum",
    "smsp__sass_average_data_bytes_per_sector_mem_global_op_ld.pct", "smsp__sass_average_data_bytes_per_sector_mem_global_op_st.pct",
    "l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum", "l1tex__t_requests_pipe_lsu_mem_global_op_ld.sum",
    "l1tex__t_sectors_pipe_lsu_mem_global_op_st.sum", "l1tex__t_requests_pipe_lsu_mem_global_op_st.sum",
    "sm__cycles_elapsed.avg", "sm__cycles_active.avg",
]


def metrics(tag, rep):
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    hdr, units = rows[0], rows[1]
    ix = {h: i for i, h in enumerate(hdr)}
    out = os.path.join(PROF, tag + "_metrics.csv")
    with open(out, "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(["kernel", "metric", "value", "unit"])
        for r in rows[2:]:
            name = re.sub(r"\(.*", "", r[ix["Kernel Name"]])
            for m in METRICS:
                if m in ix:
                    w.writerow([name, m, r[ix[m]], units[ix[m]]])
            # warp stall breakdown
            for h in hdr:
                if h.startswith("smsp__average_warps_issue_stalled_") and h.endswith("_per_issue_active.ratio"):
                    w.writerow([name, h, r[ix[h]], units[ix[h]]])
    print("wrote", out)


def launches(tag, path):
    rows = [r for r in csv.reader(open(path)) if r and r[0].isdigit()]
    out = os.path.join(PROF, tag + "_launches.csv")
    with open(out, "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(["id", "kernel", "block", "grid", "gpu_time_ns"])
        for r in rows:
            name = re.sub(r"\(.*", "", r[4])
            w.writerow([r[0], name, r[7], r[8], r[-1]])
    print("wrote", out)


def sass():
    lib = os.path.join(ROOT, "smpl_b200", "lib", "libsmplgpu.so")
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    d = os.path.join(PROF, "sass")
    os.makedirs(d, exist_ok=True)
    cur, name = [], None
    def flush():
        if name and cur:
            # "void bfs_tiles_kernel<4>" -> bfs_tiles_kernel_rpt4, "void states_valid32_kernel<1>" -> states_valid32_kernel_1
            short = re.sub(r"^void\s+", "", name)
            short = re.sub(r"<(\d+)>", r"_rpt\1" if short.startswith("bfs_tiles_kernel") else r"_\1", short)
            short = re.sub(r"[^A-Za-z0-9_]", "", short)
            with open(os.path.join(d, short + ".sass"), "w") as f:
                f.write("\n".join(cur) + "\n")
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            flush()
            cur = []
            sym = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            name = re.sub(r"\(.*", "", sym).replace("smplgpu::", "")
        if name:
            cur.append(line.rstrip())
    flush()
    print("wrote", d)


if __name__ == "__main__":
    os.makedirs(PROF, exist_ok=True)
    tag = sys.argv[1]
    if len(sys.argv) > 2 and sys.argv[2] != "-":
        metrics(tag, sys.argv[2])
    if len(sys.argv) > 3 and sys.argv[3] != "-":
        launches(tag, sys.argv[3])
    sass()
