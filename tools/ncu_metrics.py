"""Extract the per-launch figures bench.py quotes from committed ncu captures (development tool).

    python tools/ncu_metrics.py nuts=gpurun_out/r2_nuts.ncu-rep counts=gpurun_out/r2_counts.ncu-rep > profiles/r02_ncu_metrics.json

For every `name=report` the FIRST kernel of the report whose name contains the given key
(`nuts` -> nuts_group_kernel, `counts` -> counts_stream_kernel) is read with `ncu --page raw --csv`:
DRAM bytes, duration, issue / pipe utilisation, instruction counts, stall ratios."""
import csv
import json
import subprocess
import sys

KEYS = {"nuts": "nuts_group_kernel", "counts": "counts_stream_kernel"}
METRICS = {
    "duration_ms": "gpu__time_duration.sum",
    "dram_bytes_read": "dram__bytes_read.sum",
    "dram_bytes_write": "dram__bytes_write.sum",
    "registers_per_thread": "launch__registers_per_thread",
    "grid_size": "launch__grid_size",
    "warps_active_pct": "sm__warps_active.avg.pct_of_peak_sustained_active",
    "issue_active_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active",
    "pipe_fp64_pct": "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active",
    "pipe_xu_pct": "sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active",
    "pipe_alu_pct": "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active",
    "pipe_fma_pct": "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active",
    "pipe_lsu_pct": "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active",
    "warp_instructions": "smsp__inst_executed.sum",
    "active_threads_per_instruction": "smsp__thread_inst_executed_per_inst_executed.ratio",
    "icache_hit_rate_pct": "sm__icc_request_hit_rate.pct",
    "dram_throughput_pct": "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
}


def to_bytes(value, unit):
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
    return float(value) * scale


def to_ms(value, unit):
    scale = {"ns": 1e-6, "us": 1e-3, "ms": 1, "s": 1e3}.get(unit, 1)
    return float(value) * scale


out = {}
for arg in sys.argv[1:]:
    name, rep = arg.split("=", 1)
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    hdr, units = rows[0], rows[1]
    row = next((r for r in rows[2:] if KEYS.get(name, name) in r[hdr.index("Kernel Name")]), None)
    if row is None:
        continue
    d = {"kernel": row[hdr.index("Kernel Name")], "report": rep}
    for key, metric in METRICS.items():
        if metric not in hdr:
            continue
        i = hdr.index(metric)
        try:
            v = float(row[i].replace(",", ""))
        except ValueError:
            continue
        if key.startswith("dram_bytes"):
            v = to_bytes(v, units[i])
        elif key == "duration_ms":
            v = to_ms(v, units[i])
        d[key] = v
    if "dram_bytes_read" in d:
        d["dram_bytes_per_launch"] = d["dram_bytes_read"] + d.get("dram_bytes_write", 0.0)
    stalls = {}
    for i, h in enumerate(hdr):
        if "average_warps_issue_stalled" in h and h.endswith("per_issue_active.ratio") and "not_issued" not in h:
            try:
                stalls[h.replace("smsp__average_warps_issue_stalled_", "").replace("_per_issue_active.ratio", "")] = float(row[i])
            except ValueError:
                pass
    d["stalls_warps_per_issue"] = dict(sorted(stalls.items(), key=lambda kv: -kv[1])[:8])
    out[name] = d
json.dump(out, sys.stdout, indent=1)
print()
