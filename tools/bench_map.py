"""Throughput of the MAP-only screening path (mdg_map_batch, device-resident inputs) and of its profile intervals
(mdg_map_profile at level 0.68, device-resident inputs and MAP rows) on one GPU.

Sizes: 10 000 fitted TaxIDs of the cfg2 generator and 1 000 000 of the cfg3 generator (eight independently generated
shares, rank r = jumped block r, as bench.py's multi-GPU workload). Every size gets a warm-up call, then calls are
repeated until at least `--min-seconds` of work has been timed: CUDA events around the whole window and the host clock
around it (ending in a synchronise). For the ratio, one timed mdg_fit_batch step (six NUTS runs per TaxID) on the
10 000-TaxID batch after a warm-up step. The profile block times mdg_map_profile the same way at both sizes, on the
rows of one mdg_map_batch call. Prints one JSON line; writes nothing unless --out is given.

    python tools/bench_map.py [--out profiles/r05_map_profile_1gpu.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    """card name, power limit and SM clocks, read-only query"""
    fields = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={fields}", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    return dict(zip(fields.split(","), [v.strip() for v in out.split(",")]))


def cfg2_batch(n):
    from metadamage_b200 import synthetic as syn

    tid, k, N, _ = syn.dense_fit_batch(n, seed=syn.SEEDS["cfg2"])
    return tid, k, N


def to_device(dev, tid, k, N):
    import torch

    return (torch.from_numpy(tid).to(dev), torch.from_numpy(k.view(np.int32)).to(dev), torch.from_numpy(N.view(np.int32)).to(dev))


def time_map(ctx, dev, name, tid, k, N, min_seconds):
    import torch

    from metadamage_b200._abi import MAP_RESULT_DTYPE

    n = len(tid)
    dt, dk, dN = to_device(dev, tid, k, N)
    out = torch.empty(n * MAP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    ctx.map_batch_device(dt, dk, dN, out)  # warm-up at this size
    torch.cuda.synchronize(dev)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, map_ms, asm_ms, evals = 0, 0.0, 0.0, 0
    t0 = time.perf_counter()
    start.record()
    while True:
        ctx.map_batch_device(dt, dk, dN, out)
        t = ctx.timings()
        calls += 1
        map_ms += t["map_ms"]
        asm_ms += t["assemble_ms"]
        evals += sum(t["leapfrogs"])
        if time.perf_counter() - t0 >= min_seconds:
            break
    stop.record()
    torch.cuda.synchronize(dev)
    host_s = time.perf_counter() - t0
    ev_s = start.elapsed_time(stop) / 1e3
    res = np.frombuffer(out.cpu().numpy().tobytes(), MAP_RESULT_DTYPE)
    return {
        "workload": name, "taxids": n, "calls": calls, "event_s": round(ev_s, 4), "host_s": round(host_s, 4),
        "ms_per_call": round(ev_s * 1e3 / calls, 3), "map_ms_per_call": round(map_ms / calls, 3),
        "assemble_ms_per_call": round(asm_ms / calls, 3),
        "taxids_per_s": round(n * calls / ev_s), "fits_per_s": round(6 * n * calls / ev_s),
        "grad_evals_per_s": round(evals / ev_s), "grad_evals_per_taxid": round(evals / (n * calls), 1),
        "valid_share": round(float(np.mean((res["status"] & 0x12) == 0)), 4),
    }


def time_profile(ctx, dev, name, tid, k, N, min_seconds):
    import torch

    from metadamage_b200._abi import MAP_INTERVAL_DTYPE, MAP_RESULT_DTYPE, PROFILE_AT_BOUND

    n = len(tid)
    dt, dk, dN = to_device(dev, tid, k, N)
    rows = torch.empty(n * MAP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    ctx.map_batch_device(dt, dk, dN, rows)
    out = torch.empty(n * MAP_INTERVAL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    ctx.map_profile_device(dk, dN, rows, out)  # warm-up at this size
    torch.cuda.synchronize(dev)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, kern_ms, evals = 0, 0.0, 0
    t0 = time.perf_counter()
    start.record()
    while True:
        ctx.map_profile_device(dk, dN, rows, out)
        t = ctx.timings()
        calls += 1
        kern_ms += t["map_ms"]
        evals += sum(t["leapfrogs"])
        if time.perf_counter() - t0 >= min_seconds:
            break
    stop.record()
    torch.cuda.synchronize(dev)
    host_s = time.perf_counter() - t0
    ev_s = start.elapsed_time(stop) / 1e3
    iv = np.frombuffer(out.cpu().numpy().tobytes(), MAP_INTERVAL_DTYPE)
    ends = iv["end"][:, 0]
    return {
        "workload": name, "taxids": n, "calls": calls, "event_s": round(ev_s, 4), "host_s": round(host_s, 4),
        "ms_per_call": round(ev_s * 1e3 / calls, 3), "profile_kernel_ms_per_call": round(kern_ms / calls, 3),
        "taxids_per_s": round(n * calls / ev_s), "ends_per_s": round(6 * n * calls / ev_s),
        "grad_evals_per_s": round(evals / ev_s), "grad_evals_per_taxid": round(evals / (n * calls), 1),
        "interval_valid_share": round(float(np.mean((iv["status"] & 0x41) == 0)), 4),
        "all_position_ends_at_bound_share": round(float(np.mean((ends["flags"] & PROFILE_AT_BOUND) != 0)), 5),
        "ends_at_bound_share": round(float(np.mean((iv["end"]["flags"] & PROFILE_AT_BOUND) != 0)), 5),
    }


def time_fit(ctx, dev, tid, k, N):
    import torch

    from metadamage_b200._abi import FIT_RESULT_DTYPE

    n, R = k.shape
    dt, dk, dN = to_device(dev, tid, k, N)
    out = torch.empty(n * FIT_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    med = torch.empty((3, n, R), dtype=torch.float32, device=dev)
    ctx.fit_batch_device(dt, dk, dN, out, median=med[0], hpdi_lo=med[1], hpdi_hi=med[2])  # warm-up step
    torch.cuda.synchronize(dev)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    start.record()
    ctx.fit_batch_device(dt, dk, dN, out, median=med[0], hpdi_lo=med[1], hpdi_hi=med[2])
    stop.record()
    torch.cuda.synchronize(dev)
    host_s = time.perf_counter() - t0
    ev_s = start.elapsed_time(stop) / 1e3
    return {"workload": "cfg2", "taxids": n, "event_s": round(ev_s, 4), "host_s": round(host_s, 4), "taxids_per_s": round(n / ev_s)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--min-seconds", type=float, default=1.0, help="timed work per size")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from metadamage_b200.backend import Context

    if not torch.cuda.is_available():
        raise SystemExit("bench_map: no CUDA device")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    ctx = Context(0)
    small = cfg2_batch(10_000)
    from metadamage_b200 import synthetic as syn

    large = syn.dense_fit_batch_shares(1_000_000, 8)
    sizes = [time_map(ctx, dev, "cfg2", *small, args.min_seconds), time_map(ctx, dev, "cfg3", *large, args.min_seconds)]
    profile = [time_profile(ctx, dev, "cfg2", *small, args.min_seconds), time_profile(ctx, dev, "cfg3", *large, args.min_seconds)]
    fit = time_fit(ctx, dev, *small)
    ctx.close()
    line = {
        "metric": "mdg_map_batch and mdg_map_profile (level 0.68) throughput, device-resident inputs, 1 GPU",
        "gpu": info["name"], "power_limit": info["power.limit"], "sm_clock": info["clocks.sm"], "sm_clock_max": info["clocks.max.sm"],
        "sizes": sizes,
        "profile_sizes": profile,
        "profile_vs_map_time": [round(p["ms_per_call"] / m["ms_per_call"], 2) for p, m in zip(profile, sizes)],
        "fit_batch_step": fit,
        "map_vs_fit_speedup_10k": round(fit["event_s"] / (sizes[0]["event_s"] / sizes[0]["calls"]), 1),
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
