#!/usr/bin/env python
"""bench.py — TaxID damage fits/sec on N B200s (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference [--max-cores C] ...   # the CPU arm

A "step" is one pass of the hot path over one batch: counts_reduce (K1) over the synthetic mismatch
matrix, then MAP + 6 NUTS runs + WAIC + posterior predictive + row assembly (K3-K7) for every TaxID that
passes the cuts. Steps go through the asynchronous C-ABI (mdg_fit_batch_submit / _wait); `--inflight 2` keeps two
batches in flight per GPU so that the tail of a batch — a handful of long sequential chains — runs under the
next one. The default is 1: with the straggler-free chains of numpyro's default adaptation the overlap costs 2-3 %
(two different NUTS kernels sharing the SMs' instruction caches; profiles/r02_nuts_tuning.md) and buys nothing.
All K steps are inside the timed region and the last one is drained before the clock stops.

Workload: N = 1 -> BASELINE config 2 (10 000 fitted TaxIDs, seed 20240001, +-15 positions).
          N > 1 -> BASELINE config 3's generator (seed 20240002, min-alignments 10, min-y-sum 10), partitioned
                   by TaxID over the GPUs: rank r fits its own contiguous share (`--taxa-per-gpu`, default
                   125 000 = 1M / 8; the r-th jumped Philox block of the seed), so at N = 8 every step IS one pass
                   over config 3's 1M TaxIDs (`cfg3_full_pass` repeats that reading of the line; with another
                   `--taxa-per-gpu` the full-size pass is timed on its own). Batches of that size also keep the
                   workload's straggler chains (up to 850 000 leapfrogs in one run; mean 9 800) inside the step.

  value            whole-job fits/s with inputs resident in HBM (device pointers through the C-ABI)
  e2e              the same through the host-buffer C-ABI calls (pinned host inputs and outputs, H2D + D2H
                   inside the timed region)
  e2e_seam         N = 1: wall time of the reference-facing Python seams counts.compute_counts_with_dask(cfg) +
                   fits.compute_fits(df_counts, cfg) on the same workload written as a TSV file
  roofline         the dominant kernel (NUTS): SURVEY.md 8d flop model x gradient evaluations counted by the
                   kernel / time during which a NUTS kernel was running (CUDA events on the launch streams),
                   against the FP64 FMA peak measured live on this GPU (SM clock sampled during that kernel)
  roofline_counts  K1 on the 10M-row stress input (BASELINE config 5): 111 algorithmic B/row against
                   MEASURED_PEAKS.json hbm_gbs
  cpu_baseline     the reference on the host cores: numpyro itself if `import numpyro, jax` works (probed at run
                   time), else the C restatement (oracle), on a bounded sample of the same workload
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "taxid_damage_fits_per_sec"
UNIT = "fits/s"
ALGO_BYTES_PER_ROW = 111  # SURVEY.md 8d
# SURVEY.md 8d nominal FP64 flop model per log-density-gradient evaluation
FLOPS_PER_GRAD = {0: 300 * 30 + 55, 1: 190 * 30 + 165, 2: 300 * 15 + 55, 3: 190 * 15 + 165, 4: 300 * 15 + 55, 5: 190 * 15 + 165}
NCU_METRICS = os.path.join(ROOT, "profiles", "r02_ncu_metrics.json")  # written by tools/ncu_metrics.py from the .ncu-rep files
DUMP_BYTES = 64 * 10**6  # --dump-outputs: bytes written in all


def model_flops(leapfrogs, max_position):
    scale = max_position / 15.0
    return sum(l * (FLOPS_PER_GRAD[r] * scale) for r, l in enumerate(leapfrogs))


def workload(args, rank, world, n_fit=None):
    """Rank `rank`'s share of the workload (see the module docstring)."""
    from metadamage_b200 import synthetic as syn

    n_fit = n_fit or args.taxa_per_gpu
    if world == 1:
        return syn.make_mismatch_matrix(0, max_position=args.max_position, seed=syn.SEEDS["cfg2"], n_fit=n_fit)
    return syn.make_mismatch_matrix(0, max_position=args.max_position, seed=syn.SEEDS["cfg3"], n_fit=n_fit, jump=rank,
                                    tax_id_start=1 + rank * 100_000_000)


def workload_config(args, world):
    """The same dict for the GPU arm and the reference arm (the driver compares them)."""
    P = args.max_position
    if world == 1:
        what = f"cfg2: synthetic heavy-tailed mismatch matrix, seed 20240001, {args.taxa_per_gpu} fitted TaxIDs"
    else:
        what = (f"cfg3 share: synthetic heavy-tailed mismatch matrix, seed 20240002, min-alignments 10, min-y-sum 10, partitioned by "
                f"TaxID over {world} GPUs, {args.taxa_per_gpu} fitted TaxIDs per GPU and step")
    return {
        "workload": what + f", +-{P} positions, counts + MAP + 6 NUTS runs (500 warm-up + 1000 draws) + WAIC + predictive D_max",
        "taxa_per_gpu": args.taxa_per_gpu, "max_position": P,
        "partition": f"by TaxID over {world} GPU(s), no collective on the fit path",
        "pipelining": f"{args.inflight} batch(es) in flight per GPU (mdg_fit_batch_submit / _wait); every step is drained inside the timed region",
        "l2": "flushed between steps (256 MiB write); the counts inputs (>= 133 MB) exceed L2 as well"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period_ms=200):
        self.device = device
        self.period_ms = period_ms
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_metric(kernel, key):
    """A per-launch figure from the tool-generated summary of the committed ncu captures (None if absent)."""
    try:
        return json.load(open(NCU_METRICS))[kernel][key]
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------------------
# the CPU arm
# --------------------------------------------------------------------------------------------------------------
def sample_size(n_fit, cores):
    """ONE rule for every CPU leg: 64 TaxIDs per host thread (about 10 s of work), at most the whole workload."""
    return max(8, min(int(n_fit), 64 * int(cores)))


def cpu_baseline(g, cores, n_sample=None):
    """The reference's algorithm on the host cores, on a bounded, evenly spread sample of the TaxIDs the GPU fits.
    numpyro itself when it can be imported (kind "reference"), else the C restatement (kind "port")."""
    sel = np.flatnonzero(g["passes"])
    n_sample = n_sample or sample_size(len(sel), cores)
    pick = sel[np.linspace(0, len(sel) - 1, n_sample).astype(int)]
    from oracle import numpyro_arm

    numpyro, why = numpyro_arm.probe()
    if numpyro is not None and g["k"].shape[1] == 30:
        try:
            n_ref = max(200, min(n_sample, 256))
            pick_ref = sel[np.linspace(0, len(sel) - 1, n_ref).astype(int)]
            rows, t_first, t_rest = numpyro_arm.fit_rows(g["tax_ids"][pick_ref], g["k"][pick_ref], g["N"][pick_ref])
            value = (n_ref - 1) / t_rest
            return {"value": value, "unit": UNIT, "cores": 1, "kind": "reference",
                    "sample": f"{n_ref} of the {len(sel)} fitted TaxIDs, evenly spread; the reference's own fit_single_group_without_timeout "
                              f"(numpyro {numpyro.__version__}), one process; first fit incl. jit {t_first:.1f} s, the others {t_rest:.1f} s; "
                              f"including the first fit: {n_ref / (t_first + t_rest):.3f} fits/s"}, t_first + t_rest
        except Exception as exc:  # the probe found the modules but the reference does not run on them
            why = f"numpyro importable but the reference did not run: {type(exc).__name__}: {exc}"
    from oracle import oracle as O

    # loads the library the build left; nothing is compiled at run time, the tree may be read-only
    cfg = O.default_config()
    t0 = time.perf_counter()
    out = O.fit_batch(g["tax_ids"][pick], g["k"][pick], g["N"][pick], cfg, n_threads=cores)
    dt = time.perf_counter() - t0
    ok = int(((out["result"]["status"] & 1) == 0).sum())
    return {"value": n_sample / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_sample} of the {len(sel)} fitted TaxIDs of the same workload, evenly spread (64 per host thread); "
                      f"full fit (MAP + 6 NUTS runs 500+1000 + WAIC + predictive); {dt:.1f} s; {ok} ok; "
                      f"restated reference in C, OpenMP over TaxIDs (numpyro probe: {why})"}, dt


def run_reference(args):
    """The reference arm: the reference's algorithm on the host cores, each step a bounded sample of the same
    workload and configuration as the GPU arm. Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    if world > 1 and args.taxa_per_gpu is None:
        args.taxa_per_gpu = 125_000
    args.taxa_per_gpu = args.taxa_per_gpu or 10_000
    cores = args.max_cores or os.cpu_count() or 1
    # the sample is drawn from rank 0's share of the GPU arm's workload; a bounded share is enough to draw it from
    g = workload(args, 0, world, n_fit=min(args.taxa_per_gpu, 10_000))
    n_fit = int(g["passes"].sum())
    n_sample = sample_size(n_fit, cores)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(g, cores, n_sample=max(4, 2 * cores))
    times, last = [], None
    for _ in range(args.steps):
        last, dt = cpu_baseline(g, cores, n_sample=n_sample)
        times.append(dt)
    n_eff = n_sample if last["kind"] == "port" else None
    value = (n_sample * len(times) / sum(times)) if n_eff else last["value"]
    last["value"] = value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": last,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------
# the GPU arm
# --------------------------------------------------------------------------------------------------------------
def counts_stress(ctx, torch, dev, n_rows=10_000_000, reps=5):
    """BASELINE config 5: 10M-row counts aggregation, device resident, HBM-bound."""
    P = 15
    gen = torch.Generator(device=dev)
    gen.manual_seed(20240004)
    n_tax = (n_rows + 2 * P - 1) // (2 * P)
    tax = torch.repeat_interleave(torch.arange(1, n_tax + 1, device=dev, dtype=torch.int64), 2 * P)[:n_rows].contiguous()
    u = torch.rand(n_tax, device=dev, generator=gen)
    n_al = torch.clamp((10.0 / (1.0 - u) ** (1 / 1.1)), 10, 6e7).to(torch.int32)
    n_al_row = torch.repeat_interleave(n_al, 2 * P)[:n_rows].contiguous()
    pos = torch.arange(n_rows, device=dev) % (2 * P)
    is_rev = (pos >= P).to(torch.uint8)
    pos0 = (pos % P).to(torch.uint8)
    frac = torch.rand((16, n_rows), device=dev, generator=gen) * 0.05
    frac[::5] = 0.2  # the diagonal carries the coverage
    counts16 = (frac * n_al_row.to(torch.float32)[None, :]).to(torch.int32).contiguous()
    cols = dict(tax_id=tax, n_alignments=n_al_row, is_reverse=is_rev, pos0=pos0, counts16=counts16)
    outs = dict(
        n_fwd_ref=torch.empty(n_rows, dtype=torch.int32, device=dev), n_rev_ref=torch.empty(n_rows, dtype=torch.int32, device=dev),
        f_fwd=torch.empty(n_rows, dtype=torch.float32, device=dev), f_rev=torch.empty(n_rows, dtype=torch.float32, device=dev),
        z=torch.empty(n_rows, dtype=torch.int8, device=dev), y_sum_total=torch.empty(n_rows, dtype=torch.int64, device=dev),
        keep=torch.empty(n_rows, dtype=torch.uint8, device=dev), tax_id=torch.empty(n_tax, dtype=torch.int64, device=dev),
        n_alignments=torch.empty(n_tax, dtype=torch.int32, device=dev), first_row=torch.empty(n_tax, dtype=torch.int64, device=dev),
        k=torch.empty((n_tax, 2 * P), dtype=torch.int32, device=dev), N=torch.empty((n_tax, 2 * P), dtype=torch.int32, device=dev),
    )
    times = []
    kept = 0
    for _ in range(reps + 2):
        kept = ctx.counts_reduce_device(cols, outs)
        times.append(ctx.timings()["counts_ms"])
    ms = float(np.mean(times[2:]))
    peak, which = hbm_peak()
    achieved = ALGO_BYTES_PER_ROW * n_rows / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": ncu_metric("counts", "dram_bytes_per_launch") if n_rows == 10_000_000 else None,
            "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, read by tools/ncu_metrics.py from the committed "
                              "ncu --set full capture (profiles/r02_ncu_metrics.json); null if that file is absent",
            "kernel": "counts_stream_kernel + scans + permute (K1) of one mdg_counts_reduce call", "rows": n_rows, "kept_taxa": int(kept), "kernel_ms": ms,
            "algorithmic_bytes_per_row": ALGO_BYTES_PER_ROW, "peak_source": which,
            "note": "inputs (780 MB) exceed L2; mean of %d calls after 2 warm-ups, CUDA events on the launch stream" % reps}


class DeviceBatch:
    """Device-resident inputs of one workload plus two sets of output buffers (two steps are in flight)."""

    def __init__(self, torch, dev, g, R, n_sets=2):
        from metadamage_b200._abi import FIT_RESULT_DTYPE

        n_rows, n_in_tax = len(g["tax_id"]), len(g["tax_ids"])
        self.n_rows, self.n_in_tax = n_rows, n_in_tax
        self.cols = dict(
            tax_id=torch.from_numpy(g["tax_id"]).to(dev), n_alignments=torch.from_numpy(g["n_alignments"].view(np.int32)).to(dev),
            is_reverse=torch.from_numpy(g["is_reverse"]).to(dev), pos0=torch.from_numpy(g["pos0"]).to(dev),
            counts16=torch.from_numpy(g["counts16"].view(np.int32)).to(dev))
        self.sets = []
        for _ in range(n_sets):
            outs = dict(
                n_fwd_ref=torch.empty(n_rows, dtype=torch.int32, device=dev), n_rev_ref=torch.empty(n_rows, dtype=torch.int32, device=dev),
                f_fwd=torch.empty(n_rows, dtype=torch.float32, device=dev), f_rev=torch.empty(n_rows, dtype=torch.float32, device=dev),
                z=torch.empty(n_rows, dtype=torch.int8, device=dev), y_sum_total=torch.empty(n_rows, dtype=torch.int64, device=dev),
                keep=torch.empty(n_rows, dtype=torch.uint8, device=dev), tax_id=torch.empty(n_in_tax, dtype=torch.int64, device=dev),
                n_alignments=torch.empty(n_in_tax, dtype=torch.int32, device=dev), first_row=torch.empty(n_in_tax, dtype=torch.int64, device=dev),
                k=torch.empty((n_in_tax, R), dtype=torch.int32, device=dev), N=torch.empty((n_in_tax, R), dtype=torch.int32, device=dev),
                noise=torch.empty((n_in_tax, 3), dtype=torch.float64, device=dev))
            self.sets.append(dict(outs=outs, res=torch.empty(n_in_tax * FIT_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev),
                                  med=torch.empty((3, n_in_tax, R), dtype=torch.float32, device=dev)))
        self.last = None  # (output set, fitted TaxIDs) of the last step submitted


def device_step_outputs(s, n_fit):
    """The outputs of one device-resident step as float32 / float64 host arrays: the per-TaxID group (the
    counts that fed the fit, every field of the fit result rows, the predictive median and HPDI) and the
    per-input-row group of the counts stage."""
    from metadamage_b200._abi import FIT_RESULT_DTYPE

    def host(t, dtype, view=None):  # device tensor -> host array; `view`: the unsigned type its bits hold
        a = t.cpu().numpy()
        return (a if view is None else a.view(view)).astype(dtype)

    o = s["outs"]
    taxa = {"counts_tax_id": host(o["tax_id"][:n_fit], np.float64), "counts_k": host(o["k"][:n_fit], np.float64, np.uint32),
            "counts_N": host(o["N"][:n_fit], np.float64, np.uint32), "counts_noise": host(o["noise"][:n_fit], np.float64)}
    res = s["res"][:n_fit * FIT_RESULT_DTYPE.itemsize].cpu().numpy().view(FIT_RESULT_DTYPE)
    for name in FIT_RESULT_DTYPE.names:
        if name == "run":
            for diag in res["run"].dtype.names:
                taxa[f"fit_run_{diag}"] = res["run"][diag].astype(np.float64)  # [n_fit][6 runs]
        else:
            taxa[f"fit_{name}"] = res[name].astype(np.float64)
    for i, name in enumerate(("median", "hpdi_lo", "hpdi_hi")):
        taxa[f"fit_{name}"] = host(s["med"][i, :n_fit], np.float32)
    rows = {"counts_n_fwd_ref": host(o["n_fwd_ref"], np.float64, np.uint32), "counts_n_rev_ref": host(o["n_rev_ref"], np.float64, np.uint32),
            "counts_f_fwd": host(o["f_fwd"], np.float32), "counts_f_rev": host(o["f_rev"], np.float32), "counts_z": host(o["z"], np.float32),
            "counts_y_sum_total": host(o["y_sum_total"], np.float64, np.uint64), "counts_keep": host(o["keep"], np.float32)}
    return [taxa, rows]


def finite_parts(group):
    """Every file of a dump holds finite numbers. An array with NaN or +-inf entries (the noise statistic is NaN,
    as in the reference, for a TaxID without usable mismatch counts) is written with 0 in their place, beside
    <name>_nonfinite holding what each entry was: 0 finite, 1 NaN, 2 +inf, 3 -inf."""
    out = {}
    for name, a in group.items():
        bad = ~np.isfinite(a)
        if bad.any():
            out[name + "_nonfinite"] = np.where(np.isnan(a), 1, np.where(a == np.inf, 2, np.where(bad, 3, 0))).astype(np.float32)
            a = np.where(bad, 0, a).astype(a.dtype)
        out[name] = a
    return out


def dump_outputs(directory, groups, budget, seed=0):
    """Write every array of `groups` (dicts of arrays that share their first axis) as directory/<name>.npy, made
    finite by `finite_parts`. The groups are taken in order; one that does not fit in what is left of `budget`
    bytes (files, headers included) is cut to a fixed, seeded sample of its rows, the same rows in each of its
    arrays, so equal runs write equal files."""
    os.makedirs(directory, exist_ok=True)
    for group in groups:
        group = finite_parts(group)
        n = len(next(iter(group.values())))
        total = sum(a.nbytes for a in group.values())
        room = max(budget - 256 * len(group), 0)  # an .npy header takes 128 bytes
        keep = n if total <= room else room // -(-total // n)
        if keep < n:
            rows = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
            group = {name: a[rows] for name, a in group.items()}
        for name, a in group.items():
            path = os.path.join(directory, name + ".npy")
            np.save(path, np.ascontiguousarray(a))
            budget -= os.path.getsize(path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--taxa-per-gpu", type=int, default=None,
                    help="fitted TaxIDs per GPU per step (default: 10 000 = cfg2 on 1 GPU, 125 000 = 1M / 8 of cfg3's generator on N > 1)")
    ap.add_argument("--max-position", type=int, default=15)
    ap.add_argument("--max-cores", type=int, default=0, help="host threads of the CPU arm (default: all; the reference CLI's --max-cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-counts-stress", action="store_true")
    ap.add_argument("--no-seam", action="store_true")
    ap.add_argument("--no-full-pass", action="store_true", help="skip the 1M-TaxID single pass at N = 8")
    ap.add_argument("--full-pass-taxa", type=int, default=None,
                    help="fitted TaxIDs per GPU of the extra single pass (default: 125 000 at N = 8 = BASELINE config 3's 1M TaxIDs, none otherwise)")
    ap.add_argument("--inflight", type=int, default=1, choices=[1, 2], help="batches in flight per GPU (MDG_MAX_INFLIGHT = 2)")
    ap.add_argument("--heuristic", type=int, default=0, help="find_heuristic_step_size (0 = numpyro 0.4.1 default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the device-resident path returned in its last timed step to DIR/<name>.npy "
                         "(finite float32 / float64, NaN and inf marked in <name>_nonfinite.npy; at most 64 MB; "
                         "under torchrun DIR/rank<r>/)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from metadamage_b200 import _lib
    from metadamage_b200._abi import FIT_RESULT_DTYPE
    from metadamage_b200.backend import Context

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.taxa_per_gpu is None:
        args.taxa_per_gpu = 10_000 if world == 1 else 125_000
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctx = Context(local_rank)
    # the ctx stream carries K1 and the copies; like the library's own short-kernel streams it outranks the persistent
    # NUTS launches of the batch in flight, whose waiting CTAs would otherwise be served first
    stream = torch.cuda.Stream(dev, priority=-1)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    cfg = _lib.default_config(find_heuristic_step_size=args.heuristic)
    P = args.max_position
    R = 2 * P

    g = workload(args, rank, world)
    batch = DeviceBatch(torch, dev, g, R, args.inflight)
    n_rows, n_in_tax = batch.n_rows, batch.n_in_tax
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    stats = {"counts_ms": [], "map_ms": [], "nuts_ms": [], "nuts_union_ms": [], "ppc_ms": [], "assemble_ms": [], "launches": 0,
             "leapfrogs": np.zeros(6)}

    def book(t_counts, t_fit, record):
        if not record:
            return
        if t_counts is not None:
            stats["counts_ms"].append(t_counts["counts_ms"])
            stats["launches"] += t_counts["n_launches"]
        if t_fit is not None:
            for key in ("map_ms", "nuts_ms", "nuts_union_ms", "ppc_ms", "assemble_ms"):
                stats[key].append(t_fit[key])
            stats["launches"] += t_fit["n_launches"]
            stats["leapfrogs"] += np.array(t_fit["leapfrogs"], dtype=np.float64)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def run_pipelined(steps, submit, record=True):
        """`submit(i)` enqueues step i and returns (n_fit, ticket, counts timings); at most two steps in flight."""
        pending, n, last = [], 0, None
        for i in range(steps):
            if len(pending) == args.inflight:
                last = ctx.fit_wait(pending.pop(0))
                book(None, last["timings"], record)
            n_fit, ticket, t_counts = submit(i)
            book(t_counts, None, record)
            n += n_fit
            pending.append(ticket)
        while pending:
            last = ctx.fit_wait(pending.pop(0))
            book(None, last["timings"], record)
        return n, last

    def timed(steps, submit, record=True):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        n, last = run_pipelined(steps, submit, record)
        e1.record(stream)  # fit_wait ordered the ctx stream after every batch
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        cnt = torch.tensor([float(n)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        return float(ms.item()), float(cnt.item()), last

    def make_submit_device(b, fit_cfg):
        def submit(i):
            s = b.sets[i % len(b.sets)]
            flush.zero_()  # evict L2 between steps
            n_fit = ctx.counts_reduce_device(b.cols, s["outs"])
            t1 = ctx.timings()
            o = s["outs"]
            ticket = ctx.fit_submit_device(o["tax_id"][:n_fit], o["k"][:n_fit], o["N"][:n_fit], s["res"], fit_cfg,
                                           median=s["med"][0], hpdi_lo=s["med"][1], hpdi_hi=s["med"][2], noise3=o["noise"][:n_fit])
            b.last = (s, n_fit)
            return n_fit, ticket, t1
        return submit

    # ---------------- device-resident path (value) ----------------
    submit_device = make_submit_device(batch, cfg)
    if args.warmup:
        run_pipelined(args.warmup, submit_device, record=False)
    sampler = ClockSampler(local_rank).start()
    dev_ms, dev_fits, _ = timed(args.steps, submit_device)
    if args.dump_outputs:  # before the paths below reuse the output buffers
        where = args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}")
        dump_outputs(where, device_step_outputs(*batch.last), DUMP_BYTES // world)

    # ---------------- host-buffer path (e2e) ----------------
    def pinned(a):
        view = a.view(np.int32) if a.dtype == np.uint32 else a
        t = torch.empty(view.shape, dtype=torch.from_numpy(view[:0].copy()).dtype, pin_memory=True)
        t.numpy()[...] = view
        return t.numpy().view(a.dtype)

    def pinned_empty(shape, dtype):
        shape = shape if isinstance(shape, tuple) else (shape,)
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        t = torch.empty(max(nbytes, 1), dtype=torch.uint8, pin_memory=True)
        return t.numpy()[:nbytes].view(dtype).reshape(shape)

    h = {key: pinned(g[key]) for key in ("tax_id", "n_alignments", "is_reverse", "pos0", "counts16")}
    e2e_bytes = {"h2d": 0, "d2h": 0}
    host_sets = []
    for _ in range(args.inflight):
        host_sets.append(dict(
            counts=dict(
                n_fwd_ref=pinned_empty(n_rows, np.uint32), n_rev_ref=pinned_empty(n_rows, np.uint32), f_fwd=pinned_empty(n_rows, np.float32),
                f_rev=pinned_empty(n_rows, np.float32), z=pinned_empty(n_rows, np.int8), y_sum_total=pinned_empty(n_rows, np.uint64),
                keep=pinned_empty(n_rows, np.uint8), tax_id=pinned_empty(n_in_tax, np.int64), n_alignments=pinned_empty(n_in_tax, np.uint32),
                first_row=pinned_empty(n_in_tax, np.int64), k=pinned_empty((n_in_tax, R), np.uint32), N=pinned_empty((n_in_tax, R), np.uint32),
                noise=pinned_empty((n_in_tax, 3), np.float64)),
            fit=dict(result=pinned_empty(n_in_tax, FIT_RESULT_DTYPE), median=pinned_empty((n_in_tax, R), np.float32),
                     hpdi_lo=pinned_empty((n_in_tax, R), np.float32), hpdi_hi=pinned_empty((n_in_tax, R), np.float32))))

    def submit_host(i):
        s = host_sets[i % len(host_sets)]
        flush.zero_()
        r = ctx.counts_reduce(h["tax_id"], h["n_alignments"], h["is_reverse"], h["pos0"], h["counts16"],
                              max_position=P, want_noise=True, out=s["counts"])
        t1 = ctx.timings()
        ticket = ctx.fit_submit(r["tax_id"], r["k"], r["N"], cfg, noise3=r["noise"], out=s["fit"])
        n_fit = r["n_tax"]
        e2e_bytes["h2d"] = sum(h[key].nbytes for key in h) + n_fit * (8 + 2 * R * 4 + 24)
        e2e_bytes["d2h"] = (n_rows * (4 + 4 + 4 + 4 + 1 + 8 + 1) + n_fit * (8 + 4 + 8 + 2 * R * 4 + 24)
                            + n_fit * (FIT_RESULT_DTYPE.itemsize + 3 * R * 4))
        return n_fit, ticket, t1

    run_pipelined(1, submit_host, record=False)
    e2e_ms, e2e_fits, last_host = timed(args.steps, submit_host)
    clocks = sampler.stop()
    chain_leapfrogs = np.array(last_host["result"]["run"]["n_leapfrog"], dtype=np.float64)
    status = np.array(last_host["result"]["status"])

    # ---------------- the north star's reduced unit (SURVEY.md 8d): no forward-only / reverse-only refits ----------------
    submit_reduced = make_submit_device(batch, cfg.copy(do_fwd_rev=0))
    run_pipelined(1, submit_reduced, record=False)
    red_ms, red_fits, _ = timed(1, submit_reduced, record=False)

    # ---------------- N = 8: one full-size pass of BASELINE config 3 (1M TaxIDs over the box) ----------------
    full_pass = None
    n_full = args.full_pass_taxa if args.full_pass_taxa is not None else (1_000_000 // world if world == 8 else 0)
    steps_are_full_passes = n_full > 0 and n_full == args.taxa_per_gpu
    if n_full > 0 and not args.no_full_pass and not steps_are_full_passes:
        del batch, submit_device, submit_reduced
        torch.cuda.empty_cache()
        gf = workload(args, rank, world, n_fit=n_full)
        bf = DeviceBatch(torch, dev, gf, R, 1)
        submit_full = make_submit_device(bf, cfg)
        run_pipelined(1, submit_full, record=False)
        fs = ClockSampler(local_rank).start()
        t_wall = time.perf_counter()
        full_ms, full_fits, _ = timed(1, submit_full, record=False)
        t_wall = time.perf_counter() - t_wall
        full_pass = {"taxids": int(full_fits), "ms": full_ms, "value": full_fits / (full_ms * 1e-3), "unit": UNIT, "steps": 1,
                     "wall_s_incl_barriers": t_wall, "clocks": fs.stop(),
                     "what": f"ONE pass over {n_full * world} fitted TaxIDs ({n_full} per GPU, cfg3 generator, seed 20240002, rank r = jumped block r), "
                             "device resident, after one untimed pass; max over ranks of the CUDA-event time"}

    # ---------------- longest chain (a step's tail is a few sequential Markov chains) ----------------
    chain_max = torch.tensor([chain_leapfrogs.max()], dtype=torch.float64, device=dev)
    chain_sum = torch.tensor([chain_leapfrogs.sum(), float(chain_leapfrogs.size)], dtype=torch.float64, device=dev)
    # per-rank roofline inputs: NUTS-active seconds and model flops of this rank's timed device + host steps
    nuts_s = float(np.sum(stats["nuts_union_ms"])) * 1e-3
    flops = model_flops(list(stats["leapfrogs"]), P)
    rank_tf = torch.tensor([flops / nuts_s / 1e12 if nuts_s > 0 else 0.0], dtype=torch.float64, device=dev)
    all_tf = [rank_tf.clone() for _ in range(world)]
    if world > 1:
        dist.all_reduce(chain_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(chain_sum, op=dist.ReduceOp.SUM)
        dist.all_gather(all_tf, rank_tf)
    per_rank_tf = [float(t.item()) for t in all_tf]
    chain_stats = {"mean_leapfrogs_per_chain": float(chain_sum[0].item() / chain_sum[1].item()),
                   "max_leapfrogs_of_one_chain": float(chain_max.item()),
                   "failed_fits_rank0": int((status & 1).sum()),
                   "note": "a chain is sequential: a batch ends with its longest chains (--inflight 2 runs them under the next batch)"}

    # ---------------- rooflines, seam, CPU baseline (rank 0 only) ----------------
    if rank == 0:
        peak_sampler = ClockSampler(local_rank, period_ms=50).start()
        fp64_peak = max(ctx.fp64_peak_tflops() for _ in range(12))  # ~1 s of DFMA so that the clock sampler sees it
        peak_clocks = peak_sampler.stop()
        evals = float(stats["leapfrogs"].sum())
        achieved = per_rank_tf[0]
        roofline = {
            "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
            "traffic": ncu_metric("nuts", "dram_bytes_per_launch"),
            "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one NUTS launch, read by tools/ncu_metrics.py from the committed "
                              "ncu --set full capture (profiles/r02_ncu_metrics.json); null if that file is absent",
            "kernel": "nuts_group_kernel<PMD|null, 8 lanes per chain> (one launch and one queue per model and batch)",
            "flop_model": "SURVEY.md 8d nominal: PMD 300*n_obs+55, null 190*n_obs+165 flop per gradient evaluation",
            "gradient_evaluations": evals,
            "nuts_active_s": nuts_s,
            "gradient_evaluations_per_s": evals / nuts_s if nuts_s > 0 else 0.0,
            "time_base": "union over the pipelined batches of the CUDA-event intervals [first NUTS launch, last NUTS launch done] "
                         "(mdg_timings.nuts_union_ms), device and host steps of the timed regions",
            "peak_source": "FP64 FMA peak measured live on this GPU (mdg_measure_fp64_peak, best of 12 x 3 launches); not in MEASURED_PEAKS.json",
            "peak_clocks": peak_clocks,
            "over_ranks": {"min": min(per_rank_tf), "mean": float(np.mean(per_rank_tf)), "max": max(per_rank_tf), "unit": "TFLOP/s"},
            "note": "HBM traffic of the fit kernels is negligible (240 B in, ~1 KB out per TaxID): compute bound, no tensor cores",
        }
        roofline_counts = None if args.no_counts_stress else counts_stress(ctx, torch, dev)
        seam = None
        if world == 1 and not args.no_seam:
            seam = seam_timing(g, args, e2e_ms / args.steps)
        cpu = None
        if not args.no_cpu_baseline:
            cpu, _ = cpu_baseline(g, args.max_cores or os.cpu_count() or 1)
        per_step = lambda key: float(np.mean(stats[key])) if stats[key] else 0.0  # noqa: E731
        line = {
            "metric": METRIC, "value": dev_fits / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "input_shape_rank0": {"input_taxids": n_in_tax, "rows": n_rows},
            "e2e": {"value": e2e_fits / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(e2e_bytes["h2d"]),
                    "d2h_bytes_per_step": int(e2e_bytes["d2h"]), "ms_per_step": e2e_ms / args.steps},
            "e2e_seam": seam,
            "gpu_launches": int(stats["launches"]),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_counts": roofline_counts,
            "chains": chain_stats,
            "reduced_unit": {"value": red_fits / (red_ms * 1e-3), "unit": UNIT, "ms_per_step": red_ms, "steps": 1,
                             "what": "counts + MAP + PMD/null NUTS on all positions + WAIC + predictive D_max, WITHOUT the forward-only / "
                                     "reverse-only refits of fits.py:298-356 (the north star's reduced unit; `value` above is the full fit); "
                                     "one step"},
            "cfg3_full_pass": full_pass if not steps_are_full_passes else {
                "taxids": int(dev_fits / args.steps), "ms": dev_ms / args.steps, "value": dev_fits / (dev_ms * 1e-3), "unit": UNIT,
                "steps": args.steps, "clocks": clocks,
                "what": f"every timed step of this line is one pass over {n_full * world} fitted TaxIDs ({n_full} per GPU, cfg3 generator, "
                        "seed 20240002, rank r = jumped block r), device resident: `value` / `ms_per_step` repeated"},
            "cpu_baseline": cpu,
            "kernel_ms_per_step": {"counts": per_step("counts_ms"), "map": per_step("map_ms"), "nuts": per_step("nuts_ms"),
                                   "nuts_union": per_step("nuts_union_ms"), "ppc": per_step("ppc_ms"), "assemble": per_step("assemble_ms")},
            "find_heuristic_step_size": args.heuristic,
        }
        print(json.dumps(line), flush=True)
    barrier()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def seam_timing(g, args, abi_e2e_ms):
    """Wall time of the reference-facing seams on the same workload as a file: counts.compute_counts_with_dask(cfg)
    (file -> df_counts: GPU tokeniser + K1 + DataFrame) and fits.compute_fits(df_counts, cfg, mcmc_kwargs)
    (df_counts -> two DataFrames), the calls main.py:57,66 make. The median of three runs (after a warm-up run) is reported."""
    import tempfile

    from metadamage_b200 import counts, fits, synthetic as syn, utils

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "cfg2.mismatch.txt")
        syn.write_tsv(g, path)
        cfg = utils.Config(out_dir=os.path.join(tmp, "out"), max_fits=None, max_cores=1, max_position=args.max_position, min_alignments=10,
                           min_y_sum=10, substitution_bases_forward="CT", substitution_bases_reverse="GA", forced=True, version="bench")
        cfg.add_filename(path)
        runs = []
        for rep in range(4):  # one warm-up, three timed: the median run is reported
            t0 = time.perf_counter()
            df_counts = counts.compute_counts_with_dask(cfg)
            t1 = time.perf_counter()
            df_res, df_pred = fits.compute_fits(df_counts, cfg, fits.mcmc_kwargs_default())
            t2 = time.perf_counter()
            if rep > 0:
                runs.append({"counts_s": t1 - t0, "fits_s": t2 - t1, "total_s": t2 - t0, "fitted_taxids": int(len(df_res)),
                             "df_counts_rows": int(len(df_counts)), "file_bytes": os.path.getsize(path)})
        runs.sort(key=lambda r: r["total_s"])
        out = dict(runs[len(runs) // 2])
        out["runs_total_s"] = [r["total_s"] for r in runs]
    out["value"] = out["fitted_taxids"] / out["total_s"]
    out["unit"] = UNIT
    out["overhead_vs_abi_e2e"] = out["total_s"] / (abi_e2e_ms * 1e-3) - 1.0
    out["what"] = ("wall clock of counts.compute_counts_with_dask(cfg) + fits.compute_fits(df_counts, cfg, mcmc_kwargs) on the cfg2 workload "
                   "written as a 22-column TSV (file read, GPU tokeniser, K1, DataFrames, K3-K7, result DataFrames included), "
                   "median of three runs after one warm-up run; overhead is relative to one C-ABI e2e step")
    return out


def _json_only_stdout():
    """stdout carries ONE JSON line: library chatter written to file descriptor 1 (NCCL prints its version
    there under torchrun) is sent to stderr; print() keeps the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real


if __name__ == "__main__":
    _json_only_stdout()
    main()
