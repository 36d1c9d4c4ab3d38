"""What each rank of the weak-scaling bench sees, measured on ONE GPU: the 10 000-TaxID shard of rank
r (bench.workload seeds) is reduced and fitted, the step time and the longest chains are printed.
The step of an N-GPU bench is the max over its ranks' lines (development tool; on the GPU box).

usage: python tools/shard_probe.py [ranks, e.g. 0-7] [taxa_per_gpu]"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from metadamage_b200 import _lib  # noqa: E402
from metadamage_b200.backend import Context  # noqa: E402

spec = sys.argv[1] if len(sys.argv) > 1 else "0-7"
lo, hi = (spec.split("-") + [spec])[:2]
args = argparse.Namespace(max_position=15, taxa_per_gpu=int(sys.argv[2]) if len(sys.argv) > 2 else 10000)
ctx = Context(0)
cfg = _lib.default_config()
# scheduling variants (environment knobs of mdg_fit_batch), e.g. MDG_PROBE_VARIANTS="MDG_NUTS_ORDER=0;MDG_NUTS_ORDER=2,MDG_NUTS_PRIO_FRAC=8"
VARIANTS = [dict(kv.split("=") for kv in v.split(",") if kv) for v in os.environ.get("MDG_PROBE_VARIANTS", "").split(";")] or [{}]
for rank in range(int(lo), int(hi) + 1):
    g = bench.workload(args, rank, 8)
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], want_noise=True)
    best = None
    for variant in VARIANTS:
        for key, val in variant.items():
            os.environ[key] = val
        for rep in range(2):
            t0 = time.perf_counter()
            out = ctx.fit_batch(r["tax_id"], r["k"], r["N"], cfg, noise3=r["noise"])
            wall = (time.perf_counter() - t0) * 1e3
            t = ctx.timings()
            print(f"  rank {rank} {variant} rep {rep}: nuts_ms {t['nuts_ms']:.1f} fit_ms {t['total_ms']:.1f}", flush=True)
            if best is None or t["nuts_ms"] < best[0]:
                best = (t["nuts_ms"], t["total_ms"], wall)
    L = out["result"]["run"]["n_leapfrog"]
    top = np.sort(L.ravel())[::-1][:4]
    i, j = np.unravel_index(np.argmax(L), L.shape)
    # where do the longest chains sit in the coverage ranking? (0 = the TaxID with the fewest reads)
    cov_rank = np.argsort(np.argsort(r["N"].sum(1), kind="stable"), kind="stable") / len(L)
    order = np.argsort(L.max(1))[::-1][:12]
    print("  coverage percentile of the TaxIDs with the 12 longest chains:", np.round(cov_rank[order], 3).tolist(),
          "their N sums:", r["N"].sum(1)[order].tolist(), flush=True)
    print(f"rank {rank}: n_fit {len(L)} nuts_ms {best[0]:.1f} fit_ms {best[1]:.1f} wall_ms {best[2]:.1f} "
          f"mean_leapfrogs {L.mean():.0f} top4 {top.tolist()} longest: TaxID index {i} of {len(L)}, run {j}, "
          f"step size {out['result']['run']['step_size'][i, j]:.4g}", flush=True)
    run = out["result"]["run"]
    print(f"  longest chain's TaxID {int(r['tax_id'][i])}: k {r['k'][i].tolist()} N {r['N'][i].tolist()} leapfrogs per run {L[i].tolist()} "
          f"divergent {run['n_divergent'][i].tolist()} accept {np.round(run['mean_accept'][i], 3).tolist()} step {np.round(run['step_size'][i], 5).tolist()}", flush=True)
