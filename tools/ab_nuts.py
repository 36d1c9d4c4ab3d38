"""A/B of the NUTS kernels on the GPU box (development tool): fits `n` TaxIDs of BASELINE config 2 with the library
MDG_LIB_PATH names (e.g. a build of tools/ab_build.sh) and prints the CUDA-event times and leapfrog counts."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metadamage_b200 import _lib, synthetic as syn  # noqa: E402
from metadamage_b200.backend import Context  # noqa: E402

n_fit = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
warm = int(sys.argv[2]) if len(sys.argv) > 2 else 500
samp = int(sys.argv[3]) if len(sys.argv) > 3 else 1000
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 2
tid, k, N, g = syn.dense_fit_batch(n_fit)
ctx = Context(0)
cfg = _lib.default_config(num_warmup=warm, num_samples=samp, do_fwd_rev=int(os.environ.get("MDG_PT_FWD_REV", "1")))
for rep in range(reps):
    t0 = time.perf_counter()
    out = ctx.fit_batch(tid, k, N, cfg)
    wall = time.perf_counter() - t0
    t = ctx.timings()
    res = out["result"]
    lf = sum(t["leapfrogs"])
    print(f"variant={os.environ.get('MDG_VARIANT', '')} rep={rep} nuts_ms={t['nuts_ms']:.1f} total_ms={t['total_ms']:.1f} wall={wall:.3f} "
          f"leapfrogs={lf} Meval/s={lf / t['nuts_ms'] / 1e3:.1f} failed={(res['status'] & 1).sum()} "
          f"max_chain={res['run']['n_leapfrog'].max()} q_mean={np.nanmean(res['q_mean']):.6f} nsig={np.nanmedian(res['n_sigma']):.4f}", flush=True)
