"""Is a straggler chain posterior-driven or chain luck? The same counts under 64 different Philox keys (development tool)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metadamage_b200 import _lib
from metadamage_b200.backend import Context
K0 = np.array([2, 1, 2, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 1, 1, 2, 1, 1, 2, 0, 1, 0, 0, 0, 0, 1, 0], np.uint32)
N0 = np.array([5, 4, 6, 1, 1, 2, 1, 1, 2, 7, 2, 1, 3, 3, 3, 2, 3, 3, 6, 1, 2, 3, 2, 6, 3, 3, 3, 2, 6, 4], np.uint32)
TID0 = 100024416
k = np.repeat(K0[None], 64, 0); N = np.repeat(N0[None], 64, 0)
tid = np.arange(64, dtype=np.int64) + 5000
tid[0] = TID0
ctx = Context(0)
out = ctx.fit_batch(tid, k, N, _lib.default_config())
L = out["result"]["run"]["n_leapfrog"]; st = out["result"]["run"]["step_size"]
print("k", K0, "N", N0)
for r in range(6):
    print(r, "leapfrogs: median", np.median(L[:, r]), "max", L[:, r].max(), "orig", L[0, r], "step median", np.median(st[:, r]).round(4), "min", st[:, r].min().round(5))
print("n_div", out["result"]["run"]["n_divergent"].sum(0))
