"""-m gpu: the NUTS chains are pinned to the bit. SHA-256 digests of the `result`, `median`, `waic` and `trace` bytes of
`fit_batch` on a few seeded batches are kept in tests/golden/nuts_bits.json; a change to the NUTS kernel that alters
any chain (a reordered sum, a different fma, a moved Philox counter) fails here and has to regenerate the file on
purpose:

    python tests/test_gpu_nuts_bits.py --write     # on the GPU, with the build whose chains are the new reference

The cases cover P = 15, 25 and 40, forward / reverse runs on and off, the step-size heuristic on and off, a batch
that hits `max_leapfrogs_per_run`, and the degenerate inputs of test_gpu_fits.test_degenerate_inputs."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from metadamage_b200 import _lib, synthetic as syn  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "nuts_bits.json")
ARRAYS = ("result", "median", "waic", "trace")

# name -> (P, TaxIDs, seed, fit_config changes); "budget" is resolved against the unlimited fit of the same batch
CASES = {
    "P15_fwdrev1_heur0": (15, 40, 11, dict(num_warmup=120, num_samples=100)),
    "P15_fwdrev0_heur1": (15, 40, 12, dict(num_warmup=120, num_samples=100, do_fwd_rev=0, find_heuristic_step_size=1)),
    "P25_fwdrev1_heur1": (25, 32, 13, dict(num_warmup=100, num_samples=80, find_heuristic_step_size=1)),
    "P40_fwdrev0_heur0": (40, 32, 14, dict(num_warmup=100, num_samples=80, do_fwd_rev=0)),
    "P40_fwdrev1_heur1": (40, 24, 15, dict(num_warmup=80, num_samples=60, find_heuristic_step_size=1)),
    "P15_budget": (15, 48, 71, dict(num_warmup=120, num_samples=100, max_leapfrogs_per_run="budget")),
    "degenerate": (15, 4, None, dict(num_warmup=100, num_samples=100)),
}


def case_inputs(name):
    P, n, seed, _ = CASES[name]
    if seed is None:  # all-zero coverage, k = 0 everywhere, k = N everywhere, half the positions covered
        N = np.zeros((n, 2 * P), np.uint32)
        k = np.zeros((n, 2 * P), np.uint32)
        N[1] = 100
        N[2] = 100
        k[2] = 100
        N[3, :P] = 50
        k[3, :P] = 5
        return np.arange(n), k, N
    tid, k, N, _ = syn.dense_fit_batch(n, max_position=P, seed=seed)
    return tid, k, N


def case_digests(ctx, name):
    tid, k, N = case_inputs(name)
    kw = dict(CASES[name][3])
    if kw.get("max_leapfrogs_per_run") == "budget":
        del kw["max_leapfrogs_per_run"]
        free = ctx.fit_batch(tid, k, N, _lib.default_config(**kw))["result"]
        kw["max_leapfrogs_per_run"] = int(np.median(free["run"]["n_leapfrog"].max(axis=1)))
    out = ctx.fit_batch(tid, k, N, _lib.default_config(**kw), want_trace=True, want_waic=True)
    if "max_leapfrogs_per_run" in kw:
        from metadamage_b200._abi import FIT_BUDGET_EXCEEDED

        hit = (out["result"]["status"] & FIT_BUDGET_EXCEEDED) != 0
        assert 0 < hit.sum() < len(tid), "the budget case must stop some runs and not others"
    return {a: hashlib.sha256(np.ascontiguousarray(out[a]).tobytes()).hexdigest() for a in ARRAYS}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_nuts_outputs_match_recorded_digests(ctx, name):
    with open(GOLDEN) as f:
        want = json.load(f)[name]
    got = case_digests(ctx, name)
    assert got == want, f"{name}: NUTS outputs changed bits in {[a for a in ARRAYS if got[a] != want[a]]}"


if __name__ == "__main__":
    if sys.argv[1:] != ["--write"]:
        sys.exit(f"usage: python {os.path.relpath(__file__, ROOT)} --write")
    from metadamage_b200.backend import Context

    with Context(0) as c:
        table = {name: case_digests(c, name) for name in sorted(CASES)}
    with open(GOLDEN, "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {GOLDEN}: {len(table)} cases")
