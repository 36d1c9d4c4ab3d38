"""-m gpu: the posterior-predictive kernel K6 (ppc_kernel) draw for draw against the CPU replay of tests/ppc_replay.c,
and its Beta -> Binomial sampler against the oracle's and against scipy.

K6 draws, for every TaxID and predictive item, S beta-binomial variates from a Philox stream fixed by (seed, tax_id,
draw, run, dense position) and the fit's own constrained draws, sorts them and takes the median and the HPDI window.
The replay does the same on the CPU with the oracle's samplers. The two samplers differ only in how they round (the
kernel's table-driven log / exp and Newton reciprocal, a Stirling lgamma): an integer draw can change only where a
uniform lands within a few ulps of an acceptance or inversion threshold, so at the sizes here every draw, and with it
every order statistic, is expected to be identical. A wrong stream word, position, N or window moves some D_max by
about a count, which these comparisons see and the statistical gates of test_gpu_fits.py do not."""
import numpy as np
import pytest

import ppc_replay
from metadamage_b200 import _lib, synthetic as syn
from metadamage_b200._abi import FIT_FAILED
from test_model_reference import MAX_POSITIONS
from test_ppc_replay import SAMPLER_DRAWS, SAMPLER_GRID, check_against_scipy

pytestmark = pytest.mark.gpu

SHORT = dict(num_warmup=100, num_samples=257)


@pytest.fixture(scope="module")
def replay():
    ppc_replay.build()
    return ppc_replay


def predictive_batch(P, seed, n=12):
    """Synthetic TaxIDs; row 1 has no coverage at every third position (dense 0 among them, the reverse strand's
    first position not), row 2 has 10^6 reads at every position, so its draws go through BTRS."""
    tid, k, N, _ = syn.dense_fit_batch(n, max_position=P, seed=seed)
    cut = np.arange(2 * P) % 3 == 0
    cut[P] = False
    N[1, cut] = 0
    k[1, cut] = 0
    x = np.r_[np.arange(P), np.arange(P)]
    N[2] = 1_000_000
    k[2] = np.random.default_rng(seed).binomial(N[2], 0.3 * 0.7 ** x + 0.02)
    return tid, k, N


def check_against_replay(replay, tid, N, cfg, got, tag):
    res = got["result"]
    want = replay.predictive(tid, N, got["samples"], res["status"], cfg)
    bad = replay.mismatches(got, want)
    if bad:
        where = {key: np.argwhere(~np.isclose(got[key], want[key], rtol=0, atol=0, equal_nan=True))[:8].tolist()
                 for key in ("median", "hpdi_lo", "hpdi_hi")}
        raise AssertionError(f"{tag}: {bad} differ from the replay; first (TaxID, position) per array: {where}")
    failed = (res["status"] & FIT_FAILED) != 0
    for key in ("median", "hpdi_lo", "hpdi_hi"):
        assert np.array_equal(np.isnan(got[key]), (N == 0) | failed[:, None]), (tag, key)
    assert np.array_equal(np.isnan(res["D_max"]), (N[:, 0] == 0) | failed), tag
    return want


LAYOUT_CASES = ([(P, 1, 1) for P in MAX_POSITIONS] +
                [(P, quirks, fwd_rev) for P in (1, 15, 64) for quirks, fwd_rev in ((0, 1), (1, 0))])


@pytest.mark.parametrize("P,quirks,fwd_rev", LAYOUT_CASES)
def test_predictive_matches_replay(ctx, replay, P, quirks, fwd_rev):
    """median / hpdi_lo / hpdi_hi (float32) and D_max, D_max_lower_hpdi, D_max_upper_hpdi, D_max_forward,
    D_max_reverse (FP64) of fit_batch equal the replay of the fit's own draws bit for bit, at every lane layout of P.
    In the quirks-on, fwd/rev-on case a leapfrog budget (chosen as in test_leapfrog_budget_is_the_timeout_analogue)
    fails some TaxIDs and not others: their rows are NaN, the others unaffected."""
    tid, k, N = predictive_batch(P, seed=400 + P)
    kw = dict(SHORT, reference_quirks=quirks, do_fwd_rev=fwd_rev)
    if quirks and fwd_rev:
        free = ctx.fit_batch(tid, k, N, _lib.default_config(**kw))["result"]
        kw["max_leapfrogs_per_run"] = int(np.median(free["run"]["n_leapfrog"].max(axis=1)))
    cfg = _lib.default_config(**kw)
    got = ctx.fit_batch(tid, k, N, cfg, want_samples=True)
    failed = (got["result"]["status"] & FIT_FAILED) != 0
    if "max_leapfrogs_per_run" in kw:
        assert 0 < failed.sum() < len(tid), failed
    else:
        assert not failed.any(), failed
    want = check_against_replay(replay, tid, N, cfg, got, (P, quirks, fwd_rev))
    if not failed[2]:  # the high-coverage row drew in BTRS: BINV (n p < 10 at p <= 0.5) never returns more than 2000
        assert want["y"][2, 0].min() > 2000
    if fwd_rev:  # row 1 has no coverage at dense 0 but has it at dense P
        assert np.isnan(got["result"]["D_max_reverse"][1]) == bool(quirks or failed[1])
        assert np.all(np.isfinite(got["result"]["D_max_forward"][~failed & (N[:, 0] > 0)]))
    else:
        assert np.all(np.isnan(got["result"]["D_max_forward"])) and np.all(np.isnan(got["result"]["D_max_reverse"]))


SAMPLE_COUNTS = (1, 2, 3, 31, 32, 33, 63, 64, 65, 1000, 1025, 4096)
HPDI_PROBS = (0.68, 0.5, 0.95, 1.0)


@pytest.mark.parametrize("S", SAMPLE_COUNTS)
def test_sample_count_and_hpdi_boundaries(ctx, replay, S):
    """At P = 15: S below a warp, at the 64-key floor of the sort, at and around each doubling of the padded length,
    odd and even (the median of one or of two middle draws), and each HPDI probability; 1.0 makes the window
    S - 1 draws long. Exact against the replay."""
    tid, k, N = predictive_batch(15, seed=500 + S, n=8)
    for prob in HPDI_PROBS:
        cfg = _lib.default_config(num_warmup=100, num_samples=S, hpdi_prob=prob)
        got = ctx.fit_batch(tid, k, N, cfg, want_samples=True)
        assert not (got["result"]["status"] & FIT_FAILED).any()
        want = check_against_replay(replay, tid, N, cfg, got, (S, prob))
        if prob == 1.0 and S > 1:  # the window spans the sorted draws
            y = np.sort(want["y"][0, 0])
            assert got["result"]["D_max_lower_hpdi"][0] == y[0] / N[0, 0]
            assert got["result"]["D_max_upper_hpdi"][0] == y[-1] / N[0, 0]


@pytest.mark.parametrize("fwd_rev", [1, 0])
def test_scratch_layout_without_samples(ctx, fwd_rev):
    """Without want_samples K6 reads the draws from a 1- or 3-run scratch (sample_slot maps the run kinds onto it);
    with it, from the 6-run output. Rows and predictive arrays are bit-identical either way."""
    tid, k, N = predictive_batch(15, seed=600 + fwd_rev)
    cfg = _lib.default_config(do_fwd_rev=fwd_rev, reference_quirks=0, **SHORT)
    a = ctx.fit_batch(tid, k, N, cfg, want_samples=True)
    b = ctx.fit_batch(tid, k, N, cfg)
    for key in ("result", "median", "hpdi_lo", "hpdi_hi"):
        assert a[key].tobytes() == b[key].tobytes(), (fwd_rev, key)


# ------------------------------------------------------------------ the device sampler
def grid_id(point):
    return "-".join(f"{v:g}" for v in point)


@pytest.mark.parametrize("alpha,beta,n", SAMPLER_GRID, ids=[grid_id(p) for p in SAMPLER_GRID])
def test_device_sampler_matches_oracle_and_scipy(ctx, oracle, alpha, beta, n):
    """mdg_test_betabinom_draws (the kernel's beta_variate and binomial_variate) against the oracle's sampler on the
    same streams, draw for draw, and against scipy's beta-binomial. Identical for n <= 10^6.

    At n = 2^32 - 1 two comparisons cancel, and the two implementations' last-ulp differences can flip a draw there:
    BTRS's h - lgamma(k+1) - lgamma(n-k+1) (terms near 10^11, ~1e-5 apart between the two lgammas) and
    floor(n p + ...), which allow 10^-4 of the draws to differ; and, at shape a ~ 10^11 (phi ~ 10^12), the
    Marsaglia-Tsang acceptance test log u < x^2/2 + d - d v + d log v. The kernel forms d log v as
    d (log(d v) - log d): a few ulps of log d ~ 27 times d ~ 3e11 move the threshold by ~1e-3, and log u has density
    <= 1 there, so each attempt's decision flips with probability ~1e-3 (a flipped attempt redraws from a different
    point of the stream: the two draws then differ by about the sampling spread, not by one). That adds
    2^-52 (alpha |log alpha| + beta |log beta|) to the allowed fraction (6e-3 at (3e11, 7e11); 1.0e-3 was measured
    there on a B200); at the distribution's own scale the effect is far below the binomial noise, which the moment
    tests below check."""
    got = ctx.test_betabinom_draws(alpha, beta, n, SAMPLER_DRAWS, seed=7)
    want = oracle.betabinom_draws(alpha, beta, n, SAMPLER_DRAWS, seed=7)
    diff = np.flatnonzero(got != want)
    detail = [(int(i), got[i], want[i]) for i in diff[:10]]
    if n <= 1_000_000:
        assert len(diff) == 0, ((alpha, beta, n), len(diff), detail)
    else:
        allowed = 1e-4 + 2.0**-52 * (alpha * abs(np.log(alpha)) + beta * abs(np.log(beta)))
        print(f"n = 2^32 - 1, ({alpha:g}, {beta:g}): {len(diff)} of {SAMPLER_DRAWS} draws differ (allowed {allowed:.1e})")
        assert len(diff) <= allowed * SAMPLER_DRAWS, ((alpha, beta, n), len(diff), detail)
    check_against_scipy(got, alpha, beta, n, (alpha, beta, n))


def test_device_sampler_limits(ctx):
    """alpha -> 0 puts all mass at 0, beta -> 0 all mass at n."""
    for n in (1000, 2**32 - 1):
        assert np.all(ctx.test_betabinom_draws(1e-300, 3.0, n, 4096, seed=3) == 0)
        assert np.all(ctx.test_betabinom_draws(3.0, 1e-300, n, 4096, seed=3) == n)


# ------------------------------------------------------------------ hpdi_prob validation
def test_hpdi_prob_outside_unit_interval_is_rejected(ctx):
    """hpdi_prob must satisfy 0 < hpdi_prob <= 1 (a negative value would index outside the sort buffer); the call
    returns MDG_ERR_INVALID before any launch, and the context stays usable: a following valid batch gives the same
    rows as a fresh context."""
    from metadamage_b200.backend import Context

    tid, k, N = predictive_batch(15, seed=700, n=6)
    for prob in (-0.1, 0.0, 1.5, float("nan")):
        with pytest.raises(_lib.MdgError, match="hpdi_prob") as err:
            ctx.fit_batch(tid, k, N, _lib.default_config(hpdi_prob=prob, **SHORT))
        assert err.value.code == -1, prob
    cfg = _lib.default_config(**SHORT)
    after = ctx.fit_batch(tid, k, N, cfg)
    with Context(0) as fresh:
        ref = fresh.fit_batch(tid, k, N, cfg)
    for key in ("result", "median", "hpdi_lo", "hpdi_hi"):
        assert after[key].tobytes() == ref[key].tobytes(), key
