"""The posterior-predictive replay (tests/ppc_replay.c) against the oracle's own predictive, and the predictive's
Beta -> Binomial sampler against scipy's beta-binomial at every seam of its algorithm.

The replay restates K6's item map (which run, dense position and Philox counter each predictive item draws from) on
the constrained draws a fit returns. Run on the oracle's fits, it must reproduce the oracle's median / HPDI / D_max
columns bit for bit; tests/test_gpu_predictive.py then holds the CUDA kernel to the same replay."""
import numpy as np
import pytest
from scipy import stats

import ppc_replay
from metadamage_b200 import synthetic as syn
from metadamage_b200._abi import FIT_FAILED

# (alpha, beta, n), one seam of the sampler per point
SAMPLER_GRID = [
    (0.3, 4.0, 12),            # a < 1: Marsaglia-Tsang with the U^(1/a) boost
    (0.002, 1.5, 300),         # a << 1: the boost in log space
    (1e-3, 50.0, 1000),        # a << 1, almost all mass at 0
    (0.999999, 3.0, 50),       # just below a = 1 (boost on)
    (1.0, 3.0, 50),            # a = 1 (boost off)
    (1.000001, 3.0, 50),       # just above a = 1
    (0.5, 0.5, 100),           # U-shaped Beta: p on both sides of the flip at p = 0.5
    (1000.0, 99000.0, 1000),   # n p = 10 within a few sd: BINV and BTRS
    (99000.0, 1000.0, 1000),   # the same, mirrored through the flip
    (5e5, 5e5, 10_000),        # p straddles 0.5 (the flip) in BTRS
    (3.0, 147.0, 600),         # a predictive draw at low damage
    (48000.0, 112000.0, 50_000),  # a predictive draw at high coverage and concentration
    (2.0, 30.0, 40),           # the earlier oracle test's points
    (150.0, 2000.0, 5000),
    (0.7, 2.0, 1),             # n = 1
    (2.0, 0.7, 2),             # n = 2
    (2.0, 5.0, 2**32 - 1),     # n at the uint32 limit: y / n ~ Beta(2, 5)
    (3e11, 7e11, 2**32 - 1),   # phi ~ 1e12: binomial noise dominates
]
SAMPLER_DRAWS = 200_000


def merged_bins(pmf, min_expected):
    """Edges [b0, b1), [b1, b2), ... of adjacent support points merged left to right until each holds min_expected;
    a short last bin joins the one before."""
    edges, acc = [0], 0.0
    for i, e in enumerate(pmf):
        acc += e
        if acc >= min_expected:
            edges.append(i + 1)
            acc = 0.0
    if edges[-1] != len(pmf):
        if len(edges) > 1:
            edges[-1] = len(pmf)
        else:
            edges.append(len(pmf))
    return np.array(edges)


def check_against_scipy(y, alpha, beta, n, tag):
    """y: draws of BetaBinomial(alpha, beta, n). n <= 1e5: chi-squared goodness of fit against scipy's pmf (bins
    merged to an expected count >= 20, p >= 1e-4) and the mean within 4 standard errors. n = 2^32 - 1: a KS test of
    y / n against Beta(alpha, beta) (p >= 1e-4) at small phi, z-tests (|z| < 4) of the mean and variance at large phi.
    The seeds are fixed, so each verdict is deterministic."""
    M = len(y)
    assert np.all(y == np.floor(y)) and y.min() >= 0 and y.max() <= n, tag
    dist = stats.betabinom(n, alpha, beta)
    mean, var = dist.mean(), dist.var()
    if n <= 100_000:
        assert abs(y.mean() - mean) < 4 * np.sqrt(var / M), (tag, y.mean(), mean)
        expected = dist.pmf(np.arange(n + 1)) * M
        edges = merged_bins(expected, 20.0)
        obs = np.add.reduceat(np.bincount(y.astype(np.int64), minlength=n + 1), edges[:-1])
        exp = np.add.reduceat(expected, edges[:-1])
        if len(exp) > 1:
            chi2 = ((obs - exp) ** 2 / exp).sum()
            p = stats.chi2.sf(chi2, len(exp) - 1)
            assert p >= 1e-4, (tag, chi2, len(exp), p)
    elif alpha + beta < 1e6:
        p = stats.kstest(y / n, stats.beta(alpha, beta).cdf).pvalue
        assert p >= 1e-4, (tag, p)
    else:
        z_mean = (y.mean() - mean) / np.sqrt(var / M)
        # sampling sd of the variance of M near-normal draws
        z_var = (y.var(ddof=1) - var) / (var * np.sqrt(2.0 / (M - 1)))
        assert abs(z_mean) < 4 and abs(z_var) < 4, (tag, z_mean, z_var)


@pytest.mark.parametrize("alpha,beta,n", SAMPLER_GRID)
def test_oracle_sampler_matches_scipy(oracle, alpha, beta, n):
    """The oracle's predictive sampler (the one the replay uses) against scipy's beta-binomial."""
    y = oracle.betabinom_draws(alpha, beta, n, SAMPLER_DRAWS, seed=7)
    check_against_scipy(y, alpha, beta, n, (alpha, beta, n))


def test_oracle_sampler_limits(oracle):
    """alpha -> 0 puts all mass at 0, beta -> 0 all mass at n."""
    for n in (1000, 2**32 - 1):
        assert np.all(oracle.betabinom_draws(1e-300, 3.0, n, 2000, seed=3) == 0)
        assert np.all(oracle.betabinom_draws(3.0, 1e-300, n, 2000, seed=3) == n)


# ------------------------------------------------------------------ the replay on the oracle's fits
@pytest.fixture(scope="module")
def replay():
    ppc_replay.build()
    return ppc_replay


def oracle_case(oracle, P, quirks, S, prob, fwd_rev=1):
    tid, k, N, _ = syn.dense_fit_batch(5, max_position=P, seed=60 + P)
    cut = np.arange(2 * P) % 3 == 0  # positions without coverage (dense 0 among them): NaN draws, NaN D_max and,
    cut[P] = False                    # with quirks only, NaN D_max_reverse
    N[1, cut] = 0
    k[1, cut] = 0
    N[2, P] = 0    # the reverse strand's first position: D_max_reverse NaN only without quirks
    k[2, P] = 0
    cfg = oracle.default_config(num_warmup=100, num_samples=S, reference_quirks=quirks, hpdi_prob=prob, do_fwd_rev=fwd_rev)
    out = oracle.fit_batch(tid, k, N, cfg, want_samples=True)
    assert (out["result"]["status"] & FIT_FAILED).sum() == 0  # the oracle leaves failed rows unassembled
    return tid, N, cfg, out


REPLAY_CASES = ([(P, q, 1, 257, 0.68) for P in (1, 15, 64) for q in (1, 0)] +
                [(15, 1, 0, 257, 0.68), (15, 1, 1, 64, 1.0), (15, 0, 1, 33, 0.5)])


@pytest.mark.parametrize("P,quirks,fwd_rev,S,prob", REPLAY_CASES)
def test_replay_matches_oracle_predictive(oracle, replay, P, quirks, fwd_rev, S, prob):
    """Median, HPDI ends and the five D_max columns of the oracle's fits equal the replay of its own draws, bit for
    bit: the item map (run, dense position, N, Philox counter), the Dz formula and the order statistics agree."""
    tid, N, cfg, out = oracle_case(oracle, P, quirks, S, prob, fwd_rev)
    want = replay.predictive(tid, N, out["samples"], out["result"]["status"], cfg)
    assert not replay.mismatches(out, want), (P, quirks, fwd_rev, S, prob, replay.mismatches(out, want))
    # the cases reach what they are meant to
    assert np.isnan(want["D_max"][1]) and np.isfinite(want["D_max"][0])
    if fwd_rev:
        assert np.isnan(want["D_max_reverse"][1]) == bool(quirks) and np.isnan(want["D_max_reverse"][2]) == (not quirks)
    else:
        assert np.all(np.isnan(want["D_max_forward"])) and np.all(np.isnan(want["D_max_reverse"]))
    assert np.array_equal(np.isnan(want["median"]), N == 0)


def test_replay_fails_loudly_on_draws_the_samplers_cannot_take(oracle, replay):
    """A PMD draw with q = 1 (Dz = NaN at x = 0) or an infinite phi in a fit not marked failed raises instead of
    hanging in the gamma sampler; the same draws in a failed fit are skipped."""
    tid, N, cfg, out = oracle_case(oracle, 15, 1, 257, 0.68)
    status = out["result"]["status"].copy()
    for col, value in ((0, 1.0), (0, 0.0), (3, np.inf), (3, np.nan)):
        smp = out["samples"].copy()
        smp[3, 0, 17, col] = value
        with pytest.raises(ValueError, match=r"\(row 3\), item 0, draw 17"):
            replay.draws(tid, N, smp, status, cfg)
        failed = status.copy()
        failed[3] |= FIT_FAILED
        y = replay.draws(tid, N, smp, failed, cfg)
        assert not y[3].any()
