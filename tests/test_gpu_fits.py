"""-m gpu: the CUDA fit kernels (K2-K7), called through the C-ABI, vs the oracle.

Tolerances (BASELINE.json north_star): log-density / gradient to FP64 round-off; MAP A, q, c,
phi, D_max within 1e-5 relative; MCMC summaries within 3x Monte-Carlo standard error; the NUTS
state machine additionally has to reproduce the oracle's chain transition by transition for the
first transitions (both draw from the same Philox streams)."""
import os

import numpy as np
import pytest

from conftest import (asymmetry_by_quadrature, mcse_batch_means, n_sigma_by_quadrature, null_posterior_quadrature, pmd_posterior_quadrature,
                      pmd_predictive_quadrature)
from metadamage_b200 import _lib, synthetic as syn
from test_oracle_nuts import (N_SIGMA_CASES, PMD_QUADRATURE_CASES, check_asymmetry_against_exact, check_fit_row_against_exact_posterior,
                              check_pmd_chain_against_quadrature, check_predictions_against_exact_pmf,
                              check_predictive_dmax_against_exact, synthetic_taxon)

pytestmark = pytest.mark.gpu


def test_philox_known_answers(ctx):
    key = np.array([[0, 0], [0xFFFFFFFF, 0xFFFFFFFF], [0xA4093822, 0x299F31D0]], np.uint32)
    ctr = np.array([[0, 0, 0, 0], [0xFFFFFFFF] * 4, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], np.uint32)
    out = ctx.philox(key, ctr)
    assert out.tolist() == [[0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8], [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD],
                            [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]]


def test_philox_matches_oracle_on_random_counters(ctx, oracle):
    rng = np.random.default_rng(0)
    key = rng.integers(0, 2 ** 32, (500, 2), dtype=np.uint64).astype(np.uint32)
    ctr = rng.integers(0, 2 ** 32, (500, 4), dtype=np.uint64).astype(np.uint32)
    out = ctx.philox(key, ctr)
    for i in range(0, 500, 25):
        assert list(out[i]) == list(oracle.philox(key[i], ctr[i]))


def test_special_functions(ctx):
    from scipy import special

    x = np.concatenate([10.0 ** np.linspace(-9, 9, 4000), np.linspace(0.01, 40, 4000), [9.999999, 10.0, 10.000001]])
    lg, dg = ctx.lgamma_digamma(x)
    ref_l, ref_d = special.gammaln(x), special.digamma(x)
    assert np.max(np.abs(lg - ref_l) / np.maximum(1, np.abs(ref_l))) < 5e-14
    assert np.max(np.abs(dg - ref_d) / np.maximum(1, np.abs(ref_d))) < 5e-14


def test_fast_exp_and_log(ctx):
    """The kernels' table-driven exp / log with immediate-encoded coefficients (csrc/mdg_common.cuh):
    a few ulp relative for exp, ~1e-15 absolute-ish for log (1/3 and 1/5 carry 21 significant bits)."""
    rng = np.random.default_rng(4)
    x = np.concatenate([rng.uniform(-700, 700, 20000), rng.uniform(-2, 2, 20000), [0.0, -0.0, 1e-300, -745.0, -800.0, 709.0, 710.0, np.inf, -np.inf]])
    ex, _ = ctx.exp_log(x)
    ref = np.exp(x)
    fin = np.isfinite(ref) & (ref > 1e-300)
    assert np.max(np.abs(ex[fin] - ref[fin]) / ref[fin]) < 4e-15
    assert ex[x == -np.inf][0] == 0.0 and np.isinf(ex[x == np.inf][0]) and ex[x == -800.0][0] == 0.0
    assert np.isnan(ctx.exp_log(np.array([np.nan]))[0][0])
    y = np.concatenate([10.0 ** rng.uniform(-300, 300, 20000), rng.uniform(0.5, 2.0, 20000), [1.0, 2.0, 0.5, 10.0]])
    _, lg = ctx.exp_log(y)
    ref = np.log(y)
    assert np.max(np.abs(lg - ref) / np.maximum(1.0, np.abs(ref))) < 2e-15
    assert abs(lg[y == 1.0][0]) < 2e-15


@pytest.mark.parametrize("P", [15, 25, 40])
@pytest.mark.parametrize("model", [0, 1])
def test_logp_grad_match_oracle(ctx, oracle, P, model):
    rng = np.random.default_rng(P + model)
    g = syn.make_mismatch_matrix(200, max_position=P, seed=77 + P)
    pick = np.argsort(-g["tax_n_alignments"])[:3]
    u = rng.uniform(-2, 2, (48, 4))
    u[:, 2] -= 2
    u[:, 3] += rng.uniform(0, 6, 48)
    for t in pick:
        for mask in (0, 1, 2):
            for jac in (True, False):
                a = ctx.logp_grad(g["k"][t], g["N"][t], u, model=model, lane_mask=mask, with_jacobian=jac)
                b = oracle.logp_grad(g["k"][t], g["N"][t], u, model=model, lane_mask=mask, with_jacobian=jac)
                assert np.array_equal(np.isnan(a[0]), np.isnan(b[0]))
                ok = np.isfinite(b[0])
                scale = 1e-13 * (1 + np.abs(b[0][ok]).max() + g["N"][t].max() * 20.0)
                assert np.max(np.abs(a[0][ok] - b[0][ok])) < scale
                assert np.max(np.abs(a[1][ok] - b[1][ok]) / (1 + np.abs(b[1][ok]))) < 1e-9
                assert np.max(np.abs(a[2][ok] - b[2][ok])) < scale


def test_logp_grad_high_coverage_sample(ctx, oracle, sample_inputs):
    """N(z) ~ 1e7 (the reference's sample file): lgamma terms of 1e8 must still agree to ~1e-7."""
    s = sample_inputs["ancient"]
    r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
    lgt = lambda p: np.log(p / (1 - p))  # noqa: E731
    u = np.array([[lgt(0.3), lgt(0.4), lgt(0.02), np.log(998.0)]])
    a = ctx.logp_grad(r["k"][0], r["N"][0], u, with_jacobian=False)
    assert abs(a[2].sum() - (-825.2253953129)) < 2e-6  # SURVEY.md 8c known answer
    b = oracle.logp_grad(r["k"][0], r["N"][0], u, with_jacobian=False)
    assert np.max(np.abs(a[1] - b[1]) / (1 + np.abs(b[1]))) < 1e-9


def small_batch(n, P=15, seed=5):
    tid, k, N, g = syn.dense_fit_batch(n, max_position=P, seed=seed)
    return tid, k, N


def test_map_matches_oracle(ctx, oracle, sample_inputs):
    tid, k, N = small_batch(96)
    # add the six high-coverage sample TaxIDs
    for name in ("ancient", "control"):
        s = sample_inputs[name]
        r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
        tid = np.r_[tid, r["tax_id"] + 10 ** 6]
        k = np.vstack([k, r["k"]])
        N = np.vstack([N, r["N"]])
    cfg = _lib.default_config(num_warmup=4, num_samples=4, do_fwd_rev=0)
    got = ctx.fit_batch(tid, k, N, cfg)["result"]
    exp = oracle.fit_batch(tid, k, N, oracle.default_config(num_warmup=4, num_samples=4, do_fwd_rev=0))["result"]
    conv = ((got["status"] | exp["status"]) & 2) == 0
    assert conv.mean() > 0.95
    for f in ("map_A", "map_q", "map_c", "map_phi", "map_D_max", "map_null_q", "map_null_phi"):
        rel = np.abs(got[f][conv] - exp[f][conv]) / np.maximum(np.abs(exp[f][conv]), 1e-300)
        # parameters that sit on the boundary (c -> 0) are compared absolutely
        bad = (rel > 1e-5) & (np.abs(got[f][conv] - exp[f][conv]) > 1e-9)
        assert not bad.any(), (f, rel.max())
    assert np.max(np.abs(got["map_logp"][conv] - exp["map_logp"][conv])) < 1e-6


def test_nuts_traces_follow_the_oracle(ctx, oracle):
    """Same Philox streams + same algorithm: chains must coincide until FP round-off amplifies."""
    tid, k, N = small_batch(6, seed=9)
    cfg = dict(num_warmup=150, num_samples=50)
    got = ctx.fit_batch(tid, k, N, _lib.default_config(**cfg), want_trace=True)
    exp = oracle.fit_batch(tid, k, N, oracle.default_config(**cfg), want_trace=True)
    agree = []
    for i in range(len(tid)):
        for run in range(6):
            a, b = got["trace"][i, run], exp["trace"][i, run]
            d = np.nanmax(np.abs(a - b), axis=1)
            assert d[0] < 1e-9, (i, run, d[:3])
            bad = np.flatnonzero(d > 1e-6)
            agree.append(int(bad[0]) if len(bad) else len(d))
    assert min(agree) >= 3 and np.median(agree) >= 15, agree


def test_nuts_summaries_within_mcse_of_oracle(ctx, oracle):
    """3 x MCSE gate on posterior D_max (= A + c) mean and std, q_mean, concentration_mean."""
    taxa = [synthetic_taxon(40 + i, A=a, c=c) for i, (a, c) in enumerate([(0.25, 0.02), (0.05, 0.01), (0.4, 0.03), (0.002, 0.01)])]
    tid = np.arange(4, dtype=np.int64) + 900
    k = np.stack([t[0] for t in taxa])
    N = np.stack([t[1] for t in taxa])
    kw = dict(num_warmup=500, num_samples=3000, do_map=0)
    got = ctx.fit_batch(tid, k, N, _lib.default_config(**kw), want_samples=True)
    exp = oracle.fit_batch(tid, k, N, oracle.default_config(**kw), want_samples=True)
    for i in range(4):
        sa, sb = got["samples"][i, 0], exp["samples"][i, 0]
        for name, fa, fb in (("D_max", sa[:, 1] + sa[:, 2], sb[:, 1] + sb[:, 2]), ("q", sa[:, 0], sb[:, 0]),
                             ("log_delta", np.log(sa[:, 3] - 2), np.log(sb[:, 3] - 2))):
            se = np.hypot(mcse_batch_means(fa), mcse_batch_means(fb))
            assert abs(fa.mean() - fb.mean()) < 3 * se + 1e-12, (i, name, fa.mean(), fb.mean(), se)
            se_sd = np.hypot(mcse_batch_means((fa - fa.mean()) ** 2), mcse_batch_means((fb - fb.mean()) ** 2))
            assert abs(fa.var() - fb.var()) < 3.5 * se_sd + 1e-14, (i, name, "var")
        r, e = got["result"][i], exp["result"][i]
        assert abs(r["D_max_marginalized_mean"] - (sa[:, 1] + sa[:, 2]).mean()) < 1e-10
        assert abs(r["D_max_marginalized_std"] - (sa[:, 1] + sa[:, 2]).std()) < 1e-10
        assert abs(r["q_mean"] - sa[:, 0].mean()) < 1e-10 and abs(r["concentration_mean"] - sa[:, 3].mean()) < 1e-7
        # predictive D_max is quantised to 1/(2 N(z=1)); allow the MC error of a median
        sd_pred = np.sqrt(max(e["D_max"] * (1 - e["D_max"]), 1e-6) / N[i, 0]) + (sb[:, 1] + sb[:, 2]).std()
        assert abs(r["D_max"] - e["D_max"]) < 4 * 1.2533 * sd_pred / np.sqrt(3000) + 1.0 / N[i, 0]
        assert abs(r["D_max_lower_hpdi"] - e["D_max_lower_hpdi"]) < 0.25 * sd_pred + 2.0 / N[i, 0]
        assert abs(r["D_max_upper_hpdi"] - e["D_max_upper_hpdi"]) < 0.25 * sd_pred + 2.0 / N[i, 0]
        # n_sigma: both are noisy functions of 2 x 3000 draws; compare on the scale of the WAIC sums
        assert abs(r["run"][0]["waic"] - e["run"][0]["waic"]) < 1.5 and abs(r["run"][1]["waic"] - e["run"][1]["waic"]) < 1.5
        assert abs(r["n_sigma"] - e["n_sigma"]) < 0.35 * (1 + abs(e["n_sigma"]))


def test_null_model_chains_match_quadrature(ctx):
    """Ground truth without any sampler: the null model's 2-D posterior integrated on a grid with
    scipy's beta-binomial pmf (conftest.null_posterior_quadrature). The CUDA chains (null / all
    positions, and null / forward-only through the half-warp kernel) must agree within 4 x MCSE."""
    cases = [(21, dict(n_lo=200, n_hi=3000)), (22, dict(n_lo=5, n_hi=60, A=0.0, c=0.05)), (23, dict(n_lo=20000, n_hi=90000, phi=3000.0))]
    taxa = [synthetic_taxon(seed, **kw) for seed, kw in cases]
    tid = np.arange(len(taxa), dtype=np.int64) + 7021
    k = np.stack([t[0] for t in taxa])
    N = np.stack([t[1] for t in taxa])
    got = ctx.fit_batch(tid, k, N, _lib.default_config(num_warmup=500, num_samples=4000, do_map=0), want_samples=True)
    for i in range(len(taxa)):
        for run, sl in ((1, slice(0, 30)), (3, slice(0, 15))):  # null/all, null/forward
            truth = null_posterior_quadrature(k[i, sl], N[i, sl])
            smp = got["samples"][i, run]
            q, ld = smp[:, 0], np.log(smp[:, 3] - 2.0)
            assert abs(q.mean() - truth["mean_q"]) < 4 * mcse_batch_means(q) + 1e-12, (i, run, q.mean(), truth["mean_q"])
            assert abs(ld.mean() - truth["mean_logdelta"]) < 4 * mcse_batch_means(ld) + 1e-12, (i, run, ld.mean(), truth["mean_logdelta"])
            assert abs(q.var() - truth["var_q"]) < 5 * mcse_batch_means((q - q.mean()) ** 2) + 0.02 * truth["var_q"], (i, run, "var q")
            assert abs(ld.var() - truth["var_logdelta"]) < 5 * mcse_batch_means((ld - ld.mean()) ** 2) + 0.02 * truth["var_logdelta"], (i, run)


def test_pmd_model_chains_match_quadrature(ctx):
    """Ground truth without any sampler for the PMD model: its 4-D posterior integrated on tensor grids
    with scipy's beta-binomial (conftest.pmd_posterior_quadrature). The CUDA chains — all positions
    (full-warp kernel) and forward-only / reverse-only (the two halves of the half-warp kernel) — must
    agree within 4 x MCSE in the means and 5 x MCSE + 3 % in the variances of q, A, c, log(delta) and
    D_max = A + c."""
    taxa = [synthetic_taxon(seed, **kw) for seed, kw in PMD_QUADRATURE_CASES]
    tid = np.arange(len(taxa), dtype=np.int64) + 7131
    k = np.stack([t[0] for t in taxa])
    N = np.stack([t[1] for t in taxa])
    got = ctx.fit_batch(tid, k, N, _lib.default_config(num_warmup=500, num_samples=4000, do_map=0), want_samples=True)
    for i, runs in ((0, ((0, slice(0, 30)), (2, slice(0, 15)))), (1, ((0, slice(0, 30)), (4, slice(15, 30))))):
        for run, sl in runs:
            truth = pmd_posterior_quadrature(k[i, sl], N[i, sl])
            check_pmd_chain_against_quadrature(got["samples"][i, run], truth, (i, run))


def test_n_sigma_and_dmax_match_exact_posterior(ctx):
    """The path's headline outputs from the CUDA kernels (NUTS + fused WAIC accumulation + assembly) against
    the exact posterior: n_sigma, the PMD and null WAIC, D_max mean and std, and the predictive kernel's D_max
    (median of y_rep / N at z = 1) with its 68 % HPDI against the exact predictive pmf — quadrature, no sampler."""
    taxa = [synthetic_taxon(seed, **kw) for seed, kw in N_SIGMA_CASES]
    tid = np.arange(len(taxa), dtype=np.int64) + 7161
    k = np.stack([t[0] for t in taxa])
    N = np.stack([t[1] for t in taxa])
    got = ctx.fit_batch(tid, k, N, _lib.default_config(num_warmup=500, num_samples=4000, do_map=0, do_fwd_rev=0))
    for i in range(len(taxa)):
        check_fit_row_against_exact_posterior(got["result"][i], n_sigma_by_quadrature(k[i], N[i]), i)
        check_predictive_dmax_against_exact(got["result"][i], pmd_predictive_quadrature(k[i], N[i]), 4000, i)


def test_max_position_25_matches_exact_posterior(ctx):
    """BASELINE config 4's geometry (--max-position 25: 50 positions, two per lane in the full-warp kernel)
    against the exact posterior: n_sigma, both WAICs, D_max mean and std by quadrature."""
    P, A, q, c, phi = 25, 0.2, 0.3, 0.02, 150.0
    rng = np.random.default_rng(41)
    N = rng.integers(50, 600, 2 * P).astype(np.uint32)
    z = np.r_[np.arange(P), np.arange(P)]
    Dz = A * (1 - q) ** z + c
    k = rng.binomial(N, rng.beta(Dz * phi, (1 - Dz) * phi)).astype(np.uint32)
    cfg = _lib.default_config(num_warmup=500, num_samples=4000, do_map=0, do_fwd_rev=0)
    got = ctx.fit_batch(np.array([7241], np.int64), k[None], N[None], cfg)
    check_fit_row_against_exact_posterior(got["result"][0], n_sigma_by_quadrature(k, N), "P25")


def test_fit_predictions_match_exact_predictive(ctx):
    """The predictive kernel's per-position median and 68 % HPDI (df_fit_predictions, fits.py:632-665) against
    the exact posterior-predictive pmf at forward and reverse positions near and far from the read end."""
    seed, kw = N_SIGMA_CASES[1]
    k, N = synthetic_taxon(seed, **kw)
    cfg = _lib.default_config(num_warmup=500, num_samples=4000, do_map=0, do_fwd_rev=0)
    out = ctx.fit_batch(np.array([7192], np.int64), k[None], N[None], cfg)
    check_predictions_against_exact_pmf(out, k, N, 4000)


def test_forward_reverse_refits_match_exact_posterior(ctx):
    """The half-warp kernels' WAIC accumulation and the assembly of n_sigma_forward / n_sigma_reverse /
    asymmetry (fits.py:298-356) against their exact values by quadrature."""
    seed, kw = N_SIGMA_CASES[1]
    k, N = synthetic_taxon(seed, **kw)
    got = ctx.fit_batch(np.array([7191], np.int64), k[None], N[None], _lib.default_config(num_warmup=500, num_samples=4000, do_map=0))
    check_asymmetry_against_exact(got["result"][0], asymmetry_by_quadrature(k, N), seed)


def test_waic_and_assembly_are_consistent(ctx):
    """The row assembled on the device equals a host recomputation from the device's own
    per-position WAIC blocks and draws (fits.py:147-227)."""
    tid, k, N = small_batch(12, seed=21)
    out = ctx.fit_batch(tid, k, N, _lib.default_config(num_warmup=200, num_samples=500), want_samples=True, want_waic=True)
    for i in range(len(tid)):
        r, w = out["result"][i], out["waic"][i]
        wi = lambda run: -2 * (w[run, 0] - w[run, 1])  # noqa: E731
        d = wi(0) - wi(1)
        assert abs(r["n_sigma"] - (wi(1).sum() - wi(0).sum()) / np.sqrt(30 * d.var())) < 1e-8 * (1 + abs(r["n_sigma"]))
        df = (wi(2) - wi(3))[:15]
        assert abs(r["n_sigma_forward"] - (wi(3)[:15].sum() - wi(2)[:15].sum()) / np.sqrt(15 * df.var())) < 1e-8 * (1 + abs(r["n_sigma_forward"]))
        cat = np.r_[wi(2)[:15], wi(4)[15:]]
        dd = wi(0) - cat
        assert abs(r["asymmetry"] - (cat.sum() - wi(0).sum()) / np.sqrt(30 * dd.var())) < 1e-8 * (1 + abs(r["asymmetry"]))
        assert abs(r["run"][0]["waic"] - wi(0).sum()) < 1e-8
        assert r["N_sum_total"] == N[i].sum() and r["y_sum_total"] == k[i].sum()
        assert abs(r["q_mean_forward"] - out["samples"][i, 2][:, 0].mean()) < 1e-10
        assert abs(r["q_mean_reverse"] - out["samples"][i, 4][:, 0].mean()) < 1e-10
        assert np.isnan(out["samples"][i, 1][:, 1]).all()  # null runs have no A, c
        m, lo, hi = out["median"][i], out["hpdi_lo"][i], out["hpdi_hi"][i]
        assert np.all(lo <= m + 1e-7) and np.all(m <= hi + 1e-7)
        assert abs(m[0] - r["D_max"]) < 1e-6


def test_noise_paths_agree(ctx, oracle, fits_golden):
    """mism12 -> noise on the device equals the reference's add_noise_estimates (fits.py:359-376)."""
    m12 = fits_golden["noise_mism12"].astype(np.uint32)
    n = len(m12)
    rng = np.random.default_rng(0)
    N = rng.integers(50, 500, (n, 30)).astype(np.uint32)
    k = rng.binomial(N, 0.05).astype(np.uint32)
    out = ctx.fit_batch(np.arange(n), k, N, _lib.default_config(num_warmup=5, num_samples=5, do_fwd_rev=0, do_map=0), mism12=m12)
    got = np.stack([out["result"][f] for f in ("normalized_noise", "normalized_noise_forward", "normalized_noise_reverse")], 1)
    np.testing.assert_allclose(got, fits_golden["noise_expected"], rtol=1e-12)


def test_partition_and_order_invariance_bitwise(ctx):
    """Philox streams keyed by (seed, tax_id): any split / order of the batch is bit-identical."""
    tid, k, N = small_batch(40, seed=33)
    cfg = _lib.default_config(num_warmup=80, num_samples=120)
    full = ctx.fit_batch(tid, k, N, cfg)
    a = ctx.fit_batch(tid[:13], k[:13], N[:13], cfg)
    b = ctx.fit_batch(tid[13:], k[13:], N[13:], cfg)
    assert full["result"].tobytes() == np.concatenate([a["result"], b["result"]]).tobytes()
    assert full["median"].tobytes() == np.concatenate([a["median"], b["median"]]).tobytes()
    perm = np.random.default_rng(1).permutation(40)
    p = ctx.fit_batch(tid[perm], k[perm], N[perm], cfg)
    assert full["result"][perm].tobytes() == p["result"].tobytes()
    again = ctx.fit_batch(tid, k, N, cfg)
    assert full["result"].tobytes() == again["result"].tobytes()  # which group / warp / CTA picked a chain up changes nothing
    other = ctx.fit_batch(tid, k, N, cfg.copy(seed=7))
    assert other["result"]["q_mean"].tobytes() != full["result"]["q_mean"].tobytes()
    # the library's internal chunking (scratch reuse between chunks) changes nothing either
    os.environ["MDG_FIT_CHUNK"] = "7"
    try:
        chunked = ctx.fit_batch(tid, k, N, cfg)
    finally:
        del os.environ["MDG_FIT_CHUNK"]
    assert full["result"].tobytes() == chunked["result"].tobytes()
    assert full["median"].tobytes() == chunked["median"].tobytes()


def test_schedule_variants_are_bit_identical(ctx):
    """How the chains are scheduled — the coverage order of the queue, which forward / reverse runs go first, the
    chunk size — must not change a single bit of the rows: every chain is a function of (seed, tax_id, run, data)
    only."""
    g = syn.make_mismatch_matrix(0, seed=77, n_fit=300)
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], want_noise=True)
    cfg = _lib.default_config(num_warmup=60, num_samples=80)
    base = ctx.fit_batch(r["tax_id"], r["k"], r["N"], cfg, noise3=r["noise"], want_waic=True)
    # (the coverage order is the default from 32 768 TaxIDs per chunk on; MDG_NUTS_ORDER=2 forces it for this small batch)
    variants = [{"MDG_NUTS_ORDER": "2"}, {"MDG_NUTS_ORDER": "2", "MDG_NUTS_PRIO_FRAC": "1"}, {"MDG_NUTS_ORDER": "2", "MDG_NUTS_PRIO_FRAC": "0"},
                {"MDG_NUTS_ORDER": "2", "MDG_FIT_CHUNK": "64"}, {"MDG_FIT_CHUNK": "64"}]
    for env in variants:
        os.environ.update(env)
        try:
            got = ctx.fit_batch(r["tax_id"], r["k"], r["N"], cfg, noise3=r["noise"], want_waic=True)
        finally:
            for key in env:
                del os.environ[key]
        assert got["result"].tobytes() == base["result"].tobytes(), env
        assert got["median"].tobytes() == base["median"].tobytes(), env
        assert got["waic"].tobytes() == base["waic"].tobytes(), env


@pytest.mark.parametrize("P", [25, 40])
def test_other_max_positions(ctx, oracle, P):
    """BASELINE config 4: --max-position 25 with swapped substitutions: damage lives in CT/GA, so
    looking at GA/CT must find no signal."""
    g = syn.make_mismatch_matrix(0, max_position=P, seed=syn.SEEDS["cfg4"], n_fit=24, fwd="GA", rev="CT")
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], fwd="GA", rev="CT", max_position=P)
    kw = dict(num_warmup=200, num_samples=300)
    got = ctx.fit_batch(r["tax_id"], r["k"], r["N"], _lib.default_config(**kw))
    res = got["result"]
    assert (res["status"] & 1).sum() == 0
    assert np.median(res["n_sigma"]) < 2.0
    exp = oracle.fit_batch(r["tax_id"][:4], r["k"][:4], r["N"][:4], oracle.default_config(**kw))["result"]
    for f in ("map_A", "map_q", "map_c", "map_phi"):
        ok = ((res["status"][:4] | exp["status"]) & 2) == 0
        assert np.all((np.abs(res[f][:4] - exp[f])[ok] < 1e-5 * np.abs(exp[f])[ok]) | (np.abs(res[f][:4] - exp[f])[ok] < 1e-9))
    assert got["median"].shape == (24, 2 * P)


def test_degenerate_inputs(ctx):
    """All-zero coverage, k = 0 everywhere, k = N everywhere: no hang, finite status handling."""
    N = np.zeros((4, 30), np.uint32)
    k = np.zeros((4, 30), np.uint32)
    N[1] = 100
    N[2] = 100
    k[2] = 100
    N[3, :15] = 50
    k[3, :15] = 5
    out = ctx.fit_batch(np.arange(4), k, N, _lib.default_config(num_warmup=100, num_samples=100))["result"]
    assert np.isnan(out["D_max"][0])  # 0 / 0 like the reference
    assert (out["status"] & 1).sum() == 0
    assert out["D_max"][1] < 0.05 and out["D_max"][2] > 0.9


def test_device_resident_path_matches_host_path(ctx):
    import torch

    tid, k, N = small_batch(32, seed=44)
    cfg = _lib.default_config(num_warmup=60, num_samples=64)
    host = ctx.fit_batch(tid, k, N, cfg)
    dev = torch.device("cuda", 0)
    from metadamage_b200._abi import FIT_RESULT_DTYPE

    out = torch.zeros(len(tid) * FIT_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    med = torch.zeros((len(tid), 30), dtype=torch.float32, device=dev)
    ctx.fit_batch_device(torch.from_numpy(tid).to(dev), torch.from_numpy(k.view(np.int32)).to(dev),
                         torch.from_numpy(N.view(np.int32)).to(dev), out, cfg, median=med)
    ctx.synchronize()
    res = out.cpu().numpy().view(FIT_RESULT_DTYPE)
    assert res.tobytes() == host["result"].tobytes()
    assert med.cpu().numpy().tobytes() == host["median"].tobytes()


def test_leapfrog_budget_is_the_timeout_analogue(ctx, oracle):
    """mdg_fit_config.max_leapfrogs_per_run bounds the work of one NUTS run the way the reference's per-fit
    timeout does (fits.py:37-38, 472-474, 520-521): a TaxID with a run over budget comes back with
    MDG_FIT_FAILED | MDG_FIT_BUDGET_EXCEEDED (the host drops it with a warning); every other TaxID is
    bit-identical to the unlimited fit; the oracle flags the same TaxIDs."""
    from metadamage_b200._abi import FIT_BUDGET_EXCEEDED, FIT_FAILED

    tid, k, N = small_batch(48, seed=71)
    kw = dict(num_warmup=120, num_samples=100)
    free = ctx.fit_batch(tid, k, N, _lib.default_config(**kw))["result"]
    longest = free["run"]["n_leapfrog"].max(axis=1)
    budget = int(np.median(longest))
    lim = ctx.fit_batch(tid, k, N, _lib.default_config(max_leapfrogs_per_run=budget, **kw))["result"]
    over = longest > budget
    assert 0 < over.sum() < len(tid)
    assert np.all((lim["status"][over] & (FIT_FAILED | FIT_BUDGET_EXCEEDED)) == (FIT_FAILED | FIT_BUDGET_EXCEEDED))
    assert np.all((lim["status"][~over] & FIT_BUDGET_EXCEEDED) == 0)
    assert lim[~over].tobytes() == free[~over].tobytes()
    assert np.all(np.isnan(lim["D_max"][over])) and np.all(np.isnan(lim["n_sigma"][over]))
    # no run of a flagged TaxID went past the budget by more than the trip that noticed it
    assert lim["run"]["n_leapfrog"].max() <= budget + 1
    # the oracle applies the same rule to its own chains (they coincide with the kernel's only until round-off
    # amplifies, so run lengths differ between the two; each side is checked against its own unlimited run)
    exp_free = oracle.fit_batch(tid, k, N, oracle.default_config(**kw))["result"]
    exp = oracle.fit_batch(tid, k, N, oracle.default_config(max_leapfrogs_per_run=budget, **kw))["result"]
    over_o = exp_free["run"]["n_leapfrog"].max(axis=1) > budget
    assert np.array_equal((exp["status"] & FIT_BUDGET_EXCEEDED) != 0, over_o)
    assert np.array_equal((exp["status"] & FIT_FAILED) != 0, over_o)
    assert exp[~over_o].tobytes() == exp_free[~over_o].tobytes()
    assert abs(int(over_o.sum()) - int(over.sum())) <= 8
