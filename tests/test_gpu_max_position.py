"""-m gpu: the fit and counts kernels at every max_position where a lane layout changes (test_model_reference's
MAX_POSITIONS, 1 to 64), against the 40-digit model reference, the oracle and the device's own draws.

Each kernel lays the 2P positions (P for a forward-only or reverse-only run) out over lanes in its own way: MAP's
eval_model with NPL positions per lane and a spare slot, NUTS's eval_group over 8 lanes per chain with index 0 the
spare, the fused WAIC accumulators in [4][NS][32] per warp. A NUTS gradient that is wrong still samples a valid
posterior, so the statistical gates cannot see it: these tests compare value by value."""
import functools

import numpy as np
import pytest
from scipy import special, stats

from metadamage_b200 import _lib, synthetic as syn
from metadamage_b200._abi import FIT_FAILED
from test_gpu_counts import assert_same
from test_model_reference import (MAX_POSITIONS, boundary_taxon, check_logp_grad_against_reference, model_ll_mp,
                                  reference_points, used_positions)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def map_oracle(oracle):
    from oracle import map_oracle as M

    M.build()
    return M


def batch(n, P, seed):
    tid, k, N, _ = syn.dense_fit_batch(n, max_position=P, seed=seed)
    return tid, k, N


# ------------------------------------------------------------------ MAP's evaluator (eval_model) through the test hook
@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_eval_model_matches_reference_and_oracle(ctx, oracle, P):
    """logp, gradient and per-position ll of eval_model (the layout of map_kernel: NPL = 1, 2 or 4 positions per
    lane, no spare slot at P = 16, 32, 64) against the 40-digit reference on a few points per case, and against the
    oracle on 48 random points per case with the tolerances of test_logp_grad_match_oracle."""
    k, N = boundary_taxon(P)
    for model in (0, 1):
        u_ref = reference_points(model, seed=P)[::2]  # bulk and edge points; mpmath is slow at P = 64
        for mask in (0, 1, 2):
            for jac in (True, False):
                tag = (P, model, mask, jac)
                logp, grad, ll = ctx.logp_grad(k, N, u_ref, model=model, lane_mask=mask, with_jacobian=jac)
                check_logp_grad_against_reference(k, N, u_ref, model, mask, jac, logp, grad, tag)
                if jac:
                    continue  # ll does not depend on the Jacobian
                used = list(used_positions(P, mask))
                for e in range(len(u_ref)):
                    ref = model_ll_mp(k, N, u_ref[e], model, mask)
                    if ref is None:
                        continue
                    for i in used:
                        v, scale = ref[i]
                        assert abs(ll[e, i] - v) <= 1e-13 * (1 + scale), (tag, e, i, ll[e, i], v)
                    assert np.all(np.delete(ll[e], used) == 0.0), (tag, e)
    rng = np.random.default_rng(P)
    g = syn.make_mismatch_matrix(200, max_position=P, seed=77 + P)
    u = rng.uniform(-2, 2, (48, 4))
    u[:, 2] -= 2
    u[:, 3] += rng.uniform(0, 6, 48)
    for t in np.argsort(-g["tax_n_alignments"])[:3]:  # the tolerance's 20 N_max term is sized for high coverage
        for model in (0, 1):
            for mask in (0, 1, 2):
                for jac in (True, False):
                    a = ctx.logp_grad(g["k"][t], g["N"][t], u, model=model, lane_mask=mask, with_jacobian=jac)
                    b = oracle.logp_grad(g["k"][t], g["N"][t], u, model=model, lane_mask=mask, with_jacobian=jac)
                    assert np.array_equal(np.isnan(a[0]), np.isnan(b[0]))
                    ok = np.isfinite(b[0])
                    scale = 1e-13 * (1 + np.abs(b[0][ok]).max() + g["N"][t].max() * 20.0)
                    assert np.max(np.abs(a[0][ok] - b[0][ok])) < scale, (P, model, mask, jac)
                    assert np.max(np.abs(a[1][ok] - b[1][ok]) / (1 + np.abs(b[1][ok]))) < 1e-9, (P, model, mask, jac)
                    assert np.max(np.abs(a[2][ok] - b[2][ok])) < scale, (P, model, mask, jac)


# ------------------------------------------------------------------ NUTS's evaluator (eval_group) through the traces
TRACE_CASES = [(P, 0) for P in MAX_POSITIONS] + [(P, 1) for P in (1, 16, 64)]


@pytest.mark.parametrize("P,heuristic", TRACE_CASES)
def test_nuts_traces_follow_the_oracle(ctx, oracle, P, heuristic):
    """Same Philox streams and the same algorithm as the oracle: all six runs of 5 TaxIDs coincide with the
    oracle's chains until round-off amplifies (test_gpu_fits.test_nuts_traces_follow_the_oracle, at every layout)."""
    tid, k, N = batch(5, P, seed=9 + P)
    cfg = dict(num_warmup=150, num_samples=50, find_heuristic_step_size=heuristic)
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


# ------------------------------------------------------------------ fused WAIC blocks and the assembly
@functools.lru_cache(maxsize=None)
def fit_with_waic(ctx, P):
    """A small fit with draws and WAIC blocks; two TaxIDs lose coverage at some positions (N = 0 there)."""
    tid, k, N = batch(5, P, seed=31 + P)
    N[1, ::3] = 0
    k[1, ::3] = 0
    N[3, P - 1] = 0
    k[3, P - 1] = 0
    out = ctx.fit_batch(tid, k, N, _lib.default_config(num_warmup=120, num_samples=100), want_samples=True, want_waic=True)
    return tid, k, N, out


def waic_from_draws(k, N, smp, model, positions):
    """lppd_i = logsumexp(ll) - log S and pWAIC_i = var(ll) (ddof = 0) per position, in FP64 with scipy, from the
    run's S constrained draws (q, A, c, phi)."""
    q, A, c, phi = smp[:, 0], smp[:, 1], smp[:, 2], smp[:, 3]
    P = len(k) // 2
    out = {}
    for i in positions:
        x = i if i < P else i - P
        Dz = A * (1 - q) ** x + c if model == 0 else q
        ll = stats.betabinom.logpmf(k[i], N[i], Dz * phi, (1 - Dz) * phi)
        out[i] = (special.logsumexp(ll) - np.log(len(ll)), ll.var())
    return out


@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_fused_waic_blocks_match_the_draws(ctx, P):
    """Every per-position WAIC term the NUTS kernel accumulates on the fly, recomputed from the same run's draws.
    The kernel evaluates the log-likelihood at the unconstrained state u; the draws are the constrained theta (q, A,
    c, phi) rounded once, and the log-likelihood's sensitivity to its parameters grows with N_i, so the tolerance is
    1e-10 x (1 + N_i) absolute. Positions a run does not use stay exactly 0; the run's waic and lppd are the sums of
    its blocks."""
    tid, k, N, out = fit_with_waic(ctx, P)
    res, waic, smp = out["result"], out["waic"], out["samples"]
    assert (res["status"] & FIT_FAILED).sum() == 0
    for i in range(len(tid)):
        for run in range(6):
            used = list(used_positions(P, run // 2))
            w = waic[i, run]
            ref = waic_from_draws(k[i], N[i], smp[i, run], run % 2, used)
            for j in used:
                lppd, pw = ref[j]
                tol = 1e-10 * (1 + float(N[i, j]))
                assert abs(w[0, j] - lppd) <= tol, (P, i, run, j, w[0, j], lppd)
                assert abs(w[1, j] - pw) <= tol, (P, i, run, j, w[1, j], pw)
            assert np.all(np.delete(w, used, axis=1) == 0.0), (P, i, run)
            blocks_waic = (-2.0 * (w[0, used] - w[1, used])).sum()
            blocks_lppd = w[0, used].sum()
            r = res["run"][i, run]
            assert abs(r["waic"] - blocks_waic) <= 1e-9 * abs(blocks_waic), (P, i, run, r["waic"], blocks_waic)
            assert abs(r["lppd"] - blocks_lppd) <= 1e-9 * abs(blocks_lppd), (P, i, run, r["lppd"], blocks_lppd)


def asymmetry_rule(wi_all, wi_fwd, wi_rev, P):
    """fits.py:204-227: the forward-only and reverse-only PMD refits against the all-position PMD fit"""
    cat = np.r_[wi_fwd[:P], wi_rev[P:]]
    dd = wi_all - cat
    return (cat.sum() - wi_all.sum()) / np.sqrt(2 * P * dd.var())


@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_assembly_from_the_waic_blocks(ctx, oracle, P):
    """n_sigma, n_sigma_forward, n_sigma_reverse (the oracle's rule on the device's blocks) and the asymmetry. At
    P = 1 a half run has one position, so the variance under n_sigma_forward / _reverse is 0 and they are +-inf with
    the sign of the WAIC difference."""
    tid, k, N, out = fit_with_waic(ctx, P)
    res, waic = out["result"], out["waic"]
    for i in range(len(tid)):
        w = waic[i]
        wi = lambda run: -2 * (w[run, 0] - w[run, 1])  # noqa: E731
        r = res[i]
        assert r["status"] & FIT_FAILED == 0
        cases = (("n_sigma", wi(0), wi(1)), ("n_sigma_forward", wi(2)[:P], wi(3)[:P]), ("n_sigma_reverse", wi(4)[P:], wi(5)[P:]))
        for name, pmd, null in cases:
            want = oracle.n_sigma(pmd, null)
            if np.isinf(want) or np.isnan(want):
                assert r[name] == want or (np.isnan(want) and np.isnan(r[name])), (P, i, name, r[name], want)
            else:
                assert abs(r[name] - want) <= 1e-8 * (1 + abs(want)), (P, i, name, r[name], want)
        if P == 1:
            for name, pmd, null in cases[1:]:
                if null.sum() != pmd.sum():  # equal only where the strand has no coverage (every term is 0): 0 / 0
                    assert np.isinf(r[name]) and np.sign(r[name]) == np.sign(null.sum() - pmd.sum()), (i, name, r[name])
        want = asymmetry_rule(wi(0), wi(2), wi(4), P)
        assert abs(r["asymmetry"] - want) <= 1e-8 * (1 + abs(want)), (P, i, r["asymmetry"], want)
        m, lo, hi = out["median"], out["hpdi_lo"], out["hpdi_hi"]
        for a in (m, lo, hi):
            assert a.shape == (len(tid), 2 * P)
            assert np.array_equal(np.isnan(a), N == 0), P


# ------------------------------------------------------------------ MAP: fit_batch's map_* fields and map_batch
def close(a, b, rtol, atol=0.0):
    return np.abs(a - b) <= rtol * np.abs(b) + atol


@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_map_fits_match_oracle(ctx, oracle, map_oracle, P):
    """fit_batch's map_* fields and map_batch (do_fwd_rev 0 and 1) against the oracle and map_oracle with the
    tolerances of test_map_matches_oracle / test_map_batch_matches_oracle; map_batch's all-position runs are
    bit-identical to fit_batch's map_* (both run map_fit_group in the same layout)."""
    tid, k, N = batch(48, P, seed=5 + P)
    kw = dict(num_warmup=4, num_samples=4, do_fwd_rev=0)
    fit = ctx.fit_batch(tid, k, N, _lib.default_config(**kw))["result"]
    exp = oracle.fit_batch(tid, k, N, oracle.default_config(**kw))["result"]
    conv = ((fit["status"] | exp["status"]) & 2) == 0
    assert conv.mean() > 0.9, conv.mean()
    for f in ("map_A", "map_q", "map_c", "map_phi", "map_D_max", "map_null_q", "map_null_phi"):
        bad = ~close(fit[f][conv], exp[f][conv], 1e-5, 1e-9)
        assert not bad.any(), (P, f)
    assert np.max(np.abs(fit["map_logp"][conv] - exp["map_logp"][conv])) < 1e-6
    for fwd_rev in (0, 1):
        got = ctx.map_batch(tid, k, N, _lib.default_config(do_fwd_rev=fwd_rev))
        want = map_oracle.map_batch(tid, k, N, oracle.default_config(do_fwd_rev=fwd_rev))
        r = got["run"]
        for a, b in (("q", "map_q"), ("A", "map_A"), ("c", "map_c"), ("phi", "map_phi"), ("logp", "map_logp")):
            assert r[:, 0][a].tobytes() == fit[b].tobytes(), (P, fwd_rev, a)
        for a, b in (("q", "map_null_q"), ("phi", "map_null_phi"), ("logp", "map_null_logp")):
            assert r[:, 1][a].tobytes() == fit[b].tobytes(), (P, fwd_rev, a)
        for f in ("N_z1_forward", "N_z1_reverse", "N_sum_total", "y_sum_forward", "y_sum_reverse"):
            assert np.array_equal(got[f], want[f]), f
        for run in range(6 if fwd_rev else 2):
            g, e = got["run"][:, run], want["run"][:, run]
            conv = ((g["flags"] | e["flags"]) & 0x2) == 0
            assert conv.mean() >= 0.9, (P, run, conv.mean())
            # A PMD mode with c on its boundary (c < 1e-9; with few positions per strand, most of them): the log density
            # is flat along logit c there (an unconstrained sd of 1e4 to 1e5), so where each optimiser stops along it
            # follows rounding. c agrees to its 1e-9 absolute tolerance, but c_std = c x that sd does not, so c_std is
            # not compared on these rows. Rarely one side also stops short of the mode in the other parameters (at
            # P = 7 the oracle stopped 0.4 below the kernel's log density, with an indefinite Hessian); at most two such
            # rows per run are left out of the comparisons.
            edge = np.zeros(len(tid), bool)
            if run % 2 == 0:
                edge = conv & ((g["c"] < 1e-9) | (e["c"] < 1e-9))
                short = edge & (np.abs(g["logp"] - e["logp"]) > 1e-6)
                assert short.sum() <= 2, (P, run, np.flatnonzero(short))
                conv &= ~short
            # With one position per strand (P = 1), q of a forward-only or reverse-only PMD fit is identified by its
            # prior alone: the Hessian along q is nearly singular and whether it is positive definite (the
            # MDG_FIT_COV_INVALID flag) can go either way by rounding. There the flags and the standard deviations are
            # compared only where both sides found a positive-definite Hessian.
            cov = conv & ((e["flags"] & 0x10) == 0)
            if P == 1:
                cov &= (g["flags"] & 0x10) == 0
                assert np.array_equal(g["flags"][cov], e["flags"][cov]), (P, run)
            else:
                assert np.array_equal(g["flags"][conv], e["flags"][conv]), (P, run)
            for f in (("q", "A", "c", "phi") if run % 2 == 0 else ("q", "phi")):
                assert close(g[f][conv], e[f][conv], 1e-5, 1e-9).all(), (P, run, f)
            for f in (("q_std", "A_std", "c_std", "phi_std") if run % 2 == 0 else ("q_std", "phi_std")):
                sel = cov & ~edge if f == "c_std" else cov
                assert close(g[f][sel], e[f][sel], 1e-4, 1e-9).all(), (P, run, f)
            for f in ("logp", "loglik"):
                assert np.max(np.abs(g[f][conv] - e[f][conv])) < 1e-6, (P, run, f)


# ------------------------------------------------------------------ shapes and memory at MDG_MAX_POSITION
def test_every_cta_slot_at_max_position_64(ctx):
    """12 000 TaxIDs at P = 64 (the 17-slot shared-memory layout of the NUTS kernel, one CTA per SM, and the WAIC
    accumulators sized for it) fill every CTA slot; the rows equal those of two calls on the halves, bit for bit."""
    P = 64
    tid, k, N = syn.dense_fit_batch_shares(12_000, 1, max_position=P)
    N[::7, 40:] = 0  # rows with uncovered positions
    k[::7, 40:] = 0
    cfg = _lib.default_config(num_warmup=12, num_samples=12)
    full = ctx.fit_batch(tid, k, N, cfg, want_waic=True)
    h = len(tid) // 2 + 17
    a = ctx.fit_batch(tid[:h], k[:h], N[:h], cfg, want_waic=True)
    b = ctx.fit_batch(tid[h:], k[h:], N[h:], cfg, want_waic=True)
    for key in ("result", "median", "hpdi_lo", "hpdi_hi", "waic"):
        assert full[key].tobytes() == np.concatenate([a[key], b[key]]).tobytes(), key
    for key in ("median", "hpdi_lo", "hpdi_hi"):
        assert full[key].shape == (len(tid), 2 * P)
        assert np.array_equal(np.isnan(full[key]), N == 0), key
    assert (full["result"]["status"] & FIT_FAILED).sum() == 0


# ------------------------------------------------------------------ counts at the same P
@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_counts_match_oracle_at_max_position(ctx, oracle, P):
    """Input generated at P = 64, reduced at max_position P: rows with |z| > P are cut, and the dense rows are 2P
    wide (not a multiple of 4 when P is odd). Bit-exact with the oracle."""
    g = syn.make_mismatch_matrix(2000, max_position=64, seed=303)
    kw = dict(max_position=P, min_alignments=10, min_y_sum=10)
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], want_noise=True, **kw)
    o = oracle.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], **kw)
    assert r["n_tax"] > 0 and r["k"].shape[1] == 2 * P
    assert_same(r, o)
