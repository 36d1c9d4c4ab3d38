"""Pins of the oracle's model / sampler building blocks against independent implementations:
scipy.stats.betabinom, scipy.special, finite differences, Random123 known answers, and the
reference's own WAIC / n_sigma / asymmetry functions (fits_golden.npz)."""
import numpy as np
import pytest
from scipy import optimize, special, stats


def unconstrained(q, A, c, phi):
    lg = lambda p: np.log(p / (1 - p))  # noqa: E731
    return np.array([lg(q), lg(A), lg(c), np.log(phi - 2.0)])


def test_philox_known_answers(oracle):
    """Philox4x32-10 vectors of the Random123 distribution (kat_vectors)."""
    assert list(oracle.philox([0, 0], [0, 0, 0, 0])) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert list(oracle.philox([0xFFFFFFFF] * 2, [0xFFFFFFFF] * 4)) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert list(oracle.philox([0xA4093822, 0x299F31D0], [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344])) == \
        [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_special_functions(oracle):
    x = np.concatenate([10.0 ** np.linspace(-8, 8, 200), np.linspace(0.05, 25, 300)])
    np.testing.assert_allclose(oracle.digamma(x), special.digamma(x), rtol=2e-14, atol=2e-14)
    np.testing.assert_allclose(oracle.lgamma(x), special.gammaln(x), rtol=2e-14, atol=2e-14)


def dense_sample(oracle, sample_inputs, name):
    s = sample_inputs[name]
    return oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])


def test_loglik_known_answers(oracle, sample_inputs):
    """SURVEY.md 8c: sum of scipy betabinom.logpmf at A=0.4, q=0.3, c=0.02, phi=1000 (FP64)."""
    u = unconstrained(0.3, 0.4, 0.02, 1000.0)[None, :]
    expected = {"ancient": [-825.2253953129, -705.0723966804, -715.4612424145],
                "control": [-10695.9844079475, -7618.8591743020, -7055.8278667361]}
    z = np.r_[np.arange(15), np.arange(15)]
    Dz = 0.4 * 0.7 ** z + 0.02
    for name, vals in expected.items():
        r = dense_sample(oracle, sample_inputs, name)
        for t, val in enumerate(vals):
            logp, grad, ll = oracle.logp_grad(r["k"][t], r["N"][t], u, with_jacobian=False)
            # lgamma sums of magnitude 1e8 cancel to 1e1: 1e-7 absolute is the FP64 floor
            assert abs(ll.sum() - val) < 2e-6
            ref = stats.betabinom.logpmf(r["k"][t], r["N"][t], Dz * 1000.0, (1 - Dz) * 1000.0)
            np.testing.assert_allclose(ll[0], ref, atol=2e-7)
            # log prior at the same point
            assert abs((logp[0] - ll.sum()) - (-4.7556037322)) < 1e-9
    r = dense_sample(oracle, sample_inputs, "ancient")
    _, _, ll = oracle.logp_grad(r["k"][0], r["N"][0], u, with_jacobian=False)
    assert abs(ll[0, 0] - (-13.1755879209)) < 1e-7


@pytest.mark.parametrize("model", [0, 1])
@pytest.mark.parametrize("mask", [0, 1, 2])
@pytest.mark.parametrize("jac", [True, False])
def test_gradient_matches_finite_differences(oracle, model, mask, jac):
    rng = np.random.default_rng(10 * model + mask)
    N = rng.integers(5, 400, 30).astype(np.uint32)
    k = rng.binomial(N, 0.1).astype(np.uint32)
    for trial in range(5):
        u = rng.uniform(-1.5, 1.5, 4)
        u[2] -= 2.0
        u[3] += 3.0
        if model == 1:
            u[1] = u[3]
        logp, grad, _ = oracle.logp_grad(k, N, u[None, :], model=model, lane_mask=mask, with_jacobian=jac)
        D = 4 if model == 0 else 2
        if not np.isfinite(logp[0]):
            continue
        for j in range(D):
            h = 1e-5
            up, um = u.copy(), u.copy()
            up[j] += h
            um[j] -= h
            fp = oracle.logp_grad(k, N, up[None, :], model=model, lane_mask=mask, with_jacobian=jac)[0][0]
            fm = oracle.logp_grad(k, N, um[None, :], model=model, lane_mask=mask, with_jacobian=jac)[0][0]
            fd = (fp - fm) / (2 * h)
            assert abs(fd - grad[0, j]) < 1e-5 * (1 + abs(fd))


def test_invalid_region_is_nan(oracle):
    """A + c >= 1 -> clip(Dz,0,1) = 1 -> beta = 0 -> NaN in the reference (fits.py:50)."""
    N = np.full(30, 100, np.uint32)
    k = np.full(30, 10, np.uint32)
    u = unconstrained(0.3, 0.8, 0.5, 100.0)[None, :]
    logp, _, _ = oracle.logp_grad(k, N, u)
    assert np.isnan(logp[0])


def test_zero_coverage_positions_contribute_nothing(oracle):
    rng = np.random.default_rng(1)
    N = rng.integers(5, 400, 30).astype(np.uint32)
    k = rng.binomial(N, 0.1).astype(np.uint32)
    u = unconstrained(0.3, 0.2, 0.02, 50.0)[None, :]
    _, _, ll = oracle.logp_grad(k, N, u)
    N2, k2 = N.copy(), k.copy()
    N2[7] = 0
    k2[7] = 0
    _, _, ll2 = oracle.logp_grad(k2, N2, u)
    assert ll2[0, 7] == 0.0  # BetaBinomial(N=0).log_prob(0) = 0
    np.testing.assert_array_equal(np.delete(ll2[0], 7), np.delete(ll[0], 7))


def test_waic_nsigma_asymmetry_match_reference(oracle, fits_golden):
    """fits.get_lppd_and_waic / compute_n_sigma / compute_assymmetry... (fits.py:147-227)."""
    g = fits_golden
    for name in ("pmd", "null"):
        lp = g[f"logprob_{name}"]
        lppd_i = special.logsumexp(lp, 0) - np.log(lp.shape[0])
        np.testing.assert_allclose(lppd_i, g[f"{name}_lppd_i"], rtol=1e-13)
    assert abs(oracle.n_sigma(g["pmd_waic_i"], g["null_waic_i"]) - float(g["n_sigma"])) < 1e-10
    # full oracle path: per-sample log-likelihood -> lppd_i / pWAIC_i from constrained draws
    k, N = g["data_y"].astype(np.uint32), g["data_N"].astype(np.uint32)
    th = g["theta_pmd"]
    u = np.stack([np.log(th[:, 0] / (1 - th[:, 0])), np.log(th[:, 1] / (1 - th[:, 1])),
                  np.log(th[:, 2] / (1 - th[:, 2])), np.log(th[:, 3] - 2.0)], 1)
    _, _, ll = oracle.logp_grad(k, N, u)
    np.testing.assert_allclose(ll, g["logprob_pmd"], atol=5e-9)
    waic_i = -2 * ((special.logsumexp(ll, 0) - np.log(len(ll))) - ll.var(0))
    np.testing.assert_allclose(waic_i, g["pmd_waic_i"], rtol=1e-8)


def test_median_and_hpdi(oracle, fits_golden):
    x = fits_golden["median_in"]
    for j in range(x.shape[1]):
        med, lo, hi = oracle.median_hpdi(x[:, j], 0.68)
        assert med == fits_golden["median_out"][j]
        # numpyro.diagnostics.hpdi restated: narrowest window holding int(0.68*S) steps
        s = np.sort(x[:, j])
        L = int(0.68 * len(s))
        i = np.argmin(s[L:] - s[: len(s) - L])
        assert (lo, hi) == (s[i], s[i + L])


def test_adaptation_schedule(oracle):
    """numpyro 0.4.1 build_adaptation_schedule (Stan windows) for the reference's 500 warm-up steps."""
    assert oracle.adaptation_schedule(500) == [(0, 74), (75, 99), (100, 149), (150, 249), (250, 449), (450, 499)]
    assert oracle.adaptation_schedule(10) == [(0, 9)]
    assert oracle.adaptation_schedule(100) == [(0, 14), (15, 89), (90, 99)]


def test_map_matches_independent_optimiser(oracle, sample_inputs):
    """MAP (new deliverable): LM-Newton result vs scipy on the same constrained-space density."""
    for name, idx in (("ancient", 0), ("control", 0), ("control", 2)):
        r = dense_sample(oracle, sample_inputs, name)
        k, N = r["k"][idx], r["N"][idx]
        m = oracle.map_fit(k, N)
        assert m["converged"]

        def f(u):
            v = -oracle.logp_grad(k, N, u[None, :], with_jacobian=False)[0][0]
            return v if np.isfinite(v) else 1e30

        u0 = unconstrained(m["q"], m["A"], m["c"], m["phi"])
        res = optimize.minimize(f, u0 + 0.3, method="Nelder-Mead", options=dict(xatol=1e-9, fatol=1e-11, maxiter=8000))
        assert -res.fun <= m["logp"] + 2e-5  # nothing better nearby (1e-6 is the FP64 noise of the lgamma sums at N ~ 1e7)
        _, grad, _ = oracle.logp_grad(k, N, u0[None, :], with_jacobian=False)
        assert np.max(np.abs(grad)) < 1e-4 * max(1.0, N.max() * 1e-3)
    # indicative values of SURVEY.md 8c
    r = dense_sample(oracle, sample_inputs, "ancient")
    m = oracle.map_fit(r["k"][0], r["N"][0])
    assert abs(m["A"] - 0.393) < 2e-3 and abs(m["q"] - 0.533) < 2e-3 and abs(m["c"] - 0.0248) < 2e-4
