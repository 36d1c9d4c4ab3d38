"""The oracle's MAP-only screening (orc_map_batch, the restatement of mdg_map_batch) against independent
computations: the Laplace covariance from a Hessian taken directly in theta with scipy's densities, the
forward-only / reverse-only fits against scipy.optimize on the masked data, the likelihood-ratio tail against
scipy's chi-square and ndtri_exp, and D_max_std against the exact posterior by quadrature."""
import numpy as np
import pytest
from scipy import optimize, special, stats

from conftest import pmd_posterior_quadrature
from metadamage_b200 import synthetic as syn
from test_oracle_nuts import PMD_QUADRATURE_CASES, synthetic_taxon


@pytest.fixture(scope="module")
def map_oracle(oracle):
    """the MAP-only restatement (oracle/map_oracle.c, compiled with the oracle it builds on)"""
    from oracle import map_oracle as M

    M.build()
    return M


def sample_batch(oracle, sample_inputs):
    tid, k, N = [], [], []
    for name in ("ancient", "control"):
        s = sample_inputs[name]
        r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
        tid.append(r["tax_id"] + (10 ** 6 if name == "control" else 0))
        k.append(r["k"])
        N.append(r["N"])
    return np.concatenate(tid), np.vstack(k), np.vstack(N)


def positions(P, mask):
    """dense slots and |z| - 1 of lane mask 0 (all), 1 (forward), 2 (reverse)"""
    slots = np.arange(2 * P) if mask == 0 else (np.arange(P) if mask == 1 else np.arange(P, 2 * P))
    return slots, slots % P


def log_post_theta(theta, k, N, model, mask):
    """constrained-space log posterior (no Jacobian) with scipy.stats: theta = (q, A, c, phi) or (q, phi)"""
    P = len(k) // 2
    slots, x = positions(P, mask)
    if model == 0:
        q, A, c, phi = theta
        Dz = A * (1.0 - q) ** x + c
        lp = stats.beta.logpdf(q, 2, 3) + stats.beta.logpdf(A, 2, 3) + stats.beta.logpdf(c, 1, 9)
    else:
        q, phi = theta
        Dz = np.full(len(x), q)
        lp = stats.beta.logpdf(q, 2, 3)
    if not (np.all(Dz > 0) and np.all(Dz < 1) and phi > 2.0):
        return -np.inf
    lp += stats.expon.logpdf(phi - 2.0, scale=1000.0)
    ll = stats.betabinom.logpmf(k[slots], N[slots], Dz * phi, (1.0 - Dz) * phi).sum()
    return lp + ll, ll


def theta_of(run, model):
    return np.array([run["q"], run["A"], run["c"], run["phi"]] if model == 0 else [run["q"], run["phi"]])


def hessian_cov_theta(theta, sd, k, N, model, mask):
    """inverse of the negative Hessian of log_post_theta in theta: central differences with steps rel_step * sd and
    twice that, Richardson-extrapolated. The steps are a compromise between the round-off of scipy's log-pmf, which
    grows with N (lgamma terms of 1e8 at N ~ 1e7), and the higher derivatives of a less Gaussian posterior at low N."""
    rel_step = 0.08 if N.max() > 10 ** 5 else 0.01
    H1 = hessian_theta(theta, rel_step * sd, k, N, model, mask)
    H2 = hessian_theta(theta, 2 * rel_step * sd, k, N, model, mask)
    return np.linalg.inv(-(4.0 * H1 - H2) / 3.0)


def hessian_theta(theta, h, k, N, model, mask):
    D = len(theta)
    f = lambda t: log_post_theta(t, k, N, model, mask)[0]  # noqa: E731
    H = np.zeros((D, D))
    for i in range(D):
        for j in range(i, D):
            ei, ej = np.eye(D)[i] * h[i], np.eye(D)[j] * h[j]
            if i == j:
                H[i, i] = (f(theta + ei) - 2.0 * f(theta) + f(theta - ei)) / h[i] ** 2
            else:
                H[i, j] = H[j, i] = (f(theta + ei + ej) - f(theta + ei - ej) - f(theta - ei + ej) + f(theta - ei - ej)) / (4.0 * h[i] * h[j])
    return H


def interior_cfg2_batch(map_oracle, n=20):
    """cfg2 TaxIDs whose PMD and null modes are away from every bound, with clean fits"""
    tid, k, N, _ = syn.dense_fit_batch(600)
    res = map_oracle.map_batch(tid, k, N)
    r0, r1 = res["run"][:, 0], res["run"][:, 1]
    ok = (res["status"] == 0) & (r0["A"] > 0.02) & (r0["c"] > 2e-3) & (r0["q"] > 0.02) & (r0["q"] < 0.98)
    ok &= (r0["phi"] > 5.0) & (r1["phi"] > 5.0) & (r0["phi"] < 1e5) & (r1["phi"] < 1e5)
    pick = np.flatnonzero(ok)[:n]
    assert len(pick) == n
    return tid[pick], k[pick], N[pick], res[pick]


def check_laplace(row, k, N, tag):
    for run_kind, model in ((0, 0), (1, 1)):
        run = row["run"][run_kind]
        assert run["flags"] == 0, (tag, run_kind)
        theta = theta_of(run, model)
        sd = np.array([run["q_std"], run["A_std"], run["c_std"], run["phi_std"]] if model == 0 else [run["q_std"], run["phi_std"]])
        cov = hessian_cov_theta(theta, sd, k, N, model, 0)
        np.testing.assert_allclose(sd, np.sqrt(np.diag(cov)), rtol=1e-3, err_msg=f"{tag} run {run_kind}")
        if model == 0:
            rho = cov[1, 2] / np.sqrt(cov[1, 1] * cov[2, 2])
            assert abs(row["rho_Ac"] - rho) < 1e-3 * abs(rho), (tag, row["rho_Ac"], rho)
            assert abs(row["D_max_std"] - np.sqrt(cov[1, 1] + cov[2, 2] + 2 * cov[1, 2])) < 1e-3 * row["D_max_std"], tag


def test_laplace_matches_hessian_in_theta_sample_taxa(oracle, sample_inputs, map_oracle):
    """J Sigma_u J (the oracle) == inverse Hessian taken directly in theta with scipy's densities."""
    tid, k, N = sample_batch(oracle, sample_inputs)
    res = map_oracle.map_batch(tid, k, N)
    assert len(res) == 6
    for i in range(len(res)):
        check_laplace(res[i], k[i], N[i], tid[i])


def test_laplace_matches_hessian_in_theta_cfg2(map_oracle):
    tid, k, N, res = interior_cfg2_batch(map_oracle)
    for i in range(len(res)):
        check_laplace(res[i], k[i], N[i], tid[i])


def test_forward_reverse_fits_match_independent_optimiser(oracle, sample_inputs, map_oracle):
    """Forward-only and reverse-only MAP fits: logp / loglik are scipy's on the masked positions, the mode is a
    stationary point, and Nelder-Mead from a perturbed start finds nothing better."""
    tid, k, N = sample_batch(oracle, sample_inputs)
    res = map_oracle.map_batch(tid, k, N)
    for i in (0, 3, 5):
        for run_kind in (2, 3, 4, 5):
            model, mask = run_kind & 1, run_kind // 2
            run = res[i]["run"][run_kind]
            assert run["flags"] == 0, (i, run_kind)
            theta = theta_of(run, model)
            lp, ll = log_post_theta(theta, k[i], N[i], model, mask)
            scale = 1e-9 * max(1.0, abs(lp))
            assert abs(run["logp"] - lp) < 1e-6 + scale and abs(run["loglik"] - ll) < 1e-6 + scale, (i, run_kind)

            def f(u):
                v = -oracle.logp_grad(k[i], N[i], u[None, :], model=model, lane_mask=mask, with_jacobian=False)[0][0]
                return v if np.isfinite(v) else 1e30

            u0 = np.log(theta[:-1] / (1.0 - theta[:-1])).tolist() + [np.log(theta[-1] - 2.0)]
            u0 = np.array(u0 + [0.0] * (4 - len(u0)))
            D = 4 if model == 0 else 2
            fu = lambda v: f(np.r_[v, np.zeros(4 - D)])  # noqa: E731
            opt = optimize.minimize(fu, u0[:D] + 0.3, method="Nelder-Mead", options=dict(xatol=1e-9, fatol=1e-11, maxiter=8000))
            assert -opt.fun <= run["logp"] + 2e-5, (i, run_kind, -opt.fun, run["logp"])
            _, grad, _ = oracle.logp_grad(k[i], N[i], u0[None, :], model=model, lane_mask=mask, with_jacobian=False)
            assert np.max(np.abs(grad[0, :D])) < 1e-4 * max(1.0, N[i].max() * 1e-3), (i, run_kind, grad)
        # the derived forward / reverse statistics are those of the pairs of fits
        r = res[i]["run"]
        assert res[i]["forward_D_max"] == r[2]["A"] + r[2]["c"] and res[i]["reverse_D_max"] == r[4]["A"] + r[4]["c"]
        assert res[i]["forward_lambda_LR"] == 2 * (r[2]["loglik"] - r[3]["loglik"])
        assert res[i]["reverse_lambda_LR"] == 2 * (r[4]["loglik"] - r[5]["loglik"])


def test_likelihood_ratio_tail_matches_scipy(map_oracle):
    lam = np.array([-1.0, 0.0, 1e-8, 3.0, 50.0, 5000.0])
    P, z = map_oracle.lr_tail(lam)
    lam0 = np.maximum(lam, 0.0)
    np.testing.assert_allclose(P, stats.chi2.sf(lam0, 2), rtol=1e-12, atol=0)
    np.testing.assert_allclose(z, -special.ndtri_exp(-lam0 / 2), rtol=1e-12, atol=0)
    assert np.isfinite(z[-1]) and z[-1] > 70 and P[-1] == 0.0
    assert np.all(np.isnan(map_oracle.lr_tail([np.nan])))


def test_likelihood_ratio_in_rows(oracle, sample_inputs, map_oracle):
    tid, k, N = sample_batch(oracle, sample_inputs)
    res = map_oracle.map_batch(tid, k, N)
    r = res["run"]
    np.testing.assert_array_equal(res["lambda_LR"], 2 * (r[:, 0]["loglik"] - r[:, 1]["loglik"]))
    P, z = map_oracle.lr_tail(res["lambda_LR"])
    np.testing.assert_array_equal(res["lambda_LR_P"], P)
    np.testing.assert_array_equal(res["lambda_LR_z"], z)
    # the strongly damaged ancient sample is decisive, D_max = A + c at the mode
    assert np.all(res["lambda_LR"][:3] > 150) and np.all(res["significance"][:3] > 50)
    np.testing.assert_array_equal(res["D_max"], r[:, 0]["A"] + r[:, 0]["c"])


def test_dmax_std_close_to_exact_posterior_sd(map_oracle):
    """High-coverage PMD case of the quadrature tests: the Laplace sd of A + c is within 10 % of the exact one."""
    seed, kw = PMD_QUADRATURE_CASES[0]
    k, N = synthetic_taxon(seed, **kw)
    truth = pmd_posterior_quadrature(k, N)
    res = map_oracle.map_batch(np.array([seed], np.int64), k[None, :], N[None, :])
    assert res["status"][0] == 0
    exact = np.sqrt(truth["var_D_max"])
    assert abs(res["D_max_std"][0] - exact) < 0.10 * exact, (res["D_max_std"][0], exact)


def test_all_position_fits_are_the_fit_paths_map(oracle, sample_inputs, map_oracle):
    """The all-position runs of the MAP-only path are the same fits as orc_fit_batch's map_* fields."""
    tid, k, N = sample_batch(oracle, sample_inputs)
    res = map_oracle.map_batch(tid, k, N, map_oracle.default_config(do_fwd_rev=0))
    fit = oracle.fit_batch(tid, k, N, oracle.default_config(num_warmup=4, num_samples=4, do_fwd_rev=0))["result"]
    r = res["run"]
    for a, b in (("A", "map_A"), ("q", "map_q"), ("c", "map_c"), ("phi", "map_phi"), ("logp", "map_logp")):
        np.testing.assert_array_equal(r[:, 0][a], fit[b])
    for a, b in (("q", "map_null_q"), ("phi", "map_null_phi"), ("logp", "map_null_logp")):
        np.testing.assert_array_equal(r[:, 1][a], fit[b])
    # runs not made are NaN with no evaluations
    assert np.all(np.isnan(r[:, 2:]["q"])) and np.all(r[:, 2:]["n_eval"] == 0) and np.all(np.isnan(res["forward_D_max"]))


@pytest.mark.parametrize("P", [15, 40])
def test_edge_rows_are_defined(oracle, P, map_oracle):
    """n_tax = 0 and a TaxID without any coverage give defined results."""
    empty = map_oracle.map_batch(np.zeros(0, np.int64), np.zeros((0, 2 * P), np.uint32), np.zeros((0, 2 * P), np.uint32))
    assert len(empty) == 0
    z = np.zeros((1, 2 * P), np.uint32)
    row = map_oracle.map_batch(np.array([5], np.int64), z, z)[0]
    assert row["status"] & 1 == 0 and row["N_sum_total"] == 0 and np.isfinite(row["run"][0]["q"])
