"""The oracle's profile intervals of D_max (orc_map_profile, the restatement of mdg_map_profile) against independent
computations: each end checked with scipy's densities and Nelder-Mead at that D, an inner fit by scipy.optimize with
brentq for the end, the exact posterior by quadrature, and coverage of the generator's true A + c."""
import numpy as np
import pytest
from scipy import optimize, special

from conftest import pmd_posterior_quadrature
from metadamage_b200 import synthetic as syn
from metadamage_b200._abi import FIT_FAILED, PROFILE_AT_BOUND, PROFILE_FAILED
from test_oracle_map import interior_cfg2_batch, log_post_theta, sample_batch
from test_oracle_nuts import PMD_QUADRATURE_CASES, synthetic_taxon

T68 = special.ndtri(0.84) ** 2  # chi-square(1) quantile at 0.68


@pytest.fixture(scope="module")
def map_oracle(oracle):
    from oracle import map_oracle as M

    M.build()
    return M


@pytest.fixture(scope="module")
def prof():
    import map_profile_oracle as P

    P.build()
    return P


def theta_at(e):
    return np.array([e["q"], e["A"], e["c"], e["phi"]])


def v_of(theta, D):
    """(logit q, logit s, log(phi - 2)) of theta on A + c = D"""
    q, A, c, phi = theta
    return np.array([np.log(q / (1 - q)), np.log(A / c), np.log(phi - 2.0)])


def theta_of_v(v, D):
    s = 1.0 / (1.0 + np.exp(-v[1]))
    return np.array([1.0 / (1.0 + np.exp(-v[0])), D * s, D * (1.0 - s), np.exp(v[2]) + 2.0])


def check_ends(oracle, k, N, row, iv, tag):
    assert iv["threshold"] == pytest.approx(T68, rel=1e-12) and iv["level"] == 0.68
    for prof in range(3):
        run = row["run"][2 * prof]
        Dhat = run["A"] + run["c"]
        ends = iv["end"][prof]
        assert ends[0]["D"] <= Dhat <= ends[1]["D"], (tag, prof)
        for side in range(2):
            e = ends[side]
            assert (e["flags"] & (PROFILE_FAILED | FIT_FAILED)) == 0 and e["n_eval"] > 0, (tag, prof, side)
            at_bound = bool(e["flags"] & PROFILE_AT_BOUND)
            assert at_bound or abs(e["A"] + e["c"] - e["D"]) <= 4e-16 * e["D"], (tag, prof, side)
            lp = log_post_theta(theta_at(e), k, N, 0, prof)[0]
            assert abs(e["logp"] - lp) < 1e-6 + 1e-9 * abs(lp), (tag, prof, side, e["logp"], lp)
            if not at_bound:
                assert abs(2 * (run["logp"] - e["logp"]) - T68) < 1e-5, (tag, prof, side)
            # nothing better on A + c = D (the oracle's density, whose values were just checked against scipy's)
            D = e["A"] + e["c"]

            def f(v):
                th = theta_of_v(v, D)
                u = np.r_[np.log(th[:3] / (1 - th[:3])), np.log(th[3] - 2.0)]
                val = -oracle.logp_grad(k, N, u[None, :], model=0, lane_mask=prof, with_jacobian=False)[0][0]
                return val if np.isfinite(val) else 1e30

            opt = optimize.minimize(f, v_of(theta_at(e), D) + 0.2, method="Nelder-Mead",
                                    options=dict(xatol=1e-9, fatol=1e-11, maxiter=4000))
            assert -opt.fun <= e["logp"] + 2e-5, (tag, prof, side, -opt.fun, e["logp"])


def test_each_end_sample_taxa(oracle, sample_inputs, map_oracle, prof):
    tid, k, N = sample_batch(oracle, sample_inputs)
    rows = map_oracle.map_batch(tid, k, N)
    iv = prof.map_profile(k, N, rows)
    assert np.array_equal(iv["tax_id"], tid)
    for i in range(len(iv)):
        check_ends(oracle, k[i], N[i], rows[i], iv[i], tid[i])


def test_each_end_interior_cfg2(oracle, map_oracle, prof):
    tid, k, N, rows = interior_cfg2_batch(map_oracle)
    iv = prof.map_profile(k, N, rows)
    for i in range(len(iv)):
        check_ends(oracle, k[i], N[i], rows[i], iv[i], tid[i])


def scipy_profile(k, N, theta0, D, mask):
    """max of scipy's log posterior on A + c = D by Nelder-Mead then Powell from theta0 (independent of the oracle)"""
    def f(v):
        lp = log_post_theta(theta_of_v(v, D), k, N, 0, mask)
        return -lp[0] if isinstance(lp, tuple) else 1e30

    v0 = v_of(theta0, theta0[1] + theta0[2])
    opt = optimize.minimize(f, v0, method="Nelder-Mead", options=dict(xatol=1e-10, fatol=1e-12, maxiter=6000))
    opt = optimize.minimize(f, opt.x, method="Powell", options=dict(xtol=1e-10, ftol=1e-13))
    return -opt.fun


def test_ends_match_independent_profile(map_oracle, prof):
    tid, k, N, rows = interior_cfg2_batch(map_oracle, n=20)
    iv = prof.map_profile(k, N, rows)
    for i in (0, 7, 13):
        run = rows[i]["run"][0]
        theta0 = np.array([run["q"], run["A"], run["c"], run["phi"]])
        Dhat = run["A"] + run["c"]
        for side in range(2):
            end = iv[i]["end"][0][side]["D"]
            h = lambda D: 2 * (run["logp"] - scipy_profile(k[i], N[i], theta0, D, 0)) - T68  # noqa: E731
            far = Dhat + 2.0 * (end - Dhat)
            root = optimize.brentq(h, Dhat + 0.05 * (end - Dhat), far, xtol=1e-12, rtol=1e-12)
            assert abs(root - end) <= 1e-4 * end, (tid[i], side, root, end)


def test_ends_close_to_exact_posterior():
    """High-coverage PMD case of the quadrature tests: each end is within 10 % of the interval width of the exact
    posterior's mean +- z sd of A + c (z = Phi^-1(0.84)), the tolerance of the D_max_std test."""
    from oracle import map_oracle
    import map_profile_oracle as P

    seed, kw = PMD_QUADRATURE_CASES[0]
    k, N = synthetic_taxon(seed, **kw)
    truth = pmd_posterior_quadrature(k, N)
    rows = map_oracle.map_batch(np.array([seed], np.int64), k[None, :], N[None, :])
    iv = P.map_profile(k[None, :], N[None, :], rows)[0]
    z = special.ndtri(0.84)
    sd = np.sqrt(truth["var_D_max"])
    lo, hi = truth["mean_D_max"] - z * sd, truth["mean_D_max"] + z * sd
    width = hi - lo
    ends = iv["end"][0]
    assert abs(ends[0]["D"] - lo) < 0.10 * width and abs(ends[1]["D"] - hi) < 0.10 * width, (ends["D"], lo, hi)


def test_coverage_of_true_damage(map_oracle, prof):
    """On 2 000 cfg2 TaxIDs, the share of 0.68 profile intervals that cover the generator's true A + c, next to that of
    D_max +- D_max_std (DESIGN K3p records both). The generator's damage is not drawn from the prior: at cfg2's
    coverage the mode sits above the truth for most TaxIDs (the Beta(2, 3) prior on A), and the profile interval, which
    extends further up than down there, misses below more often than the symmetric one. Hence a loose band."""
    tid, k, N, g = syn.dense_fit_batch(2000)
    truth = (g["truth"]["A"] + g["truth"]["c"])[g["passes"]]
    rows = map_oracle.map_batch(tid, k, N, map_oracle.default_config(do_fwd_rev=0))
    iv = prof.map_profile(k, N, rows, map_oracle.default_config(do_fwd_rev=0))
    ends = iv["end"][:, 0]
    ok = (iv["status"] & (PROFILE_FAILED | FIT_FAILED)) == 0
    assert ok.mean() > 0.99
    cover = (ends[ok, 0]["D"] <= truth[ok]) & (truth[ok] <= ends[ok, 1]["D"])
    lap = np.isfinite(rows["D_max_std"]) & ok
    cover_lap = np.abs(rows["D_max"][lap] - truth[lap]) <= rows["D_max_std"][lap]
    print(f"profile coverage {cover.mean():.4f} of {ok.sum()}, Laplace coverage {cover_lap.mean():.4f} of {lap.sum()}, "
          f"ends at a bound {np.mean(ends[ok]['flags'] & PROFILE_AT_BOUND != 0):.4f}")
    assert 0.45 <= cover.mean() <= 0.82 and 0.45 <= cover_lap.mean() <= 0.82


@pytest.mark.parametrize("P", [15, 40])
def test_edge_cases(map_oracle, prof, P):
    empty = prof.map_profile(np.zeros((0, 2 * P), np.uint32), np.zeros((0, 2 * P), np.uint32), map_oracle.map_batch(
        np.zeros(0, np.int64), np.zeros((0, 2 * P), np.uint32), np.zeros((0, 2 * P), np.uint32)))
    assert len(empty) == 0
    # no coverage at all: the MAP is the prior's mode, the profile the prior's
    z = np.zeros((1, 2 * P), np.uint32)
    rows = map_oracle.map_batch(np.array([5], np.int64), z, z)
    iv = prof.map_profile(z, z, rows)[0]
    assert iv["tax_id"] == 5 and (iv["status"] & (PROFILE_FAILED | FIT_FAILED)) == 0
    assert np.all(np.isfinite(iv["end"]["D"])) and np.all(iv["end"]["D"][:, 0] < iv["end"]["D"][:, 1])
    # without forward / reverse fits their ends are NaN with no evaluations and no flags
    tid, k, N, _ = syn.dense_fit_batch(6, max_position=P)
    cfg = map_oracle.default_config(do_fwd_rev=0)
    rows = map_oracle.map_batch(tid, k, N, cfg)
    iv = prof.map_profile(k, N, rows, cfg)
    assert np.all(np.isnan(iv["end"]["D"][:, 1:])) and np.all(iv["end"]["n_eval"][:, 1:] == 0)
    assert np.all(iv["end"]["flags"][:, 1:] == 0) and np.all(np.isfinite(iv["end"]["D"][:, 0]))
    # a failed MAP run gives NaN ends flagged MDG_FIT_FAILED, and the row status carries it
    rows["run"][0, 0]["flags"] = FIT_FAILED
    iv2 = prof.map_profile(k, N, rows, cfg)
    assert np.all(np.isnan(iv2["end"]["D"][0, 0])) and np.all(iv2["end"]["flags"][0, 0] == FIT_FAILED)
    assert iv2["status"][0] == FIT_FAILED and iv2[1:].tobytes() == iv[1:].tobytes()
    for level in (0.0, 1.0, -0.5, np.nan):
        with pytest.raises(ValueError):
            prof.map_profile(k, N, rows, cfg, level=level)
