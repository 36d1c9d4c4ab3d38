"""The damage model's log density restated at 40 significant digits with mpmath: the reference for the FP64 log
density and gradient that the oracle (and, in test_gpu_max_position.py, the CUDA kernels) evaluate.

The model is fits.py:43-67: q ~ Beta(2, 3), A ~ Beta(2, 3), c ~ Beta(1, 9), delta ~ Exponential(1/1000),
phi = delta + 2, D_z = A (1 - q)^(|z| - 1) + c (null model: D_z = q), y_z ~ BetaBinomial(D_z phi, (1 - D_z) phi, N_z)
with log C(N, k) included, in the unconstrained coordinates (logit q, logit A, logit c, log delta) with the log
Jacobian optional. The gradient is mpmath's numerical derivative of the same 40-digit function. Every P of the
lane-layout boundary set MAX_POSITIONS is checked, for both models, all three lane masks and both Jacobian settings."""
import mpmath as mp
import numpy as np
import pytest

from metadamage_b200 import synthetic as syn

# Every max_position (P) at which some kernel's lane layout changes. MAP / eval_model spread 2P (or P for the
# forward-only and reverse-only runs) positions over NPL = 1, 2 or 4 positions per lane of a warp, with a spare
# slot when the positions do not fill NPL * 32; NUTS eval_group spreads them over 8 lanes per chain, index 0 being
# the spare, in ns = (n_obs + 8) / 8 slots.
MAX_POSITIONS = (
    1,   # one position per strand: a half run fits a single observation, so n_sigma_forward/_reverse divide by a zero variance
    2,   # the smallest P at which a half run's per-position WAIC terms have a variance
    3,   # odd: dense rows of width 2P = 6 are not a multiple of 4; NUTS fills 7 of a slot's 8 indices
    4,   # P = 4m: NUTS all-position runs (2P + spare = 9 indices) leave one index in the last slot
    7,   # P = 8m - 1: NUTS half runs (P + spare = 8 indices) fill their one slot exactly
    8,   # P = 4m and 8m: NUTS half and all-position runs both end with a single-index slot
    15,  # the suite's default geometry and the reference's sample file; NUTS half runs fill two slots exactly
    16,  # 2P = 32: the MAP warp has no spare slot (NPL = 1), so lgamma(phi) etc. come from the separate branch
    17,  # the first P past NPL = 1: MAP all-position runs take NPL = 2
    31,  # P = 8m - 1: NUTS half runs fill 4 slots exactly; MAP has a single spare slot (62 of 64)
    32,  # no spare slot for MAP all-position runs (NPL = 2) nor for the test hook's half runs (NPL = 1)
    33,  # the first P past NPL = 2: MAP all-position runs take NPL = 3, rounded up to 4
    48,  # NPL = 3 rounded up to 4: 96 of 128 slots used
    63,  # P = 8m - 1: NUTS half runs fill 8 slots exactly
    64,  # MDG_MAX_POSITION: no MAP spare slot at NPL = 4 (half runs: NPL = 2); NUTS has 17 slots, its largest shared memory
)

DPS = 40
PHI_MIN = 2
PRIORS = dict(q=(2, 3), A=(2, 3), c=(1, 9), rate=mp.mpf(1) / 1000)


def _to_mp(x):
    # a double converts to an mpf exactly; an mpf (mpmath's perturbed argument inside mp.diff) is kept as it is
    return x if isinstance(x, mp.mpf) else mp.mpf(float(x))


def _log_sigmoid(u):
    return -mp.log1p(mp.exp(-u))


def _log_beta(a, b):
    return mp.loggamma(a) + mp.loggamma(b) - mp.loggamma(a + b)


def used_positions(P, mask):
    """Dense indices of a run: 0 = all 2P positions, 1 = forward only (the first P), 2 = reverse only (the last P)."""
    return range(2 * P) if mask == 0 else (range(P) if mask == 1 else range(P, 2 * P))


def model_terms_mp(k, N, u, model, mask, jac, with_log_binom=True):
    """Every additive term of the log joint at 40 digits: (prior terms, {dense index: terms of that position}),
    or None where some D_z leaves (0, 1) (clip(D_z, 0, 1) in the reference gives NaN there). log(1 - sigmoid(u))
    is taken as log sigmoid(-u), so |u| up to 700 keeps all its digits."""
    P = len(k) // 2
    D = 4 if model == 0 else 2
    u = [_to_mp(x) for x in list(u)[:D]]
    prior = []

    def beta_prior(uj, a, b):
        lx, l1mx = _log_sigmoid(uj), _log_sigmoid(-uj)
        prior.extend([(a - 1) * lx, (b - 1) * l1mx, -_log_beta(a, b)])
        if jac:  # log |d sigmoid(u) / du| = log x + log(1 - x)
            prior.extend([lx, l1mx])

    beta_prior(u[0], *PRIORS["q"])
    if model == 0:
        beta_prior(u[1], *PRIORS["A"])
        beta_prior(u[2], *PRIORS["c"])
    delta = mp.exp(u[D - 1])
    prior.extend([mp.log(PRIORS["rate"]), -PRIORS["rate"] * delta])
    if jac:
        prior.append(u[D - 1])
    phi = delta + PHI_MIN
    q, log1mq = mp.exp(_log_sigmoid(u[0])), _log_sigmoid(-u[0])
    A = mp.exp(_log_sigmoid(u[1])) if model == 0 else None
    c = mp.exp(_log_sigmoid(u[2])) if model == 0 else None
    lg_phi = mp.loggamma(phi)
    per_pos = {}
    for i in used_positions(P, mask):
        x = i if i < P else i - P
        Dz = A * mp.exp(x * log1mq) + c if model == 0 else q
        if not 0 < Dz < 1:
            return None
        a, b = Dz * phi, (1 - Dz) * phi
        kk, nn = int(k[i]), int(N[i])
        t = [mp.loggamma(kk + a), mp.loggamma(nn - kk + b), -mp.loggamma(nn + phi), -mp.loggamma(a), -mp.loggamma(b), lg_phi]
        if with_log_binom:
            t += [mp.loggamma(nn + 1), -mp.loggamma(kk + 1), -mp.loggamma(nn - kk + 1)]
        per_pos[i] = t
    return prior, per_pos


def model_logp_mp(k, N, u, model, mask, jac):
    """log joint (+ log Jacobian if `jac`) at 40 digits; NaN where some D_z reaches 0 or 1."""
    with mp.workdps(DPS):
        parts = model_terms_mp(k, N, u, model, mask, jac)
        if parts is None:
            return mp.nan
        prior, per_pos = parts
        return mp.fsum(prior + [x for t in per_pos.values() for x in t])


def model_logp_scale(k, N, u, model, mask, jac):
    """sum of |terms| of the log joint: the size of what a double-precision evaluation cancels"""
    with mp.workdps(DPS):
        parts = model_terms_mp(k, N, u, model, mask, jac)
        if parts is None:
            return float("nan")
        prior, per_pos = parts
        return float(mp.fsum(abs(x) for x in prior + [x for t in per_pos.values() for x in t]))


def model_ll_mp(k, N, u, model, mask):
    """Per-position log-likelihood log BetaBinomial(k_i | N_i, ...) (log C(N, k) included) and the sum of |terms| of
    each: {dense index: (value, scale)}, or None where some D_z leaves (0, 1)."""
    with mp.workdps(DPS):
        parts = model_terms_mp(k, N, u, model, mask, False)
        if parts is None:
            return None
        return {i: (float(mp.fsum(t)), float(mp.fsum(abs(x) for x in t))) for i, t in parts[1].items()}


def model_grad_mp(k, N, u, model, mask, jac):
    """d log joint / du_j at 40 digits by mpmath's numerical derivative (mp.diff raises its own working precision
    for the step). The perturbation h reaches model_terms_mp as an mpf: it is never rounded back to a double.
    log C(N, k) does not depend on u and is left out."""
    D = 4 if model == 0 else 2
    with mp.workdps(DPS):
        u0 = [_to_mp(x) for x in list(u)[:D]]
        out = []
        for j in range(D):
            def f(h, j=j):
                parts = model_terms_mp(k, N, [u0[i] + h if i == j else u0[i] for i in range(D)], model, mask, jac, with_log_binom=False)
                prior, per_pos = parts
                return mp.fsum(prior + [x for t in per_pos.values() for x in t])
            out.append(float(mp.diff(f, 0)))
        return np.array(out)


def reference_points(model, seed):
    """Unconstrained points (rows of 4; the null model uses columns 0 and 1 = logit q, log delta): two from the bulk,
    and the edges the kernels special-case:
      - |u_j| just below the kernels' 700 validity bound on the sigmoid lanes (for the null model only at -699.5:
        sigmoid(u) rounds to 1 in FP64 from u ~ 37 on, so D_z = q would reach 1 in the kernels but not at 40 digits);
      - u_c << 0 (c -> 0);
      - large delta (phi ~ 1.6e5, 160 times the prior mean);
      - D_z reaching 1: A = c = 1/2 exactly (D_z = 1 at z = 1 in FP64 and at 40 digits), and A + c well above 1."""
    rng = np.random.default_rng(seed)
    bulk = rng.uniform(-2, 2, (2, 4))
    bulk[:, 2] -= 2
    bulk[:, 3] += rng.uniform(1, 6, 2)
    if model == 0:
        edges = [[0.4, -1.0, -699.5, 5.0],     # c -> 0 at the bound
                 [699.5, 0.5, -3.0, 2.0],      # q -> 1: (1 - q)^x = 0 from x = 2 on
                 [-699.5, -699.5, -40.0, 1.0],  # q, A -> 0, c -> 0
                 [0.3, -0.5, -2.0, 12.0],      # large delta
                 [0.2, 0.0, 0.0, 4.0],         # A = c = 1/2: D_z(z = 1) = 1 -> NaN
                 [-1.0, 3.0, 2.5, 3.0]]        # A + c > 1 -> NaN
    else:
        edges = [[-699.5, 3.0, 0, 0],           # q -> 0 at the bound
                 [0.3, 12.0, 0, 0],             # large delta
                 [3.0, -699.5, 0, 0]]           # delta -> 0 (phi = 2)
    return np.vstack([bulk, np.array(edges, np.float64)])


def model_grad_scale(k, N, u, model, mask):
    """Per component j: sum over the used positions of |psi| x |d(argument) / du_j| over the six digamma values of
    the analytic gradient (psi(k + a), psi(a), psi(N - k + b), psi(b), psi(N + phi), psi(phi), with a = D_z phi and
    b = (1 - D_z) phi). An FP64 evaluation of that gradient cancels these products, so eps times this sum bounds its
    rounding error; it matters at large delta, where d phi / d log delta = delta multiplies digamma values of ~log phi
    whose differences are ~N / phi."""
    from scipy.special import digamma

    P = len(k) // 2
    D = 4 if model == 0 else 2
    u = np.asarray(u, np.float64)
    sg = lambda x: 1.0 / (1.0 + np.exp(-x))  # noqa: E731
    q, delta = sg(u[0]), np.exp(u[D - 1])
    phi = delta + PHI_MIN
    out = np.zeros(D)
    for i in used_positions(P, mask):
        x = i if i < P else i - P
        kk, nn = float(k[i]), float(N[i])
        if model == 0:
            A, c = sg(u[1]), sg(u[2])
            w = (1.0 - q) ** x
            Dz = A * w + c
            dD = np.array([A * w * x * q, A * (1 - A) * w, c * (1 - c)])  # |dD_z / du_j| of the sigmoid lanes
        else:
            Dz = q
            dD = np.array([q * (1 - q)])
        a, b = Dz * phi, (1.0 - Dz) * phi
        pa = abs(digamma(kk + a)) + abs(digamma(a))
        pb = abs(digamma(nn - kk + b)) + abs(digamma(b))
        pp = abs(digamma(nn + phi)) + abs(digamma(phi))
        out[:D - 1] += (pa + pb) * phi * dD
        out[D - 1] += (pa * Dz + pb * (1.0 - Dz) + pp) * delta
    return out


def check_logp_grad_against_reference(k, N, u, model, mask, jac, logp, grad, tag):
    """logp within 1e-13 x (1 + sum of |terms|) of the 40-digit value; the gradient within 1e-12 relative
    (|g - g_ref| <= 1e-12 (1 + |g_ref|) per component) plus eps x model_grad_scale, FP64's own rounding of the
    digamma differences (it dominates only at the large-delta point); NaN in the same places."""
    D = 4 if model == 0 else 2
    for e in range(len(u)):
        ref = model_logp_mp(k, N, u[e], model, mask, jac)
        assert np.isnan(logp[e]) == bool(mp.isnan(ref)), (tag, e, u[e], logp[e], ref)
        if mp.isnan(ref):
            continue
        scale = model_logp_scale(k, N, u[e], model, mask, jac)
        assert abs(logp[e] - float(ref)) <= 1e-13 * (1 + scale), (tag, e, u[e], logp[e], float(ref), scale)
        g = model_grad_mp(k, N, u[e], model, mask, jac)
        tol = 1e-12 * (1 + np.abs(g)) + np.finfo(np.float64).eps * model_grad_scale(k, N, u[e], model, mask)
        err = np.abs(grad[e][:D] - g)
        assert np.all(err <= tol), (tag, e, u[e], grad[e][:D], g, err / tol)


def boundary_taxon(P, seed=77):
    """The highest-coverage of 50 synthetic TaxIDs at max_position P (dense k, N of 2P positions)."""
    g = syn.make_mismatch_matrix(50, max_position=P, seed=seed + P)
    t = int(np.argmax(g["tax_n_alignments"]))
    return g["k"][t], g["N"][t]


@pytest.mark.parametrize("P", MAX_POSITIONS)
def test_oracle_logp_grad_matches_mpmath(oracle, P):
    k, N = boundary_taxon(P)
    assert N.sum() > 0
    for model in (0, 1):
        u = reference_points(model, seed=P)
        for mask in (0, 1, 2):
            for jac in (True, False):
                logp, grad, _ = oracle.logp_grad(k, N, u, model=model, lane_mask=mask, with_jacobian=jac)
                check_logp_grad_against_reference(k, N, u, model, mask, jac, logp, grad, (P, model, mask, jac))


def test_oracle_logp_grad_matches_mpmath_high_coverage(oracle, sample_inputs):
    """N(z) ~ 1e7 (the reference's sample file, P = 15): the terms cancel over ~10 orders of magnitude."""
    s = sample_inputs["ancient"]
    r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
    t = int(np.argmax(r["N"].sum(axis=1)))
    k, N = r["k"][t], r["N"][t]
    assert N.max() > 1e6
    for model in (0, 1):
        u = reference_points(model, seed=15)
        for mask in (0, 1, 2):
            for jac in (True, False):
                logp, grad, _ = oracle.logp_grad(k, N, u, model=model, lane_mask=mask, with_jacobian=jac)
                check_logp_grad_against_reference(k, N, u, model, mask, jac, logp, grad, ("sample", model, mask, jac))


def test_reference_per_position_terms_sum_to_logp():
    """The per-position terms that test_gpu_max_position.py compares with the kernels' `ll` output add up, with the
    prior, to model_logp_mp."""
    k, N = boundary_taxon(16)
    u = reference_points(0, seed=1)[0]
    for mask in (0, 1, 2):
        ll = model_ll_mp(k, N, u, 0, mask)
        assert sorted(ll) == list(used_positions(16, mask))
        with mp.workdps(DPS):
            prior, _ = model_terms_mp(k, N, u, 0, mask, True)
            total = mp.fsum(prior) + sum(v for v, _ in ll.values())
            assert abs(total - model_logp_mp(k, N, u, 0, mask, True)) < 1e-9
