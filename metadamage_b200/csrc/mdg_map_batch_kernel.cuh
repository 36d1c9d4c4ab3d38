// mdg_map_batch_kernel.cuh — K3m: the MAP-only screening path (mdg_map_batch). Six MAP fits per TaxID ({PMD, null} x
// {all positions, forward only, reverse only}) through map_fit_group (K3, the same code map_kernel runs), a Laplace
// covariance at each mode, then one row per TaxID with A + c, its standard deviation and the likelihood-ratio
// statistic. No random numbers, no NUTS scratch.
#pragma once
#include "mdg_post_kernels.cuh"

namespace mdg {

struct MapBatchLaunch {
    const uint32_t* k;
    const uint32_t* N;
    int n_tax, P;
    int n_runs;  // 6, or 2 without the forward-only / reverse-only fits
    Priors pr;
    unsigned int* work_counter;
    mdg_map_run* rec;  // [n_tax][MDG_NUM_RUNS]
};

// One run: MAP fit, log-likelihood at the mode, Laplace covariance.
//
// Laplace step. f(u) = -log p(theta(u)) carries no Jacobian term, so grad_u f = J grad_theta f with
// J = diag(d theta_j / d u_j), and the Hessian in u is H_u = J H_theta J + diag(d^2 theta_j / d u_j^2 * df/dtheta_j).
// At a stationary point df/dtheta = 0, the second term vanishes, and J H_u^-1 J = H_theta^-1 exactly: the covariance
// of theta is obtained from the Hessian in u without differentiating in theta, where the mode may sit close to a
// bound. H_u is the central difference of the analytic gradient with the Newton loop's step rule, symmetrised;
// H_u^-1 comes column by column from chol_solve, which also tells whether H_u is positive definite.
template <int MODEL, int NPL>
__device__ void map_laplace_group(const LaneObs<NPL>& ob, const double (&logC)[NPL], int P, const Priors& pr,
                                  const double2* ptab, bool has_spare, int lig, mdg_map_run& out) {
    constexpr int D = ModelDim<MODEL>::value;
    constexpr unsigned gmask = 0xffffffffu;
    const double qnan = nan("");
    MapRecord m;
    MapTrace tr;
    map_fit_group<MODEL, NPL, true>(ob, logC, P, pr, ptab, has_spare, lig, m, &tr);
    out.q = m.theta[0]; out.A = m.theta[1]; out.c = m.theta[2]; out.phi = m.theta[3];
    out.q_std = out.A_std = out.c_std = out.phi_std = out.cov_Ac = qnan;
    out.logp = m.logp;
    out.loglik = qnan;
    out.iters = m.iters;
    out.reserved = 0u;
    uint32_t n_eval = tr.n_eval;
    if (isnan(m.theta[0])) {  // no finite starting point
        out.n_eval = n_eval;
        out.flags = MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED | MDG_FIT_COV_INVALID;
        return;
    }
    double u[D], g[D], ll[NPL], lp;
    bool ok;
#pragma unroll
    for (int j = 0; j < D; ++j) u[j] = tr.u[j];
    eval_model<MODEL, NPL, 32>(ob, u, ptab, pr.phi_min, has_spare, gmask, lig, lp, g, ll, ok);
    ++n_eval;
    double s_ll = 0.0;
#pragma unroll
    for (int s = 0; s < NPL; ++s) s_ll += ob.act[s] ? ll[s] + logC[s] : 0.0;
    out.loglik = group_sum<32>(s_ll, gmask);
    bool cov_ok = m.converged != 0u;
    if (cov_ok) {
        double H[D][D];
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const double h = 1e-4 * (1.0 + fabs(u[j]));
            double up[D], um[D], gp[D], gm[D], t0, t1;
            bool okp, okm;
#pragma unroll
            for (int i = 0; i < D; ++i) { up[i] = u[i] + (i == j ? h : 0.0); um[i] = u[i] - (i == j ? h : 0.0); }
            eval_model<MODEL, NPL, 32>(ob, up, ptab, pr.phi_min, has_spare, gmask, lig, t0, gp, ll, okp);
            eval_model<MODEL, NPL, 32>(ob, um, ptab, pr.phi_min, has_spare, gmask, lig, t1, gm, ll, okm);
            n_eval += 2;
            cov_ok = cov_ok && okp && okm;
#pragma unroll
            for (int i = 0; i < D; ++i) H[i][j] = -(gp[i] - gm[i]) / (2.0 * h);
        }
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) { double s = 0.5 * (H[i][j] + H[j][i]); H[i][j] = s; H[j][i] = s; }
        double S[D][D];
#pragma unroll
        for (int col = 0; col < D; ++col) {
            double e[D], x[D];
#pragma unroll
            for (int i = 0; i < D; ++i) { e[i] = (i == col) ? 1.0 : 0.0; x[i] = 0.0; }
            cov_ok = chol_solve<D>(H, e, x) && cov_ok;
#pragma unroll
            for (int i = 0; i < D; ++i) S[i][col] = x[i];
        }
        if (cov_ok) {
            double J[D];
#pragma unroll
            for (int j = 0; j < D - 1; ++j) J[j] = m.theta[MODEL == 0 ? j : 0] * (1.0 - m.theta[MODEL == 0 ? j : 0]);
            J[D - 1] = exp(u[D - 1]);
            double var[D];
#pragma unroll
            for (int j = 0; j < D; ++j) var[j] = J[j] * S[j][j] * J[j];
            cov_ok = var[0] > 0.0 && var[D - 1] > 0.0;
            out.q_std = sqrt(var[0]);
            out.phi_std = sqrt(var[D - 1]);
            if (MODEL == 0) {
                cov_ok = cov_ok && var[1] > 0.0 && var[2] > 0.0;
                out.A_std = sqrt(var[1]);
                out.c_std = sqrt(var[2]);
                out.cov_Ac = J[1] * S[1][2] * J[2];
            }
            if (!cov_ok) out.q_std = out.A_std = out.c_std = out.phi_std = out.cov_Ac = qnan;
        }
    }
    uint32_t flags = 0u;
    if (!m.converged) flags |= MDG_FIT_MAP_NOT_CONVERGED;
    if (!cov_ok) flags |= MDG_FIT_COV_INVALID;
    out.flags = flags;
    out.n_eval = n_eval;
}

// One warp per (TaxID, run kind) item on a persistent grid, like map_kernel. The all-position runs use map_kernel's
// lane layout (NPL positions per lane for all 2P positions, the same spare-slot rule), so their fits are the same
// operations on the same values as mdg_fit_batch's.
template <int NPL, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, MDG_MAP_MINBLOCKS) map_batch_kernel(const MapBatchLaunch p) {
    __shared__ unsigned int sh_item[WARPS];
    __shared__ double2 sh_prior[2][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    log_table_init();
    prior_table_init<0>(sh_prior[0], p.pr, 0);
    prior_table_init<1>(sh_prior[1], p.pr, 0);
    const unsigned total = (unsigned)p.n_tax * (unsigned)p.n_runs;
    for (;;) {
        if (lane == 0) sh_item[warp] = atomicAdd(p.work_counter, 1u);
        __syncwarp();
        const unsigned item = sh_item[warp];
        __syncwarp();
        if (item >= total) break;
        const int tax = (int)(item / (unsigned)p.n_runs), run = (int)(item % (unsigned)p.n_runs);
        const int model = run & 1, mask = run >> 1;
        LaneObs<NPL> ob;
        load_obs<NPL, 32>(ob, p.k + (size_t)tax * 2 * p.P, p.N + (size_t)tax * 2 * p.P, p.P, mask, lane);
        double logC[NPL];
        log_binom_coeff<NPL>(ob, logC);
        const int n_obs = mask == 0 ? 2 * p.P : p.P;
        const bool has_spare = n_obs < NPL * 32;
        mdg_map_run rec;
        if (model == 0) map_laplace_group<0, NPL>(ob, logC, p.P, p.pr, sh_prior[0], has_spare, lane, rec);
        else map_laplace_group<1, NPL>(ob, logC, p.P, p.pr, sh_prior[1], has_spare, lane, rec);
        if (lane == 0) p.rec[(size_t)tax * MDG_NUM_RUNS + run] = rec;
    }
}

// ---------------------------------------------------------------------------------------------
// likelihood-ratio tail: P = exp(-max(lambda, 0) / 2) and z = -Phi^-1(P), from log P so that z stays finite where P
// underflows (lambda > ~1490)
// ---------------------------------------------------------------------------------------------

// w >= 0 with log Phi(-w) = L, for L <= log(1/2). Newton on g(w) = log Phi(-w) - L with
// log Phi(-w) = log(erfcx(w / sqrt 2) / 2) - w^2 / 2 and g'(w) = -sqrt(2 / pi) / erfcx(w / sqrt 2). g is concave and
// decreasing and the start sqrt(-2 L) lies right of the root (Phi(-w) < exp(-w^2 / 2) / 2), so the iterates decrease
// monotonically to it.
__device__ inline double upper_tail_quantile(double L) {
    if (L == -INFINITY) return INFINITY;
    double w = sqrt(-2.0 * L);
    for (int it = 0; it < 100; ++it) {
        const double e = erfcx(w * 0.70710678118654752440);
        const double g = log(0.5 * e) - 0.5 * w * w - L;
        const double dw = g * e * 1.25331413731550025121;  // sqrt(pi / 2)
        const double wn = fmax(w + dw, 0.0);
        const bool done = fabs(wn - w) <= 2e-16 * wn;
        w = wn;
        if (done || w == 0.0) break;
    }
    return w;
}

__device__ inline void lr_tail(double lambda, double& P, double& z) {
    if (isnan(lambda)) { P = z = nan(""); return; }
    const double logP = -0.5 * fmax(lambda, 0.0);
    P = exp(logP);
    if (logP < -0.69314718055994530942) z = upper_tail_quantile(logP);  // P < 1/2: z > 0
    else z = -upper_tail_quantile(log(-expm1(logP)));                   // 1 - P <= 1/2, from expm1
}

// ---------------------------------------------------------------------------------------------
// assembly: one thread per TaxID
// ---------------------------------------------------------------------------------------------
struct MapAssembleLaunch {
    const int64_t* tax_id;
    const uint32_t* k;
    const uint32_t* N;
    const uint32_t* mism12;  // optional
    const double* noise3;    // optional
    int n_tax, P, n_runs;
    const mdg_map_run* rec;  // [n_tax][MDG_NUM_RUNS]
    mdg_map_result* out;
    unsigned long long* eval_totals;  // [MDG_NUM_RUNS]
};

__device__ __forceinline__ double map_dmax_std(const mdg_map_run& r) {
    return sqrt(r.A_std * r.A_std + r.c_std * r.c_std + 2.0 * r.cov_Ac);
}

__global__ void map_assemble_kernel(const MapAssembleLaunch p) {
    const int tax = blockIdx.x * blockDim.x + threadIdx.x;
    if (tax >= p.n_tax) return;
    const int P = p.P, R = 2 * P;
    const mdg_map_run* rr = p.rec + (size_t)tax * MDG_NUM_RUNS;
    const double qnan = nan("");
    mdg_map_result r;
    memset(&r, 0, sizeof r);
    r.tax_id = p.tax_id[tax];
    tax_sums(p.k + (size_t)tax * R, p.N + (size_t)tax * R, P, r);
    r.normalized_noise = r.normalized_noise_forward = r.normalized_noise_reverse = qnan;
    tax_noise(p.mism12, p.noise3, tax, P, r);
    for (int i = 0; i < MDG_NUM_RUNS; ++i) {
        if (i < p.n_runs) {
            r.run[i] = rr[i];
            atomicAdd(&p.eval_totals[i], (unsigned long long)rr[i].n_eval);
        } else {
            mdg_map_run& e = r.run[i];
            e.q = e.A = e.c = e.phi = e.q_std = e.A_std = e.c_std = e.phi_std = e.cov_Ac = e.logp = e.loglik = qnan;
        }
    }
    const mdg_map_run &pmd = r.run[MDG_RUN_PMD_ALL], &nul = r.run[MDG_RUN_NULL_ALL];
    r.status = (pmd.flags | nul.flags) & (MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED | MDG_FIT_COV_INVALID);
    r.D_max = pmd.A + pmd.c;
    r.D_max_std = map_dmax_std(pmd);
    r.significance = r.D_max / r.D_max_std;
    r.rho_Ac = pmd.cov_Ac / (pmd.A_std * pmd.c_std);
    r.lambda_LR = 2.0 * (pmd.loglik - nul.loglik);
    lr_tail(r.lambda_LR, r.lambda_LR_P, r.lambda_LR_z);
    const mdg_map_run &pf = r.run[MDG_RUN_PMD_FWD], &nf = r.run[MDG_RUN_NULL_FWD];
    const mdg_map_run &pv = r.run[MDG_RUN_PMD_REV], &nv = r.run[MDG_RUN_NULL_REV];
    r.forward_D_max = pf.A + pf.c;
    r.forward_D_max_std = map_dmax_std(pf);
    r.forward_lambda_LR = 2.0 * (pf.loglik - nf.loglik);
    r.reverse_D_max = pv.A + pv.c;
    r.reverse_D_max_std = map_dmax_std(pv);
    r.reverse_lambda_LR = 2.0 * (pv.loglik - nv.loglik);
    p.out[tax] = r;
}

}  // namespace mdg
