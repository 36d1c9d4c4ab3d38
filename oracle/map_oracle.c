/*
 * map_oracle.c — CPU restatement (plain C, FP64) of the MAP-only screening path, mdg_map_batch (K3m).
 * TEST INFRASTRUCTURE ONLY, like mdg_oracle.c: nothing in the product may import, link or call it.
 *
 * It is compiled as one translation unit with mdg_oracle.c, whose MAP fit (orc_map_fit), data layout
 * (fill_data, lane masks 0 / 1 / 2), log density (orc_logp_grad), transform (constrain), Cholesky
 * solve and noise (orc_noise) it uses unchanged: six fits per TaxID ({PMD, null} x {all, forward-only,
 * reverse-only positions}), the Laplace step, the likelihood-ratio tail and the per-TaxID row, in
 * the layout of mdg_map_result. The one field it does not restate is mdg_map_run.n_eval (0 here):
 * orc_map_fit does not count its gradient evaluations.
 */
#include "mdg_oracle.c"

/* ------------------------------------------------------------------------------------ */
/* K3m oracle — MAP-only screening (mdg_map_batch)                                        */
/* ------------------------------------------------------------------------------------ */

/* MAP fit of one run kind (orc_map_fit), log-likelihood at the mode and the Laplace covariance J H_u^-1 J
 * (see mdg_map_run in mdg.h for why no second-order term appears). n_eval is not counted here (0). */
static void map_laplace(const orc_data* d, mdg_map_run* out) {
    const int D = model_dim(d->model);
    double u[ORC_MAXD], lp, th[4];
    int conv;
    memset(out, 0, sizeof *out);
    int it = orc_map_fit(d, u, &lp, &conv);
    out->iters = (uint32_t)it;
    out->q_std = out->A_std = out->c_std = out->phi_std = out->cov_Ac = NAN;
    out->loglik = NAN;
    if (isnan(lp)) {
        out->q = out->A = out->c = out->phi = out->logp = NAN;
        out->flags = MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED | MDG_FIT_COV_INVALID;
        return;
    }
    constrain(d, u, th);
    out->q = th[0]; out->A = th[1]; out->c = th[2]; out->phi = th[3];
    out->logp = lp;
    double g[ORC_MAXD], ll[ORC_MAXOBS], t;
    orc_logp_grad(d, u, 0, &t, g, ll);
    double s = 0;
    for (int i = 0; i < d->n; ++i) s += ll[i];
    out->loglik = s;
    int cov_ok = conv;
    if (cov_ok) {
        double H[ORC_MAXD * ORC_MAXD], S[ORC_MAXD * ORC_MAXD];
        for (int j = 0; j < D; ++j) {
            double h = 1e-4 * (1.0 + fabs(u[j]));
            double up[ORC_MAXD], um[ORC_MAXD], gp[ORC_MAXD], gm[ORC_MAXD];
            memcpy(up, u, sizeof(double) * D); memcpy(um, u, sizeof(double) * D);
            up[j] += h; um[j] -= h;
            int okp = orc_logp_grad(d, up, 0, &t, gp, NULL);
            int okm = orc_logp_grad(d, um, 0, &t, gm, NULL);
            cov_ok = cov_ok && okp && okm;
            for (int i = 0; i < D; ++i) H[i * D + j] = -(gp[i] - gm[i]) / (2 * h);
        }
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < i; ++j) { double v = 0.5 * (H[i * D + j] + H[j * D + i]); H[i * D + j] = H[j * D + i] = v; }
        for (int col = 0; col < D; ++col) {
            double e[ORC_MAXD] = {0, 0, 0, 0}, x[ORC_MAXD] = {0, 0, 0, 0};
            e[col] = 1.0;
            cov_ok = chol_solve(D, H, e, x) && cov_ok;
            for (int i = 0; i < D; ++i) S[i * D + col] = x[i];
        }
        if (cov_ok) {
            double J[ORC_MAXD], var[ORC_MAXD];
            for (int j = 0; j < D - 1; ++j) { double v = th[d->model == 0 ? j : 0]; J[j] = v * (1.0 - v); }
            J[D - 1] = exp(u[D - 1]);
            for (int j = 0; j < D; ++j) var[j] = J[j] * S[j * D + j] * J[j];
            cov_ok = var[0] > 0 && var[D - 1] > 0;
            out->q_std = sqrt(var[0]);
            out->phi_std = sqrt(var[D - 1]);
            if (d->model == 0) {
                cov_ok = cov_ok && var[1] > 0 && var[2] > 0;
                out->A_std = sqrt(var[1]);
                out->c_std = sqrt(var[2]);
                out->cov_Ac = J[1] * S[1 * D + 2] * J[2];
            }
            if (!cov_ok) out->q_std = out->A_std = out->c_std = out->phi_std = out->cov_Ac = NAN;
        }
    }
    if (!conv) out->flags |= MDG_FIT_MAP_NOT_CONVERGED;
    if (!cov_ok) out->flags |= MDG_FIT_COV_INVALID;
}

/* exp(x^2) erfc(x) for x >= 0: erfc times exp of the exactly split square below 26, the asymptotic series above */
static double erfcx_pos(double x) {
    if (x < 26.0) {
        double hi = x * x, lo = fma(x, x, -hi);
        return erfc(x) * exp(hi) * exp(lo);
    }
    double t = 1.0 / (2.0 * x * x), term = 1.0, sum = 1.0;
    for (int n = 1; n < 12; ++n) { term *= -(2.0 * n - 1.0) * t; sum += term; }
    return sum / (x * 1.77245385090551602730);
}

/* w >= 0 with log Phi(-w) = L (L <= log 1/2): Newton from sqrt(-2 L), monotone (see the CUDA kernel) */
static double upper_tail_quantile(double L) {
    if (L == -INFINITY) return INFINITY;
    double w = sqrt(-2.0 * L);
    for (int it = 0; it < 100; ++it) {
        double e = erfcx_pos(w * 0.70710678118654752440);
        double g = log(0.5 * e) - 0.5 * w * w - L;
        double wn = fmax(w + g * e * 1.25331413731550025121, 0.0);
        int done = fabs(wn - w) <= 2e-16 * wn;
        w = wn;
        if (done || w == 0.0) break;
    }
    return w;
}

static void lr_tail(double lambda, double* P, double* z) {
    if (isnan(lambda)) { *P = *z = NAN; return; }
    double logP = -0.5 * fmax(lambda, 0.0);
    *P = exp(logP);
    if (logP < -0.69314718055994530942) *z = upper_tail_quantile(logP);
    else *z = -upper_tail_quantile(log(-expm1(logP)));
}

static double dmax_std(const mdg_map_run* r) { return sqrt(r->A_std * r->A_std + r->c_std * r->c_std + 2.0 * r->cov_Ac); }

void orc_map_one(int64_t tax_id, int P, const uint32_t* k, const uint32_t* N, const uint32_t* mism12,
                 const double* noise3, const mdg_fit_config* cfg, mdg_map_result* r) {
    const int R = 2 * P;
    memset(r, 0, sizeof *r);
    r->tax_id = tax_id;
    r->N_z1_forward = N[0]; r->N_z1_reverse = N[P];
    for (int s = 0; s < R; ++s) {
        if (s < P) { r->N_sum_forward += N[s]; r->y_sum_forward += k[s]; }
        else { r->N_sum_reverse += N[s]; r->y_sum_reverse += k[s]; }
    }
    r->N_sum_total = r->N_sum_forward + r->N_sum_reverse;
    r->y_sum_total = r->y_sum_forward + r->y_sum_reverse;
    r->normalized_noise = r->normalized_noise_forward = r->normalized_noise_reverse = NAN;
    if (mism12) {
        double nz[3]; orc_noise(P, mism12, nz);
        r->normalized_noise = nz[0]; r->normalized_noise_forward = nz[1]; r->normalized_noise_reverse = nz[2];
    } else if (noise3) {
        r->normalized_noise = noise3[0]; r->normalized_noise_forward = noise3[1]; r->normalized_noise_reverse = noise3[2];
    }
    const int n_runs = cfg->do_fwd_rev ? MDG_NUM_RUNS : 2;
    for (int i = 0; i < MDG_NUM_RUNS; ++i) {
        mdg_map_run* e = &r->run[i];
        if (i < n_runs) {
            orc_data d;
            fill_data(&d, i & 1, i / 2, P, k, N, cfg);
            map_laplace(&d, e);
        } else {
            e->q = e->A = e->c = e->phi = e->q_std = e->A_std = e->c_std = e->phi_std = e->cov_Ac = e->logp = e->loglik = NAN;
        }
    }
    const mdg_map_run *pmd = &r->run[0], *nul = &r->run[1];
    r->status = (pmd->flags | nul->flags) & (MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED | MDG_FIT_COV_INVALID);
    r->D_max = pmd->A + pmd->c;
    r->D_max_std = dmax_std(pmd);
    r->significance = r->D_max / r->D_max_std;
    r->rho_Ac = pmd->cov_Ac / (pmd->A_std * pmd->c_std);
    r->lambda_LR = 2.0 * (pmd->loglik - nul->loglik);
    lr_tail(r->lambda_LR, &r->lambda_LR_P, &r->lambda_LR_z);
    r->forward_D_max = r->run[2].A + r->run[2].c;
    r->forward_D_max_std = dmax_std(&r->run[2]);
    r->forward_lambda_LR = 2.0 * (r->run[2].loglik - r->run[3].loglik);
    r->reverse_D_max = r->run[4].A + r->run[4].c;
    r->reverse_D_max_std = dmax_std(&r->run[4]);
    r->reverse_lambda_LR = 2.0 * (r->run[4].loglik - r->run[5].loglik);
}

int orc_map_batch(int64_t n_tax, int max_position, const int64_t* tax_id, const uint32_t* k, const uint32_t* N,
                  const uint32_t* mism12, const double* noise3, const mdg_fit_config* cfg, mdg_map_result* out,
                  int n_threads) {
    const int P = max_position, R = 2 * P;
    if (P < 1 || P > MDG_MAX_POSITION) return MDG_ERR_INVALID;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#else
    (void)n_threads;
#endif
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t t = 0; t < n_tax; ++t)
        orc_map_one(tax_id[t], P, k + t * R, N + t * R, mism12 ? mism12 + t * R * 12 : NULL, noise3 ? noise3 + t * 3 : NULL,
                    cfg, out + t);
    return MDG_OK;
}

/* the likelihood-ratio tail of mdg_map_result for given lambda values */
int orc_test_lr_tail(int64_t n, const double* lambda, double* P, double* z) {
    for (int64_t i = 0; i < n; ++i) lr_tail(lambda[i], &P[i], &z[i]);
    return MDG_OK;
}
