/*
 * map_profile_oracle.c — CPU restatement (plain C, FP64) of the profile intervals of D_max, mdg_map_profile (K3p).
 * Test infrastructure only: compiled as one translation unit with oracle/map_oracle.c (and through it
 * oracle/mdg_oracle.c), whose data layout (fill_data), log density (orc_logp_grad), Cholesky solve (chol_solve) and
 * normal quantile (upper_tail_quantile) it uses unchanged. The algorithm is that of mdg_map_profile_kernel.cuh
 * step for step; see there and mdg.h for the definitions.
 */
#include "../oracle/map_oracle.c"

#define PROF_UMAX 40.0
#define PROF_WIDTH_TOL 1e-9
#define PROF_ROOT_TOL 1e-7
#define PROF_MAX_OUTER 100

static double prof_threshold(double level) {
    double w = upper_tail_quantile(log(0.5 * (1.0 - level)));
    return w * w;
}

/* log p (incl. log C(N,k)) and its gradient in v = (logit q, logit s, log(phi - phi_min)) on A + c = D */
static int prof_eval(const orc_data* d, double D, const double* v, double* lp, double* g) {
    double s = 1.0 / (1.0 + exp(-v[1])), s1 = 1.0 / (1.0 + exp(v[1]));
    double A = D * s, c = D * s1;
    double u[4] = {v[0], log(A) - log1p(-A), log(c) - log1p(-c), v[2]}, g4[4];
    int ok = orc_logp_grad(d, u, 0, lp, g4, NULL);
    g[0] = g4[0];
    g[1] = g4[1] * (s1 / (1.0 - A)) - g4[2] * (s / (1.0 - c));
    g[2] = g4[3];
    return ok && isfinite(g[1]);
}

/* maximiser of log p on A + c = D from v (map_fit_group's rules); 1 if converged */
static int prof_fit(const orc_data* d, double slack, double D, double* v, double* logp, uint32_t* n_eval) {
    double f, g[3], lp;
    int ok = prof_eval(d, D, v, &lp, g);
    ++*n_eval;
    if (!ok) return 0;
    f = -lp;
    for (int j = 0; j < 3; ++j) g[j] = -g[j];
    double lambda = 1e-3;
    int converged = 0;
    for (int it = 0; it < 200; ++it) {
        double H[9];
        for (int j = 0; j < 3; ++j) {
            double h = 1e-4 * (1.0 + fabs(v[j]));
            double vp[3], vm[3], gp[3], gm[3], t;
            memcpy(vp, v, sizeof vp); memcpy(vm, v, sizeof vm);
            vp[j] += h; vm[j] -= h;
            int okp = prof_eval(d, D, vp, &t, gp);
            int okm = prof_eval(d, D, vm, &t, gm);
            *n_eval += 2;
            for (int i = 0; i < 3; ++i) H[i * 3 + j] = (okp && okm) ? -(gp[i] - gm[i]) / (2 * h) : (i == j ? 1.0 : 0.0);
        }
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < i; ++j) { double s = 0.5 * (H[i * 3 + j] + H[j * 3 + i]); H[i * 3 + j] = H[j * 3 + i] = s; }
        int accepted = 0;
        for (int tries = 0; tries < 40 && !accepted; ++tries) {
            double Hd[9], rhs[3], dv[3];
            memcpy(Hd, H, sizeof Hd);
            for (int i = 0; i < 3; ++i) { Hd[i * 3 + i] += lambda * (fabs(H[i * 3 + i]) + 1e-8); rhs[i] = -g[i]; }
            if (!chol_solve(3, Hd, rhs, dv)) { lambda *= 10; continue; }
            double vn[3], gn[3], lpn, dmax = 0;
            for (int i = 0; i < 3; ++i) {
                vn[i] = fmin(fmax(v[i] + dv[i], -PROF_UMAX), PROF_UMAX);
                dmax = fmax(dmax, fabs(vn[i] - v[i]));
            }
            int okn = prof_eval(d, D, vn, &lpn, gn);
            ++*n_eval;
            if (okn && -lpn <= f + slack) {
                double gmax = 0;
                for (int i = 0; i < 3; ++i) { v[i] = vn[i]; g[i] = -gn[i]; gmax = fmax(gmax, fabs(gn[i])); }
                f = -lpn;
                lambda = fmax(lambda / 3.0, 1e-12);
                accepted = 1;
                if (dmax < 1e-10 || gmax < 1e-9) converged = 1;
            } else {
                lambda *= 4;
                if (dmax < 1e-13) { converged = 1; accepted = 1; }
            }
        }
        if (!accepted || converged) break;
    }
    *logp = -f;
    return converged;
}

/* pl(D): the best of three inner fits, from v (the nearest point solved), from the mode and from v with s = 1/2. One
 * start can stop on a branch that is not the maximum on A + c = D (the likelihood is multimodal in q at low coverage)
 * or on the flat end of the sigmoid in s (c -> 0 or A -> 0, where the gradient in logit s vanishes). */
static int prof_fit_best(const orc_data* d, double slack, double D, double* v, const double* vmode, double* logp,
                         uint32_t* n_eval) {
    double best[3], lbest = -INFINITY;
    int any = 0;
    for (int k = 0; k < 3; ++k) {
        double w[3], lp;
        memcpy(w, k == 1 ? vmode : v, sizeof w);
        if (k == 2) w[1] = 0.0;
        if (prof_fit(d, slack, D, w, &lp, n_eval) && lp > lbest) { lbest = lp; memcpy(best, w, sizeof best); any = 1; }
    }
    if (any) { memcpy(v, best, sizeof best); *logp = lbest; }
    return any;
}

static void prof_end(const orc_data* d, double slack, const mdg_map_run* rec, double t, int side, mdg_profile_end* out) {
    const double phi_min = d->cfg->phi_min;
    out->D = out->q = out->A = out->c = out->phi = out->logp = NAN;
    const double Dhat = rec->A + rec->c, lphat = rec->logp;
    const double bound = side ? 1.0 : 0.0, sgn = side ? 1.0 : -1.0;
    const double sd = dmax_std(rec);
    double va[3], vb[3], vx[3];
    va[0] = log(rec->q) - log1p(-rec->q);
    va[1] = log(rec->A) - log(rec->c);
    va[2] = log(rec->phi - phi_min);
    double vmode[3] = {va[0], va[1], va[2]};
    double a = Dhat, ha = -t, b = bound, hb = 0.0;
    double x = Dhat + sgn * 2.0 * sd;
    if (!(sgn * (x - Dhat) > 0.0 && sgn * (bound - x) > 0.0)) x = 0.5 * (Dhat + bound);
    double lpx = NAN;
    uint32_t flags = 0, n_eval = 0;
    int n_fit = 0, have_b = 0, done = 0;
    while (!have_b) {
        memcpy(vx, va, sizeof vx);
        if (++n_fit > PROF_MAX_OUTER || !prof_fit_best(d, slack, x, vx, vmode, &lpx, &n_eval)) { flags = MDG_PROFILE_FAILED; break; }
        double hx = 2.0 * (lphat - lpx) - t;
        if (hx > 0.0) {
            b = x; hb = hx; have_b = 1;
            memcpy(vb, vx, sizeof vb);
            done = fabs(hx) <= PROF_ROOT_TOL;
        } else {
            a = x; ha = hx;
            memcpy(va, vx, sizeof va);
            if (fabs(hx) <= PROF_ROOT_TOL) { done = 1; break; }
            if (fabs(bound - x) <= PROF_WIDTH_TOL) { flags = MDG_PROFILE_AT_BOUND; break; }
            double xn = x + sgn * fabs(x - Dhat);
            if (!(sgn * (bound - xn) > 0.5 * fabs(bound - x))) xn = 0.5 * (x + bound);
            x = xn;
        }
    }
    int kept = 0;
    while (have_b && !done && flags == 0) {
        if (fabs(b - a) <= PROF_WIDTH_TOL) break;
        double xn = a - ha * (b - a) / (hb - ha);
        double lo = fmin(a, b), hi = fmax(a, b);
        if (!(xn > lo && xn < hi)) xn = 0.5 * (a + b);
        x = xn;
        memcpy(vx, fabs(x - a) <= fabs(b - x) ? va : vb, sizeof vx);
        if (++n_fit > PROF_MAX_OUTER || !prof_fit_best(d, slack, x, vx, vmode, &lpx, &n_eval)) { flags = MDG_PROFILE_FAILED; break; }
        double hx = 2.0 * (lphat - lpx) - t;
        if (fabs(hx) <= PROF_ROOT_TOL) break;
        if (hx > 0.0) {
            b = x; hb = hx; memcpy(vb, vx, sizeof vb);
            if (kept == 1) ha *= 0.5;
            kept = 1;
        } else {
            a = x; ha = hx; memcpy(va, vx, sizeof va);
            if (kept == -1) hb *= 0.5;
            kept = -1;
        }
    }
    out->n_eval = n_eval;
    out->flags = flags;
    if (flags & MDG_PROFILE_FAILED) return;
    out->D = (flags & MDG_PROFILE_AT_BOUND) ? bound : x;
    out->q = 1.0 / (1.0 + exp(-vx[0]));
    out->A = x / (1.0 + exp(-vx[1]));
    out->c = x / (1.0 + exp(vx[1]));
    out->phi = exp(vx[2]) + phi_min;
    out->logp = lpx;
}

static void prof_nan(mdg_profile_end* e, uint32_t flags) {
    e->D = e->q = e->A = e->c = e->phi = e->logp = NAN;
    e->n_eval = 0;
    e->flags = flags;
}

void orc_map_profile_one(int P, const uint32_t* k, const uint32_t* N, const mdg_fit_config* cfg, const mdg_map_result* map,
                         double level, mdg_map_interval* r) {
    memset(r, 0, sizeof *r);
    r->tax_id = map->tax_id;
    r->level = level;
    r->threshold = prof_threshold(level);
    const int n_prof = cfg->do_fwd_rev ? 3 : 1;
    for (int prof = 0; prof < 3; ++prof) {
        const mdg_map_run* rec = &map->run[2 * prof];
        for (int side = 0; side < 2; ++side) {
            mdg_profile_end* e = &r->end[prof][side];
            if (prof >= n_prof || (rec->n_eval == 0 && isnan(rec->logp))) { prof_nan(e, 0); continue; }
            if (rec->flags & (MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED)) { prof_nan(e, MDG_FIT_FAILED); continue; }
            orc_data d;
            fill_data(&d, 0, prof, P, k, N, cfg);
            double scale = 0;
            for (int i = 0; i < d.n; ++i) scale += orc_lgamma(d.N[i] + 1.0);
            prof_end(&d, 1e-14 * scale + 1e-10, rec, r->threshold, side, e);
        }
    }
    r->status = r->end[0][0].flags | r->end[0][1].flags;
}

int orc_map_profile(int64_t n_tax, int max_position, const uint32_t* k, const uint32_t* N, const mdg_fit_config* cfg,
                    const mdg_map_result* map, double level, mdg_map_interval* out, int n_threads) {
    const int P = max_position, R = 2 * P;
    if (P < 1 || P > MDG_MAX_POSITION || !(level > 0.0 && level < 1.0)) return MDG_ERR_INVALID;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#else
    (void)n_threads;
#endif
#pragma omp parallel for schedule(dynamic, 4)
    for (int64_t t = 0; t < n_tax; ++t) orc_map_profile_one(P, k + t * R, N + t * R, cfg, map + t, level, out + t);
    return MDG_OK;
}


