// mdg_map_profile_kernel.cuh — K3p: profile intervals of D_max = A + c for the rows of the MAP-only path
// (mdg_map_profile). One warp per (TaxID, PMD run, side) item: a root search over D whose every trial is a
// constrained re-fit of the PMD model on A + c = D. It reuses eval_model, load_obs, chol_solve and
// upper_tail_quantile as they are and leaves map_fit_group and the K3m kernels untouched.
#pragma once
#include "mdg_map_batch_kernel.cuh"

namespace mdg {

struct MapProfileLaunch {
    const uint32_t* k;
    const uint32_t* N;
    const mdg_map_result* map;  // [n_tax] rows of mdg_map_batch
    int n_tax, P;
    int n_prof;  // PMD runs profiled per TaxID: 3, or 1 without the forward-only / reverse-only fits
    Priors pr;
    double level;
    unsigned int* work_counter;
    unsigned long long* eval_totals;  // [MDG_NUM_RUNS]
    mdg_map_interval* out;
};

constexpr double kProfUmax = 40.0;        // |v_j| bound of the inner fits (map_fit_group's UMAX)
constexpr double kProfWidthTol = 1e-9;    // bracket width at which a root search stops
constexpr double kProfRootTol = 1e-7;     // |h| at which a root search stops
constexpr int kProfMaxOuter = 100;        // inner fits per end

// t = chi-square(1) quantile at alpha = (Phi^-1((1 + alpha) / 2))^2, from the upper tail log((1 - alpha) / 2)
__device__ __forceinline__ double profile_threshold(double level) {
    const double w = upper_tail_quantile(log(0.5 * (1.0 - level)));
    return w * w;
}

// (q, A, c, phi) of v = (logit q, logit s, log(phi - phi_min)) on A + c = D, A = D s, c = D (1 - s)
__device__ __forceinline__ void profile_theta(double D, const double (&v)[3], double phi_min, double (&th)[4]) {
    th[0] = 1.0 / (1.0 + exp(-v[0]));
    th[1] = D / (1.0 + exp(-v[1]));
    th[2] = D / (1.0 + exp(v[1]));
    th[3] = exp(v[2]) + phi_min;
}

// log p (without log C(N,k)) and its gradient in v at fixed D. eval_model takes u = (u_q, logit A, logit c, u_delta);
// with s = sigmoid(v_1), dA/dv_1 = D s (1 - s) = -dc/dv_1 and dA/du_A = A (1 - A), so
//   d/dv_1 = D s (1 - s) (g_A / (A (1 - A)) - g_c / (c (1 - c))) = g_A (1 - s) / (1 - A) - g_c s / (1 - c).
template <int NPL>
__device__ __forceinline__ void profile_eval(const LaneObs<NPL>& ob, double D, const double (&v)[3], const double2* ptab,
                                             double phi_min, bool has_spare, int lig, double& lp, double (&g)[3], bool& ok) {
    const double s = 1.0 / (1.0 + exp(-v[1])), s1 = 1.0 / (1.0 + exp(v[1]));
    const double A = D * s, c = D * s1;
    double u[4], g4[4], ll[NPL];
    u[0] = v[0];
    u[1] = log(A) - log1p(-A);
    u[2] = log(c) - log1p(-c);
    u[3] = v[2];
    eval_model<0, NPL, 32>(ob, u, ptab, phi_min, has_spare, 0xffffffffu, lig, lp, g4, ll, ok);
    g[0] = g4[0];
    g[1] = g4[1] * (s1 / (1.0 - A)) - g4[2] * (s / (1.0 - c));
    g[2] = g4[3];
    ok = ok && isfinite(g[1]);
}

// Maximiser of log p on A + c = D from v: LM-damped Newton with a central-difference Hessian of the 3-gradient, the
// step, acceptance, slack and convergence rules of map_fit_group. On return v is the maximiser and logp = pl(D)
// (with log C(N,k)); false if the start is not finite or the fit did not converge.
template <int NPL>
__device__ bool profile_fit(const LaneObs<NPL>& ob, double sumC, double slack, double D, const double2* ptab, double phi_min,
                            bool has_spare, int lig, double (&v)[3], double& logp, uint32_t& n_eval) {
    constexpr int D3 = 3;
    double lp, g[D3];
    bool ok;
    profile_eval<NPL>(ob, D, v, ptab, phi_min, has_spare, lig, lp, g, ok);
    ++n_eval;
    if (!ok) return false;
    double f = -(lp + sumC);
#pragma unroll
    for (int j = 0; j < D3; ++j) g[j] = -g[j];
    double lambda = 1e-3;
    bool converged = false;
    for (int it = 0; it < 200; ++it) {
        double H[D3][D3];
#pragma unroll
        for (int j = 0; j < D3; ++j) {
            const double h = 1e-4 * (1.0 + fabs(v[j]));
            double vp[D3], vm[D3], gp[D3], gm[D3], t0, t1;
            bool okp, okm;
#pragma unroll
            for (int i = 0; i < D3; ++i) { vp[i] = v[i] + (i == j ? h : 0.0); vm[i] = v[i] - (i == j ? h : 0.0); }
            profile_eval<NPL>(ob, D, vp, ptab, phi_min, has_spare, lig, t0, gp, okp);
            profile_eval<NPL>(ob, D, vm, ptab, phi_min, has_spare, lig, t1, gm, okm);
            n_eval += 2;
#pragma unroll
            for (int i = 0; i < D3; ++i) H[i][j] = (okp && okm) ? -(gp[i] - gm[i]) / (2.0 * h) : (i == j ? 1.0 : 0.0);
        }
#pragma unroll
        for (int i = 0; i < D3; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) { double s = 0.5 * (H[i][j] + H[j][i]); H[i][j] = s; H[j][i] = s; }
        bool accepted = false;
        for (int tries = 0; tries < 40 && !accepted; ++tries) {
            double Hd[D3][D3], rhs[D3], dv[D3];
#pragma unroll
            for (int i = 0; i < D3; ++i) {
#pragma unroll
                for (int j = 0; j < D3; ++j) Hd[i][j] = H[i][j];
                Hd[i][i] += lambda * (fabs(H[i][i]) + 1e-8);
                rhs[i] = -g[i];
            }
            if (!chol_solve<D3>(Hd, rhs, dv)) { lambda *= 10.0; continue; }
            double vn[D3], gn[D3], lpn, dmax = 0.0;
#pragma unroll
            for (int i = 0; i < D3; ++i) {
                vn[i] = fmin(fmax(v[i] + dv[i], -kProfUmax), kProfUmax);
                dmax = fmax(dmax, fabs(vn[i] - v[i]));
            }
            bool okn;
            profile_eval<NPL>(ob, D, vn, ptab, phi_min, has_spare, lig, lpn, gn, okn);
            ++n_eval;
            if (okn && -(lpn + sumC) <= f + slack) {
                double gmax = 0.0;
#pragma unroll
                for (int i = 0; i < D3; ++i) { v[i] = vn[i]; g[i] = -gn[i]; gmax = fmax(gmax, fabs(gn[i])); }
                f = -(lpn + sumC);
                lambda = fmax(lambda / 3.0, 1e-12);
                accepted = true;
                if (dmax < 1e-10 || gmax < 1e-9) converged = true;
            } else {
                lambda *= 4.0;
                if (dmax < 1e-13) { converged = true; accepted = true; }
            }
        }
        if (!accepted || converged) break;
    }
    logp = -f;
    return converged;
}

// pl(D): the best of three inner fits, from v (the nearest point solved), from the mode and from v with s = 1/2. One
// start can stop on a branch that is not the maximum on A + c = D (the likelihood is multimodal in q at low coverage)
// or on the flat end of the sigmoid in s (c -> 0 or A -> 0, where the gradient in logit s vanishes).
template <int NPL>
__device__ bool profile_fit_best(const LaneObs<NPL>& ob, double sumC, double slack, double D, const double2* ptab,
                                 double phi_min, bool has_spare, int lig, double (&v)[3], const double (&vmode)[3],
                                 double& logp, uint32_t& n_eval) {
    double best[3], lbest = -INFINITY;
    bool any = false;
    for (int k = 0; k < 3; ++k) {
        double w[3], lp;
#pragma unroll
        for (int j = 0; j < 3; ++j) w[j] = (k == 1) ? vmode[j] : v[j];
        if (k == 2) w[1] = 0.0;
        if (profile_fit<NPL>(ob, sumC, slack, D, ptab, phi_min, has_spare, lig, w, lp, n_eval) && lp > lbest) {
            lbest = lp;
#pragma unroll
            for (int j = 0; j < 3; ++j) best[j] = w[j];
            any = true;
        }
    }
    if (any) {
#pragma unroll
        for (int j = 0; j < 3; ++j) v[j] = best[j];
        logp = lbest;
    }
    return any;
}

// One end of one run's interval: side 0 lower (towards D = 0), 1 upper (towards D = 1). h(D) = 2 (logp^ - pl(D)) - t
// is -t at the mode. Bracketing: the first trial is D^ +- 2 sd (D^ +- half the way to the bound where that leaves
// (0, 1) or sd is NaN); while h <= 0 the trial becomes the inner end of the bracket and the next trial doubles the
// distance from D^, or halves the distance to the bound where doubling would reach it. No crossing within 1e-9 of the
// bound: the end is the bound (MDG_PROFILE_AT_BOUND). Then the Illinois method on [inner, outer]. Every inner fit
// starts from the solution at the nearest point solved so far, which is always one end of the bracket (profile_fit_best).
template <int NPL>
__device__ void profile_end(const LaneObs<NPL>& ob, double sumC, double slack, const mdg_map_run& rec, double t, int side,
                            const double2* ptab, double phi_min, bool has_spare, int lig, mdg_profile_end& out) {
    const double qnan = nan("");
    out.D = out.q = out.A = out.c = out.phi = out.logp = qnan;
    out.n_eval = 0u;
    const double Dhat = rec.A + rec.c, lphat = rec.logp;
    const double bound = side ? 1.0 : 0.0, sgn = side ? 1.0 : -1.0;
    const double sd = map_dmax_std(rec);
    // bracket: a = inner end (h <= 0), b = outer end (h > 0)
    double va[3], vb[3], vx[3];
    va[0] = log(rec.q) - log1p(-rec.q);
    va[1] = log(rec.A) - log(rec.c);
    va[2] = log(rec.phi - phi_min);
    const double vmode[3] = {va[0], va[1], va[2]};
    double a = Dhat, ha = -t, b = bound, hb = 0.0;
    double x = Dhat + sgn * 2.0 * sd;
    if (!(sgn * (x - Dhat) > 0.0 && sgn * (bound - x) > 0.0)) x = 0.5 * (Dhat + bound);
    double lpx = qnan;
    uint32_t flags = 0u, n_eval = 0u;
    int n_fit = 0;
    bool have_b = false, done = false;
    // expansion
    while (!have_b) {
#pragma unroll
        for (int j = 0; j < 3; ++j) vx[j] = va[j];
        if (++n_fit > kProfMaxOuter || !profile_fit_best<NPL>(ob, sumC, slack, x, ptab, phi_min, has_spare, lig, vx, vmode, lpx, n_eval)) {
            flags = MDG_PROFILE_FAILED;
            break;
        }
        const double hx = 2.0 * (lphat - lpx) - t;
        if (hx > 0.0) {
            b = x; hb = hx; have_b = true;
#pragma unroll
            for (int j = 0; j < 3; ++j) vb[j] = vx[j];
            done = fabs(hx) <= kProfRootTol;
        } else {
            a = x; ha = hx;
#pragma unroll
            for (int j = 0; j < 3; ++j) va[j] = vx[j];
            if (fabs(hx) <= kProfRootTol) { done = true; break; }
            if (fabs(bound - x) <= kProfWidthTol) { flags = MDG_PROFILE_AT_BOUND; break; }
            double xn = x + sgn * fabs(x - Dhat);
            if (!(sgn * (bound - xn) > 0.5 * fabs(bound - x))) xn = 0.5 * (x + bound);
            x = xn;
        }
    }
    // refinement: Illinois
    int kept = 0;  // which end the last step kept: -1 a, +1 b
    while (have_b && !done && flags == 0u) {
        if (fabs(b - a) <= kProfWidthTol) break;
        double xn = a - ha * (b - a) / (hb - ha);
        const double lo = fmin(a, b), hi = fmax(a, b);
        if (!(xn > lo && xn < hi)) xn = 0.5 * (a + b);
        x = xn;
        const bool from_a = fabs(x - a) <= fabs(b - x);
#pragma unroll
        for (int j = 0; j < 3; ++j) vx[j] = from_a ? va[j] : vb[j];
        if (++n_fit > kProfMaxOuter || !profile_fit_best<NPL>(ob, sumC, slack, x, ptab, phi_min, has_spare, lig, vx, vmode, lpx, n_eval)) {
            flags = MDG_PROFILE_FAILED;
            break;
        }
        const double hx = 2.0 * (lphat - lpx) - t;
        if (fabs(hx) <= kProfRootTol) break;
        if (hx > 0.0) {
            b = x; hb = hx;
#pragma unroll
            for (int j = 0; j < 3; ++j) vb[j] = vx[j];
            if (kept == 1) ha *= 0.5;
            kept = 1;
        } else {
            a = x; ha = hx;
#pragma unroll
            for (int j = 0; j < 3; ++j) va[j] = vx[j];
            if (kept == -1) hb *= 0.5;
            kept = -1;
        }
    }
    out.n_eval = n_eval;
    out.flags = flags;
    if (flags & MDG_PROFILE_FAILED) return;
    double th[4];
    profile_theta(x, vx, phi_min, th);
    out.D = (flags & MDG_PROFILE_AT_BOUND) ? bound : x;
    out.q = th[0]; out.A = th[1]; out.c = th[2]; out.phi = th[3];
    out.logp = lpx;
}

// One warp per (TaxID, PMD run, side) item on a persistent grid, with map_batch_kernel's lane layout (NPL for all 2P
// positions, the same spare-slot rule). Ends of runs that were not made are left to map_interval_header_kernel.
template <int NPL, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, MDG_MAP_MINBLOCKS) map_profile_kernel(const MapProfileLaunch p) {
    __shared__ unsigned int sh_item[WARPS];
    __shared__ double2 sh_prior[64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    log_table_init();
    prior_table_init<0>(sh_prior, p.pr, 0);
    const double t = profile_threshold(p.level);
    const unsigned per_tax = 2u * (unsigned)p.n_prof;
    const unsigned total = (unsigned)p.n_tax * per_tax;
    for (;;) {
        if (lane == 0) sh_item[warp] = atomicAdd(p.work_counter, 1u);
        __syncwarp();
        const unsigned item = sh_item[warp];
        __syncwarp();
        if (item >= total) break;
        const int tax = (int)(item / per_tax), rem = (int)(item % per_tax);
        const int prof = rem >> 1, side = rem & 1, run = 2 * prof;  // run kinds 0, 2, 4: mask = prof
        const mdg_map_run rec = p.map[tax].run[run];
        mdg_profile_end e;
        if (rec.n_eval == 0u && isnan(rec.logp)) {  // run not made (all NaN, no evaluations)
            e.D = e.q = e.A = e.c = e.phi = e.logp = nan("");
            e.n_eval = e.flags = 0u;
        } else if (rec.flags & (MDG_FIT_FAILED | MDG_FIT_MAP_NOT_CONVERGED)) {
            e.D = e.q = e.A = e.c = e.phi = e.logp = nan("");
            e.n_eval = 0u;
            e.flags = MDG_FIT_FAILED;
        } else {
            LaneObs<NPL> ob;
            load_obs<NPL, 32>(ob, p.k + (size_t)tax * 2 * p.P, p.N + (size_t)tax * 2 * p.P, p.P, prof, lane);
            double logC[NPL], sumC = 0.0, scale = 0.0;
            log_binom_coeff<NPL>(ob, logC);
#pragma unroll
            for (int s = 0; s < NPL; ++s) { sumC += logC[s]; scale += ob.act[s] ? lgam(ob.N[s] + 1.0) : 0.0; }
            sumC = group_sum<32>(sumC, 0xffffffffu);
            scale = group_sum<32>(scale, 0xffffffffu);
            const double slack = 1e-14 * scale + 1e-10;
            const int n_obs = prof == 0 ? 2 * p.P : p.P;
            profile_end<NPL>(ob, sumC, slack, rec, t, side, sh_prior, p.pr.phi_min, n_obs < NPL * 32, lane, e);
        }
        if (lane == 0) {
            p.out[tax].end[prof][side] = e;
            atomicAdd(&p.eval_totals[run], (unsigned long long)e.n_eval);
        }
    }
}

// Row header, one thread per TaxID, after map_profile_kernel: tax_id, level, threshold, status, and the NaN ends of the
// runs that were not profiled (n_prof = 1).
__global__ void map_interval_header_kernel(const mdg_map_result* map, int n_tax, int n_prof, double level, mdg_map_interval* out) {
    const int tax = blockIdx.x * blockDim.x + threadIdx.x;
    if (tax >= n_tax) return;
    mdg_map_interval& r = out[tax];
    r.tax_id = map[tax].tax_id;
    r.reserved = 0u;
    r.level = level;
    r.threshold = profile_threshold(level);
    for (int prof = n_prof; prof < 3; ++prof)
        for (int side = 0; side < 2; ++side) {
            mdg_profile_end& e = r.end[prof][side];
            e.D = e.q = e.A = e.c = e.phi = e.logp = nan("");
            e.n_eval = e.flags = 0u;
        }
    r.status = r.end[0][0].flags | r.end[0][1].flags;
}

}  // namespace mdg
