// mdg_post_kernels.cuh — K6 posterior predictive (Beta -> Binomial draws, warp bitonic sort,
// median + HPDI; fits.py:89-120) and K5/K7 row assembly (n_sigma fits.py:194-201, asymmetry
// fits.py:204-227, noise fits.py:359-376, bookkeeping fits.py:272-283).
#pragma once
#include "mdg_fit_kernels.cuh"

namespace mdg {

// ---------------------------------------------------------------------------------------------
// per-(sample, position) Philox stream and the samplers of the predictive
// ---------------------------------------------------------------------------------------------
struct Stream {
    uint2 key;
    uint32_t c0, c1, c2, c3;
    bool have;
    double stash;
    __device__ __forceinline__ double uniform() {
        if (have) { have = false; return stash; }
        double u0, u1;
        uniform2(philox4x32(key, c0++, c1, c2, c3), u0, u1);
        stash = u1;
        have = true;
        return u0;
    }
    __device__ __forceinline__ double normal() {  // fresh block, cosine branch only
        double n0, n1;
        have = false;
        normal2(philox4x32(key, c0++, c1, c2, c3), n0, n1);
        return n0;
    }
};

// log of a Gamma(a, 1) variate: Marsaglia-Tsang with the a < 1 boost, in log space for tiny a.
// Logs of positive normal doubles go through the table-driven log_pos, divisions through the Newton
// reciprocal (the CUDA library versions cost 2-3x as many instructions; this kernel draws 3.2e8
// beta-binomial variates per 10 000 TaxIDs).
__device__ __forceinline__ double log_gamma_variate(Stream& st, double a) {
    double boost = 0.0;
    if (a < 1.0) { boost = log_pos(st.uniform()) * rcp_pos(a); a += 1.0; }
    const double dd = a - 1.0 / 3.0, cc = rsqrt(9.0 * dd);
    for (int guard = 0; guard < 1000; ++guard) {
        double x = st.normal();
        double v = 1.0 + cc * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        double u = st.uniform();
        const double ldv = log_pos(dd * v);  // = log(dd) + log(v)
        if (log_pos(u) < 0.5 * x * x + dd - dd * v + dd * (ldv - log_pos(dd))) return ldv + boost;
    }
    return log_pos(dd) + boost;
}

__device__ __forceinline__ double beta_variate(Stream& st, double a, double b) {
    double la = log_gamma_variate(st, a), lb = log_gamma_variate(st, b);
    return rcp_pos(1.0 + exp_fast(lb - la));
}

// Binomial(n, p): BINV inversion for n*min(p,1-p) < 10, BTRS (Hormann 1993) otherwise
__device__ __forceinline__ double binomial_variate(Stream& st, double n, double p) {
    if (!(n > 0.0) || !(p > 0.0)) return 0.0;
    if (p >= 1.0) return n;
    const bool flip = p > 0.5;
    if (flip) p = 1.0 - p;
    double res = 0.0;
    if (n * p < 10.0) {
        const double q = 1.0 - p, s = p * rcp_pos(q), a = (n + 1.0) * s;
        const double r0 = exp_fast(n * log1p(-p));
        for (int guard = 0; guard < 64; ++guard) {
            double r = r0, u = st.uniform(), x = 0.0;
            bool bad = false;
            while (u > r) {
                u -= r;
                x += 1.0;
                if (x > n || x > 2000.0) { bad = true; break; }
                r *= fma(a, rcp_pos(x), -s);
            }
            if (!bad) { res = x; break; }
        }
    } else {
        const double spq = sqrt(n * p * (1.0 - p));
        const double b = 1.15 + 2.53 * spq, a = -0.0873 + 0.0248 * b + 0.01 * p;
        const double c = n * p + 0.5, vr = 0.92 - 4.2 / b;
        const double alpha = (2.83 + 5.1 / b) * spq, lpq = log(p / (1.0 - p));
        const double m = floor((n + 1.0) * p);
        const double h = lgam(m + 1.0) + lgam(n - m + 1.0);
        res = m;
        for (int guard = 0; guard < 1000; ++guard) {
            double u = st.uniform() - 0.5, v = st.uniform();
            double us = 0.5 - fabs(u);
            double kk = floor((2.0 * a / us + b) * u + c);
            if (us >= 0.07 && v <= vr) { res = kk; break; }
            if (kk < 0.0 || kk > n) continue;
            v = log(v * alpha / (a / (us * us) + b));
            if (v <= h - lgam(kk + 1.0) - lgam(n - kk + 1.0) + (kk - m) * lpq) { res = kk; break; }
        }
    }
    return flip ? n - res : res;
}

// ---------------------------------------------------------------------------------------------
// K6 kernel: one warp per (TaxID, predictive position). Items per TaxID: 2P positions of the
// PMD/all run, then D_max_forward and D_max_reverse (position z = 1 of the fwd / rev runs).
// Lanes run over the draws; the warp then bitonic-sorts the S draws in shared memory.
// ---------------------------------------------------------------------------------------------
struct PpcLaunch {
    const int64_t* tax_id;
    const uint32_t* N;
    int n_tax, P;
    mdg_fit_config cfg;
    Priors pr;
    const double* samples;
    int sample_slot[MDG_NUM_RUNS];
    int sample_runs;
    const RunRecord* rec;
    unsigned int* work_counter;
    int items_per_tax;  // 2P (+2 with the fwd/rev runs)
    int s_pad;          // next power of two >= num_samples
    double* pred;       // [n_tax][2P+2][3]: median, hpdi lo, hpdi hi (FP64)
};

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) ppc_kernel(const PpcLaunch p) {
    extern __shared__ uint32_t sh_sort[];  // [WARPS][s_pad]
    __shared__ unsigned int sh_item[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* buf = sh_sort + (size_t)warp * p.s_pad;
    const int S = p.cfg.num_samples, P = p.P, n = p.s_pad;
    const unsigned total = (unsigned)p.n_tax * (unsigned)p.items_per_tax;
    log_table_init();
    for (;;) {
        if (lane == 0) sh_item[warp] = atomicAdd(p.work_counter, 1u);
        __syncwarp();
        const unsigned item = sh_item[warp];
        __syncwarp();
        if (item >= total) break;
        const int tax = (int)(item / (unsigned)p.items_per_tax), j = (int)(item % (unsigned)p.items_per_tax);
        int run_kind, dense;
        if (j < 2 * P) { run_kind = MDG_RUN_PMD_ALL; dense = j; }
        else if (j == 2 * P) { run_kind = MDG_RUN_PMD_FWD; dense = 0; }
        else { run_kind = MDG_RUN_PMD_REV; dense = p.cfg.reference_quirks ? 0 : P; }  // fits.py:343-348
        const double x = (double)(dense < P ? dense : dense - P);
        const double Nn = (double)p.N[(size_t)tax * 2 * P + dense];
        double* out = p.pred + ((size_t)tax * p.items_per_tax + j) * 3;
        const bool failed = p.rec[(size_t)tax * MDG_NUM_RUNS + run_kind].failed != 0;
        if (failed || !(Nn > 0.0) || S < 1) {
            if (lane == 0) { out[0] = nan(""); out[1] = nan(""); out[2] = nan(""); }
            continue;
        }
        const uint2 key = make_key(p.cfg.seed, p.tax_id[tax]);
        const double* smp = p.samples + ((size_t)tax * p.sample_runs + p.sample_slot[run_kind]) * (size_t)S * 4;
        for (int s = lane; s < n; s += 32) {
            uint32_t y = 0xFFFFFFFFu;
            if (s < S) {
                const double q = smp[(size_t)s * 4], A = smp[(size_t)s * 4 + 1], c = smp[(size_t)s * 4 + 2], phi = smp[(size_t)s * 4 + 3];
                double Dz = fma(A, exp_fast(x * log1p(-q)), c);
                Dz = fmin(fmax(Dz, 0.0), 1.0);
                Stream st;
                st.key = key; st.c0 = 0u; st.c1 = (uint32_t)s; st.c2 = c2word(run_kind, P_PPC); st.c3 = (uint32_t)dense; st.have = false; st.stash = 0.0;
                const double pr = beta_variate(st, Dz * phi, (1.0 - Dz) * phi);
                y = (uint32_t)binomial_variate(st, Nn, pr);
            }
            buf[s] = y;
        }
        __syncwarp();
        // bitonic sort of n = s_pad keys, 32 lanes over n/2 compare-exchanges per stage
        for (int kk = 2; kk <= n; kk <<= 1) {
            for (int jj = kk >> 1; jj > 0; jj >>= 1) {
                for (int tt = lane; tt < (n >> 1); tt += 32) {
                    const int i = 2 * tt - (tt & (jj - 1));
                    const int ixj = i + jj;
                    const uint32_t a = buf[i], b = buf[ixj];
                    const bool up = (i & kk) == 0;
                    if ((a > b) == up) { buf[i] = b; buf[ixj] = a; }
                }
                __syncwarp();
            }
        }
        // np.median and numpyro.diagnostics.hpdi(prob) on y/N
        const double med = (S & 1) ? (double)buf[S / 2] / Nn : ((double)buf[S / 2 - 1] / Nn + (double)buf[S / 2] / Nn) / 2;
        int L = (int)(p.cfg.hpdi_prob * S);
        if (L >= S) L = S - 1;
        double bw = INFINITY;
        int bi = 0x7fffffff;
        for (int i = lane; i < S - L; i += 32) {
            const double w = (double)buf[i + L] / Nn - (double)buf[i] / Nn;
            if (w < bw) { bw = w; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ow = __shfl_xor_sync(0xffffffffu, bw, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ow < bw || (ow == bw && oi < bi)) { bw = ow; bi = oi; }
        }
        if (lane == 0) {
            out[0] = med;
            out[1] = (double)buf[bi] / Nn;
            out[2] = (double)buf[bi + L] / Nn;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// K5/K7 kernel: one thread per TaxID assembles the mdg_fit_result row
// ---------------------------------------------------------------------------------------------
struct AssembleLaunch {
    const int64_t* tax_id;
    const uint32_t* k;
    const uint32_t* N;
    const uint32_t* mism12;  // optional
    const double* noise3;    // optional
    int n_tax, P;
    mdg_fit_config cfg;
    const RunRecord* rec;
    const MapRecord* map;    // NULL if !do_map
    const double* waic;      // [n_tax][6][2][2P]
    const double* pred;      // [n_tax][items_per_tax][3]
    int items_per_tax;
    mdg_fit_result* out;
    float* out_median;
    float* out_lo;
    float* out_hi;
    unsigned long long* leapfrog_totals;  // [6]
};

__device__ __forceinline__ double waic_i_at(const double* w, int R, int i) { return -2.0 * (w[i] - w[R + i]); }

// n_sigma of fits.py:194-201 over positions [lo, lo+n) of two runs' (lppd_i, pWAIC_i) blocks
__device__ inline double n_sigma_dev(const double* wa, const double* wb, int R, int lo, int n) {
    double mean = 0.0, sa = 0.0, sb = 0.0;
    for (int i = 0; i < n; ++i) {
        double a = waic_i_at(wa, R, lo + i), b = waic_i_at(wb, R, lo + i);
        mean += a - b; sa += a; sb += b;
    }
    mean /= n;
    double var = 0.0;
    for (int i = 0; i < n; ++i) {
        double d = waic_i_at(wa, R, lo + i) - waic_i_at(wb, R, lo + i) - mean;
        var += d * d;
    }
    var /= n;
    return (sb - sa) / sqrt(n * var);
}

__device__ inline double nan_std(const double* v, int n) {
    double s = 0.0; int m = 0;
    for (int i = 0; i < n; ++i) if (!isnan(v[i])) { s += v[i]; ++m; }
    if (m == 0) return nan("");
    const double mean = s / m;
    double q = 0.0;
    for (int i = 0; i < n; ++i) if (!isnan(v[i])) { double d = v[i] - mean; q += d * d; }
    return sqrt(q / m);
}

// integer bookkeeping of fits.py:272-283 (z = 1 coverage, sums of N and k per strand) into any row type with these fields
template <typename Row>
__device__ __forceinline__ void tax_sums(const uint32_t* k, const uint32_t* N, int P, Row& r) {
    const int R = 2 * P;
    r.N_z1_forward = N[0];
    r.N_z1_reverse = N[P];
    for (int s = 0; s < R; ++s) {
        if (s < P) { r.N_sum_forward += N[s]; r.y_sum_forward += k[s]; }
        else { r.N_sum_reverse += N[s]; r.y_sum_reverse += k[s]; }
    }
    r.N_sum_total = r.N_sum_forward + r.N_sum_reverse;
    r.y_sum_total = r.y_sum_forward + r.y_sum_reverse;
}

// normalized_noise, _forward, _reverse (fits.py:359-376) from the raw off-diagonal counts mism12 [n_tax][2P][12]
// (CT is column 5 and GA column 6 of the 12), else copied from noise3 [n_tax][3]; fields are left alone (the caller's
// NaN) if both are NULL
template <typename Row>
__device__ __forceinline__ void tax_noise(const uint32_t* mism12, const double* noise3, int tax, int P, Row& r) {
    const int R = 2 * P;
    const double qnan = nan("");
    if (mism12 != nullptr) {
        const uint32_t* m = mism12 + (size_t)tax * R * 12;
        double col_mean[12];
        for (int c = 0; c < 12; ++c) {
            double s = 0.0; int cnt = 0;
            for (int row = 0; row < R; ++row) {
                const bool blank = (row < P && c == 5) || (row >= P && c == 6);
                if (!blank) { s += (double)m[row * 12 + c]; ++cnt; }
            }
            col_mean[c] = cnt ? s / cnt : qnan;
        }
        double out3[3];
        for (int part = 0; part < 3; ++part) {
            const int r0 = part == 2 ? P : 0, r1 = part == 1 ? P : R;
            double s = 0.0; int cnt = 0;
            for (int row = r0; row < r1; ++row)
                for (int c = 0; c < 12; ++c) {
                    const bool blank = (row < P && c == 5) || (row >= P && c == 6);
                    const double v = blank ? qnan : (double)m[row * 12 + c] / col_mean[c];
                    if (!isnan(v)) { s += v; ++cnt; }
                }
            if (cnt == 0) { out3[part] = qnan; continue; }
            const double mean = s / cnt;
            double qq = 0.0;
            for (int row = r0; row < r1; ++row)
                for (int c = 0; c < 12; ++c) {
                    const bool blank = (row < P && c == 5) || (row >= P && c == 6);
                    const double v = blank ? qnan : (double)m[row * 12 + c] / col_mean[c];
                    if (!isnan(v)) { double d = v - mean; qq += d * d; }
                }
            out3[part] = sqrt(qq / cnt);
        }
        r.normalized_noise = out3[0]; r.normalized_noise_forward = out3[1]; r.normalized_noise_reverse = out3[2];
    } else if (noise3 != nullptr) {
        r.normalized_noise = noise3[(size_t)tax * 3];
        r.normalized_noise_forward = noise3[(size_t)tax * 3 + 1];
        r.normalized_noise_reverse = noise3[(size_t)tax * 3 + 2];
    }
}

__global__ void assemble_kernel(const AssembleLaunch p) {
    const int tax = blockIdx.x * blockDim.x + threadIdx.x;
    if (tax >= p.n_tax) return;
    const int P = p.P, R = 2 * P;
    const uint32_t* k = p.k + (size_t)tax * R;
    const uint32_t* N = p.N + (size_t)tax * R;
    const RunRecord* rr = p.rec + (size_t)tax * MDG_NUM_RUNS;
    const double* wa = p.waic + (size_t)tax * MDG_NUM_RUNS * 2 * R;
    const double* pred = p.pred + (size_t)tax * p.items_per_tax * 3;
    mdg_fit_result r;
    memset(&r, 0, sizeof r);
    const double qnan = nan("");
    r.tax_id = p.tax_id[tax];
    tax_sums(k, N, P, r);
    r.n_sigma_forward = r.D_max_forward = r.q_mean_forward = qnan;
    r.n_sigma_reverse = r.D_max_reverse = r.q_mean_reverse = r.asymmetry = qnan;
    r.normalized_noise = r.normalized_noise_forward = r.normalized_noise_reverse = qnan;
    r.map_A = r.map_q = r.map_c = r.map_phi = r.map_D_max = r.map_logp = qnan;
    r.map_null_q = r.map_null_phi = r.map_null_logp = qnan;
    uint32_t status = 0;
    const int n_runs = p.cfg.do_fwd_rev ? MDG_NUM_RUNS : 2;
    for (int i = 0; i < n_runs; ++i) {
        r.run[i].step_size = rr[i].step_size;
        r.run[i].mean_accept = rr[i].mean_accept;
        r.run[i].n_leapfrog = rr[i].n_leapfrog;
        r.run[i].n_divergent = rr[i].n_divergent;
        r.run[i].waic = rr[i].waic;
        r.run[i].lppd = rr[i].lppd;
        if (rr[i].failed) status |= MDG_FIT_FAILED;
        if (rr[i].failed == 2u) status |= MDG_FIT_BUDGET_EXCEEDED;
        if (rr[i].n_divergent) status |= MDG_FIT_HAS_DIVERGENCES;
        atomicAdd(&p.leapfrog_totals[i], (unsigned long long)rr[i].n_leapfrog);
    }
    if (p.map != nullptr) {
        const MapRecord& m0 = p.map[(size_t)tax * 2];
        const MapRecord& m1 = p.map[(size_t)tax * 2 + 1];
        r.map_q = m0.theta[0]; r.map_A = m0.theta[1]; r.map_c = m0.theta[2]; r.map_phi = m0.theta[3];
        r.map_D_max = m0.theta[1] + m0.theta[2];
        r.map_logp = m0.logp;
        r.map_iters = m0.iters;
        r.map_null_q = m1.theta[0]; r.map_null_phi = m1.theta[3]; r.map_null_logp = m1.logp;
        if (!m0.converged || !m1.converged) status |= MDG_FIT_MAP_NOT_CONVERGED;
    }
    if (!(status & MDG_FIT_FAILED)) {
        r.q_mean = rr[0].mean[0]; r.q_std = rr[0].sd[0];
        r.concentration_mean = rr[0].mean[1]; r.concentration_std = rr[0].sd[1];
        r.D_max_marginalized_mean = rr[0].mean[2]; r.D_max_marginalized_std = rr[0].sd[2];
        r.A_mean = rr[0].mean[3]; r.c_mean = rr[0].mean[4];
        r.n_sigma = n_sigma_dev(wa, wa + 2 * R, R, 0, R);
        r.D_max = pred[0]; r.D_max_lower_hpdi = pred[1]; r.D_max_upper_hpdi = pred[2];
        if (p.cfg.do_fwd_rev) {
            r.q_mean_forward = rr[2].mean[0];
            r.q_mean_reverse = rr[4].mean[0];
            r.n_sigma_forward = n_sigma_dev(wa + 2 * 2 * R, wa + 3 * 2 * R, R, 0, P);
            r.n_sigma_reverse = n_sigma_dev(wa + 4 * 2 * R, wa + 5 * 2 * R, R, P, P);
            r.D_max_forward = pred[(size_t)(2 * P) * 3];
            r.D_max_reverse = pred[(size_t)(2 * P + 1) * 3];
            // asymmetry, fits.py:204-227: combined vs concat(forward, reverse)
            const double* wf = wa + 2 * 2 * R;
            const double* wr = wa + 4 * 2 * R;
            double mean = 0.0;
            for (int i = 0; i < R; ++i) mean += waic_i_at(wa, R, i) - waic_i_at(i < P ? wf : wr, R, i);
            mean /= R;
            double var = 0.0;
            for (int i = 0; i < R; ++i) {
                double d = waic_i_at(wa, R, i) - waic_i_at(i < P ? wf : wr, R, i) - mean;
                var += d * d;
            }
            var /= R;
            r.asymmetry = (rr[2].waic + rr[4].waic - rr[0].waic) / sqrt(R * var);
        }
    } else {
        r.D_max = r.n_sigma = r.D_max_lower_hpdi = r.D_max_upper_hpdi = qnan;
        r.q_mean = r.concentration_mean = r.D_max_marginalized_mean = qnan;
    }
    for (int s = 0; s < R; ++s) {
        const bool ok = !(status & MDG_FIT_FAILED);
        if (p.out_median) p.out_median[(size_t)tax * R + s] = ok ? (float)pred[(size_t)s * 3] : nanf("");
        if (p.out_lo) p.out_lo[(size_t)tax * R + s] = ok ? (float)pred[(size_t)s * 3 + 1] : nanf("");
        if (p.out_hi) p.out_hi[(size_t)tax * R + s] = ok ? (float)pred[(size_t)s * 3 + 2] : nanf("");
    }
    tax_noise(p.mism12, p.noise3, tax, P, r);
    r.status = status;
    p.out[tax] = r;
}

}  // namespace mdg
