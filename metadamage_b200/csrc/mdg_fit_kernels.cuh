// mdg_fit_kernels.cuh — records and launch parameters shared by the fit kernels, the per-chain shared-memory
// state of K4 (NUTS, mdg_nuts_kernel.cuh) and K3 (MAP): mode of the constrained-space posterior by damped Newton,
// one warp per (TaxID, model).
#pragma once
#include "mdg_model.cuh"

namespace mdg {

constexpr int kMaxTreeDepth = 10;
constexpr int kMaxWindows = 16;
constexpr int kDaTable = 1024;  // entries of the dual-averaging tables sqrt(t), t^-0.75

struct RunRecord {
    double step_size, mean_accept;
    uint32_t n_leapfrog, n_divergent;
    double waic, lppd;
    double mean[5], sd[5];  // q, phi, A+c, A, c (posterior mean / std, ddof 0)
    uint32_t failed, pad;
};

struct FitLaunch {
    const int64_t* tax_id;
    const uint32_t* k;
    const uint32_t* N;
    int n_tax, P;
    mdg_fit_config cfg;
    Priors pr;
    int n_windows;
    int win_end[kMaxWindows];
    unsigned int* work_counter;
    int n_items;        // ONE queue per launch: n_items_all all-position runs (one per TaxID) and n_items - n_items_all
    int n_items_all;    // forward-only / reverse-only runs (two per TaxID, mask 1 + (w & 1)), in three sections: the forward /
    int n_prio;         // reverse runs of the first n_prio TaxIDs of `order`, every all-position run, the other forward / reverse runs
    const int* order;   // [n_tax] queue position -> TaxID index of the chunk (nuts_order kernels), or NULL = identity
    RunRecord* rec;     // [n_tax][6]
    double* waic;       // [n_tax][6][2][2P]: lppd_i, pWAIC_i
    double* samples;    // [n_tax][sample_runs][S][4] constrained draws, or NULL
    int sample_slot[MDG_NUM_RUNS];  // run kind -> slot in `samples`, -1 = not stored
    int sample_runs;
    double* trace;      // [n_tax][6][W+S][4] or NULL
    int n_slots;        // rounds of the position loop of the launch's longest run, ceil((n_obs + 1) / GW): shared-memory layout
    const double* da_sqrt;  // [kDaTable] sqrt(t)
    const double* da_pow;   // [kDaTable] t^-0.75 (dual averaging, hmc_util.dual_averaging kappa)
    double* waic_acc;   // WAIC accumulators, [grid * warps][4][n_slots][32]
    unsigned long long* chain_clock;  // development (MDG_CHAIN_CLOCK): [n_tax][6][2] globaltimer at chain start / end, or NULL
};

template <int D>
struct GroupShared {
    double zl[D], rl[D], gl[D], zr[D], rr[D], gr[D];  // main tree edges
    double zp[D], gp[D];                              // main proposal == chain state between transitions
    double szp[D], sgp[D];                            // subtree proposal
    double rck[kMaxTreeDepth][D], rsck[kMaxTreeDepth][D];
    double wf_mean[D], wf_m2[D];
    double acc_mean[5], acc_m2[5];
    // cold group-uniform chain state (touched once per transition / doubling, never inside the
    // gradient evaluation). Kept here, 8 bytes per value per chain, instead of in registers: the
    // compiler's spills would replicate each of them 32x in local memory (ncu: 866 B of spills per
    // thread at 128 registers = 443 KB per SM, more than the L1 holds).
    double da_x, da_xavg, da_gavg, da_prox, mean_accept, h_step, h_Er;
    double m_weight, m_sum_acc, m_pe_p, u_main, pe_cur, eps, s_pe_p;
    double m_rsum[D];
    // group-uniform values that are live ACROSS the gradient evaluation but not used inside it:
    // parked here so that the evaluation's five interleaved special-function chains get the registers
    double imm[D], s_rsum[D], zn_park[D], rh_park[D], E0, s_weight, s_sum_acc;
    double isd[D];  // 1 / sqrt(imm) = sqrt of the mass matrix diagonal (momentum r ~ N(0, M) is n * isd)
    int da_t, wf_n, window_idx, h_last, h_dir, m_nprop;
    uint32_t h_att, h_call, init_attempt, n_div;
};


template <int D>
__device__ __forceinline__ double kinetic(const double (&imm)[D], const double (&r)[D]) {
    double e = 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) e = fma(imm[j] * r[j], r[j], e);
    return 0.5 * e;
}

// generalised U-turn test (hmc_util._is_turning, diagonal mass matrix)
template <int D>
__device__ __forceinline__ bool is_turning(const double (&imm)[D], const double* r_left, const double* r_right,
                                           const double* r_sum) {
    double dl = 0.0, dr = 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double rho = r_sum[j] - (r_left[j] + r_right[j]) / 2;
        dl += imm[j] * r_left[j] * rho;
        dr += imm[j] * r_right[j] * rho;
    }
    return (dl <= 0.0) || (dr <= 0.0);
}

struct Vec4 { double v[4]; };

// ---------------------------------------------------------------------------------------------
// K3: MAP — mode of the constrained-space posterior density (no Jacobian term), LM-damped Newton
// in unconstrained coordinates with a central-difference Hessian of the analytic gradient.
// One warp per (TaxID, model).
// ---------------------------------------------------------------------------------------------
struct MapRecord {
    double theta[4];  // q, A, c, phi
    double logp;
    uint32_t iters, converged;
};

struct MapLaunch {
    const int64_t* tax_id;
    const uint32_t* k;
    const uint32_t* N;
    int n_tax, P;
    Priors pr;
    unsigned int* work_counter;
    MapRecord* rec;  // [n_tax][2]: PMD, null
};

template <int D>
__device__ __forceinline__ bool chol_solve(const double (&H)[D][D], const double (&rhs)[D], double (&x)[D]) {
    double L[D][D];
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) L[i][j] = 0.0;
    bool ok = true;
#pragma unroll
    for (int i = 0; i < D; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = H[i][j];
#pragma unroll
            for (int m = 0; m < j; ++m) s -= L[i][m] * L[j][m];
            if (i == j) { ok = ok && (s > 0.0); L[i][i] = sqrt(s); }
            else L[i][j] = s / L[j][j];
        }
    }
    if (!ok) return false;
    double y[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = rhs[i];
#pragma unroll
        for (int m = 0; m < i; ++m) s -= L[i][m] * y[m];
        y[i] = s / L[i][i];
    }
#pragma unroll
    for (int i = D - 1; i >= 0; --i) {
        double s = y[i];
#pragma unroll
        for (int m = i + 1; m < D; ++m) s -= L[m][i] * x[m];
        x[i] = s / L[i][i];
    }
    return true;
}

// What the MAP-only path (mdg_map_batch_kernel.cuh) needs beyond MapRecord: the unconstrained mode and the number
// of gradient evaluations. Only instantiations with TRACE = true fill it; map_kernel's (TRACE = false) compiles
// to the same code as without it.
struct MapTrace {
    double u[4];
    uint32_t n_eval;
};

template <int MODEL, int NPL, bool TRACE = false>
__device__ void map_fit_group(const LaneObs<NPL>& ob, const double (&logC)[NPL], int P, const Priors& pr,
                              const double2* ptab, bool has_spare, int lig, MapRecord& out, MapTrace* trace = nullptr) {
    constexpr int D = ModelDim<MODEL>::value;
    constexpr unsigned gmask = 0xffffffffu;
    constexpr double UMAX = 40.0;
    // ---- data-driven starting point ----
    double u[D];
    {
        double ktail = 0, Ntail = 0, k1 = 0, N1 = 0, kall = 0, Nall = 0;
        const double xmax = (double)(P - 1);
#pragma unroll
        for (int s = 0; s < NPL; ++s) {
            if (ob.act[s]) {
                kall += ob.k[s]; Nall += ob.N[s];
                if (ob.x[s] == 0.0) { k1 += ob.k[s]; N1 += ob.N[s]; }
                if (ob.x[s] >= xmax - 2.0) { ktail += ob.k[s]; Ntail += ob.N[s]; }
            }
        }
        ktail = group_sum<32>(ktail, gmask); Ntail = group_sum<32>(Ntail, gmask);
        k1 = group_sum<32>(k1, gmask); N1 = group_sum<32>(N1, gmask);
        kall = group_sum<32>(kall, gmask); Nall = group_sum<32>(Nall, gmask);
        double f_all = (kall + 0.5) / (Nall + 1.0);
        double c0 = (ktail + 0.5) / (Ntail + 1.0);
        double A0 = (k1 + 0.5) / (N1 + 1.0) - c0;
        c0 = fmin(fmax(c0, 1e-6), 0.5);
        A0 = fmin(fmax(A0, 1e-3), 0.45);
        f_all = fmin(fmax(f_all, 1e-6), 0.9);
        if (MODEL == 0) {
            u[0] = log(0.3 / 0.7);
            u[1] = log(A0 / (1.0 - A0));
            u[2] = log(c0 / (1.0 - c0));
            u[3] = log(100.0);
        } else {
            u[0] = log(f_all / (1.0 - f_all));
            u[1] = log(100.0);
        }
    }
    double f, g[D], ll[NPL], lp;
    bool ok;
    eval_model<MODEL, NPL, 32>(ob, u, ptab, pr.phi_min, has_spare, gmask, lig, lp, g, ll, ok);
    if (TRACE) trace->n_eval = 1;
    // f carries log C(N,k) so that its magnitude (and the step-acceptance slack) matches the
    // constrained-space log posterior; `slack` covers the cancellation noise of the lgamma sums
    double sumC = 0.0, scale = 0.0;
#pragma unroll
    for (int s = 0; s < NPL; ++s) { sumC += logC[s]; scale += ob.act[s] ? lgam(ob.N[s] + 1.0) : 0.0; }
    sumC = group_sum<32>(sumC, gmask);
    scale = group_sum<32>(scale, gmask);
    const double slack = 1e-14 * scale + 1e-10;
    out.converged = 0;
    out.iters = 0;
    if (!ok) {
#pragma unroll
        for (int j = 0; j < 4; ++j) out.theta[j] = nan("");
        out.logp = nan("");
        return;
    }
    f = -(lp + sumC);
#pragma unroll
    for (int j = 0; j < D; ++j) g[j] = -g[j];
    double lambda = 1e-3;
    int it = 0;
    bool converged = false;
    for (it = 0; it < 200; ++it) {
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
            if (TRACE) trace->n_eval += 2;
#pragma unroll
            for (int i = 0; i < D; ++i) H[i][j] = (okp && okm) ? -(gp[i] - gm[i]) / (2.0 * h) : (i == j ? 1.0 : 0.0);
        }
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) { double s = 0.5 * (H[i][j] + H[j][i]); H[i][j] = s; H[j][i] = s; }
        bool accepted = false;
        for (int tries = 0; tries < 40 && !accepted; ++tries) {
            double Hd[D][D], rhs[D], du[D];
#pragma unroll
            for (int i = 0; i < D; ++i) {
#pragma unroll
                for (int j = 0; j < D; ++j) Hd[i][j] = H[i][j];
                Hd[i][i] += lambda * (fabs(H[i][i]) + 1e-8);
                rhs[i] = -g[i];
            }
            if (!chol_solve<D>(Hd, rhs, du)) { lambda *= 10.0; continue; }
            double un[D], gn[D], lpn, dmax = 0.0;
#pragma unroll
            for (int i = 0; i < D; ++i) {
                un[i] = fmin(fmax(u[i] + du[i], -UMAX), UMAX);
                dmax = fmax(dmax, fabs(un[i] - u[i]));
            }
            bool okn;
            eval_model<MODEL, NPL, 32>(ob, un, ptab, pr.phi_min, has_spare, gmask, lig, lpn, gn, ll, okn);
            if (TRACE) trace->n_eval += 1;
            if (okn && -(lpn + sumC) <= f + slack) {
                double gmax = 0.0;
#pragma unroll
                for (int i = 0; i < D; ++i) { u[i] = un[i]; g[i] = -gn[i]; gmax = fmax(gmax, fabs(gn[i])); }
                f = -(lpn + sumC);
                lambda = fmax(lambda / 3.0, 1e-12);
                accepted = true;
                if (dmax < 1e-10 || gmax < 1e-9) converged = true;
            } else {
                lambda *= 4.0;
                if (dmax < 1e-13) { converged = true; accepted = true; }
            }
        }
        if (!accepted) break;
        if (converged) { ++it; break; }
    }
    double th[4];
    constrain<MODEL>(u, pr.phi_min, th);
#pragma unroll
    for (int j = 0; j < 4; ++j) out.theta[j] = th[j];
    out.logp = -f;
    out.iters = (uint32_t)it;
    out.converged = converged ? 1u : 0u;
    if (TRACE) {
#pragma unroll
        for (int j = 0; j < D; ++j) trace->u[j] = u[j];
    }
}

#ifndef MDG_MAP_MINBLOCKS
#define MDG_MAP_MINBLOCKS 4
#endif
template <int NPL, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, MDG_MAP_MINBLOCKS) map_kernel(const MapLaunch p) {
    __shared__ unsigned int sh_item[WARPS];
    __shared__ double2 sh_prior[2][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    log_table_init();
    prior_table_init<0>(sh_prior[0], p.pr, 0);
    prior_table_init<1>(sh_prior[1], p.pr, 0);
    for (;;) {
        if (lane == 0) sh_item[warp] = atomicAdd(p.work_counter, 1u);
        __syncwarp();
        const unsigned item = sh_item[warp];
        __syncwarp();
        if (item >= 2u * (unsigned)p.n_tax) break;
        const int tax = (int)(item >> 1), model = (int)(item & 1u);
        LaneObs<NPL> ob;
        load_obs<NPL, 32>(ob, p.k + (size_t)tax * 2 * p.P, p.N + (size_t)tax * 2 * p.P, p.P, 0, lane);
        double logC[NPL];
        log_binom_coeff<NPL>(ob, logC);
        const bool has_spare = 2 * p.P < NPL * 32;
        MapRecord rec;
        if (model == 0) map_fit_group<0, NPL>(ob, logC, p.P, p.pr, sh_prior[0], has_spare, lane, rec);
        else map_fit_group<1, NPL>(ob, logC, p.P, p.pr, sh_prior[1], has_spare, lane, rec);
        if (lane == 0) p.rec[item] = rec;
    }
}


// ---------------------------------------------------------------------------------------------
// Queue order of a chunk's TaxIDs. The chains that decide when a batch ends sit at the two ends of the coverage
// range: TaxIDs with a handful of reads (degenerate posteriors — adapted step sizes of 0.003-0.03 and 10^5..10^6
// leapfrogs in one run, against a mean of 10^4) and, an order of magnitude less extreme, the TaxIDs with the most
// reads (narrow posteriors). A chain is sequential, so the only thing a scheduler can do for them is start them
// first: a counting sort over half-octave buckets of N_sum, the buckets taken from both ends towards the middle.
// (Results do not depend on the order: every chain is keyed by (seed, tax_id, run).)
// ---------------------------------------------------------------------------------------------
constexpr int kOrderBuckets = 96;

__device__ __forceinline__ int order_bucket(unsigned long long n_sum) {
    if (n_sum < 2ull) return (int)n_sum;
    const int lg = 63 - __clzll((long long)n_sum);
    return min(kOrderBuckets - 1, 2 * lg + (int)((n_sum >> (lg - 1)) & 1ull));
}

// counters: [kOrderBuckets] histogram, then [kOrderBuckets] first queue position, then [kOrderBuckets] cursors
__global__ void nuts_order_count_kernel(const uint32_t* __restrict__ N, int n_tax, int R, unsigned char* __restrict__ bucket,
                                        unsigned int* __restrict__ counters) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tax) return;
    unsigned long long sum = 0;
    for (int j = 0; j < R; ++j) sum += N[(size_t)i * R + j];
    const int b = order_bucket(sum);
    bucket[i] = (unsigned char)b;
    atomicAdd(counters + b, 1u);
}

__global__ void nuts_order_offsets_kernel(unsigned int* __restrict__ counters) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int lo = 0, hi = kOrderBuckets - 1;
    unsigned int pos = 0;
    bool take_low = true;
    while (lo <= hi) {
        const int b = take_low ? lo++ : hi--;
        counters[kOrderBuckets + b] = pos;
        counters[2 * kOrderBuckets + b] = 0u;
        if (counters[b] != 0u) take_low = !take_low;  // alternate only over buckets that hold TaxIDs
        pos += counters[b];
    }
}

__global__ void nuts_order_scatter_kernel(const unsigned char* __restrict__ bucket, int n_tax, unsigned int* __restrict__ counters,
                                          int* __restrict__ order) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tax) return;
    const int b = bucket[i];
    order[counters[kOrderBuckets + b] + atomicAdd(counters + 2 * kOrderBuckets + b, 1u)] = i;
}

}  // namespace mdg
