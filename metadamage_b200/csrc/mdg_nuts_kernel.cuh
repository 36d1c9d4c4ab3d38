// mdg_nuts_kernel.cuh — K4 (NUTS) with K2 (log-density + gradient) and K5 (WAIC accumulation) fused in.
//
// Layout (round 2). A chain is owned by a GROUP of GW lanes (GW = 8 by default: four chains per warp), and
// the positions of its TaxID are spread over the group's lanes in `n_slots` rounds of a ROLLED loop:
// linear index i = slot * GW + lane-in-group, index 0 is a spare (k = N = 0: it evaluates exactly the
// position-independent lgamma/digamma(phi) [null model: also of alpha and beta] that every other index
// needs, and is broadcast from there), index i >= 1 is observation i - 1. Why:
//   * Per leapfrog only the per-position special functions (5 lgamma/digamma pairs per position, PMD) are
//     parallel work; the transforms, reductions, tree bookkeeping, U-turn tests and random numbers are
//     the same for every lane of a chain. One chain per warp (round 1) issued that group-uniform half of
//     the instruction stream once per chain; here it is issued once per FOUR chains (ncu, round 1: 1 096
//     warp instructions per gradient evaluation of which ~510 are the per-position part).
//   * The slot loop is rolled, so the hot code is ONE copy of the per-position block whatever max_position
//     is (round 1's two-positions-per-lane variant was unrolled, grew past the 32 KB instruction cache and
//     lost), and one kernel per model serves all-position, forward-only and reverse-only runs and any P.
//   * Groups are independent state machines: a group whose chain ends writes its outputs and pulls the next
//     (TaxID, run) item from the launch's atomic counter while its neighbours keep going.
// Every loop trip of a group does exactly one leapfrog (one log-density-gradient evaluation); what the
// evaluation was for (initial-point search, step-size heuristic, tree leaf) is bookkeeping afterwards.
//
// The NUTS transition restates numpyro 0.4.1 (hmc.py / hmc_util.py: build_tree, _iterative_build_subtree,
// _combine_tree, _is_turning, warmup_adapter, dual_averaging, welford_covariance,
// find_reasonable_step_size) as driven by fits.py:382-387 with the kwargs of fits.py:792-799; the model is
// fits.py:43-67 with numpyro's BetaBinomial.log_prob and the sigmoid / exp bijections (SURVEY.md 8c-notes).
//
// Per-position log-likelihoods of the candidate points (needed by the WAIC statistics of fits.py:147-165
// for the draw that is finally kept) live in four shared-memory buffers per warp whose ROLES (scratch,
// subtree proposal, tree proposal, current state) are permuted instead of copying values.
#pragma once
#include "mdg_fit_kernels.cuh"

namespace mdg {

// momentum r ~ N(0, M), M^-1 = diag(imm): r_j = n_j * isd_j with isd = 1 / sqrt(imm) kept per chain (it changes at
// the four adaptation-window ends only). The D standard normals are drawn ACROSS the lanes: the lane that owns
// component j evaluates the Philox block j / 2 and keeps component j % 2 of its Box-Muller pair (one Philox + one
// Box-Muller in the instruction stream instead of two of each).
template <int D>
__device__ MDG_COLD double draw_normal_lane_cold(uint2 key, uint32_t c1, uint32_t c2, uint32_t c3, int j) {
    double n0, n1;
    normal2(philox4x32(key, (uint32_t)((j >> 1) & ((D + 1) / 2 - 1)), c1, c2, c3), n0, n1);
    return (j & 1) ? n1 : n0;
}

// The five lgamma/digamma evaluations of one PMD position, x = {k + alpha, N - k + beta, N + phi, alpha, beta}
// (mdg_common.cuh lgam_digam_batch), returning what the log-likelihood needs: d14 = lgamma(x0) - lgamma(x3),
// d25 = lgamma(x1) - lgamma(x4), l3 = lgamma(x2) and the five digammas. The x < 10 shifts are organised by how
// often they happen: alpha = D phi (and with it k + alpha at low counts) is below 10 for some lane of the warp on
// most trips, the other three arguments almost never (phi < 10 or a handful of reads). So ONE branch covers the
// pair (x0, x3) and takes a single logarithm for both, log(P(x3) / P(x0)) — the two -log P(x) corrections enter
// d14 with opposite signs — and one more, rarely taken, covers the rest. (ncu, r2m capture: the five separate
// per-argument blocks were 13 % of the executed instructions at 10-17 active lanes.)
__device__ __forceinline__ void pmd_special(const double (&x)[5], double& d14, double& d25, double& l3, double (&dg)[5]) {
    bool small[5];
    double y[5], t[5], lg[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        small[i] = x[i] < 10.0;
        y[i] = x[i] + (small[i] ? 10.0 : 0.0);
        t[i] = rcp_pos(y[i]);
    }
#pragma unroll
    for (int i = 0; i < 5; ++i) stirling(y[i], t[i], lg[i], dg[i]);
    d14 = lg[0] - lg[3];
    if (small[0] | small[3]) {
        double P0, Q0, P3, Q3;
        shift_poly10(x[0], P0, Q0);
        shift_poly10(x[3], P3, Q3);
        P0 = small[0] ? P0 : 1.0; Q0 = small[0] ? Q0 : 0.0;
        P3 = small[3] ? P3 : 1.0; Q3 = small[3] ? Q3 : 0.0;
        const double r0 = rcp_pos(P0), r3 = rcp_pos(P3);
        // P3 <= P0 <= 3.4e11; the quotient leaves the normal range only for alpha < 1e-290 (|u_c| > 660)
        d14 += (P3 > 1e-280) ? log_pos(P3 * r0) : (log_pos(P3) - log_pos(P0));
        dg[0] = fma(-Q0, r0, dg[0]);
        dg[3] = fma(-Q3, r3, dg[3]);
    }
    if (small[1] | small[2] | small[4]) {
        const int idx[3] = {1, 2, 4};
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const int i = idx[m];
            if (small[i]) {
                double P, Q;
                shift_poly10(x[i], P, Q);
                lg[i] -= log_pos(P);
                dg[i] = fma(-Q, rcp_pos(P), dg[i]);
            }
        }
    }
    d25 = lg[1] - lg[4];
    l3 = lg[2];
}

enum GroupPhase : int { GP_FETCH = 0, GP_INIT = 1, GP_HEUR = 2, GP_LEAF = 3, GP_IDLE = 4 };
// What a leapfrog's bookkeeping leaves for the end of the trip, where each of these routines exists once (inlined at
// every place that wants it, they made the kernel outgrow the instruction cache). Each step falls through to the
// next one as far as it has to: a heuristic search that ends starts a transition, a transition starts a doubling.
enum PendingStep : int {
    PS_NONE = 0,
    PS_HEUR_BEGIN = 1,  // start the step-size search (hmc_util.find_reasonable_step_size) at eps
    PS_HEUR = 2,        // its next trial, or its end: eps = the step found, reset dual averaging, start a transition
    PS_RESET = 3,       // reset dual averaging, then start a transition
    PS_TRANSITION = 4,  // begin a transition from the chain state held in sh.zp / sh.gp / pe_cur
    PS_DOUBLING = 5     // start one tree doubling: pick direction, aim the next leapfrog at the chosen edge
};

// bytes of dynamic shared memory per warp: {k, N} as doubles + four log-likelihood buffers, [n_slots][32] each
__host__ __device__ constexpr size_t nuts_warp_smem_bytes(int n_slots) { return (size_t)n_slots * 32 * (16 + 4 * 8); }

// roles of the four log-likelihood buffers, 2 bits each: scratch (the evaluation writes here), subtree
// proposal, tree proposal, current state
struct LlRoles {
    unsigned v;
    __device__ __forceinline__ unsigned get(int f) const { return (v >> (2 * f)) & 3u; }
    __device__ __forceinline__ void swap(int f, int g) {
        const unsigned a = get(f), b = get(g);
        v = (v & ~((3u << (2 * f)) | (3u << (2 * g)))) | (b << (2 * f)) | (a << (2 * g));
    }
};
enum : int { LL_X = 0, LL_SUB = 1, LL_MAIN = 2, LL_CUR = 3 };

// K2: log p(y | theta(u)) + log prior(theta(u)) + log |d theta / d u| and its gradient for the chain of one
// group; writes the per-position log-likelihood (without log C(N,k)) of every linear index to `llw`.
// `myu` and `grad` are the lane's component jc of u and of the gradient (the layout of nuts_group_kernel).
template <int MODEL, int GW>
__device__ __forceinline__ void eval_group(const double2* __restrict__ kn, double* __restrict__ llw, int n_slots, int lane,
                                           int lig, int jc, unsigned gmask, int P, int mask, int n_obs, double myu,
                                           const double2* __restrict__ ptab, double phi_min, double& logp, double& grad,
                                           bool& valid) {
    constexpr int D = ModelDim<MODEL>::value;
    // --- group-uniform transforms, one parameter per lane, then broadcast (mdg_model.cuh eval_model) ---
    const bool in_range = fabs(myu) < 700.0;  // false for NaN
    const double E = exp_core(lig == D - 1 ? myu : -fabs(myu));
    const double l1p = log_pos(1.0 + E);
    const double inv = rcp_pos(1.0 + E);
    const double sp = fmax(myu, 0.0) + l1p;          // softplus(u)
    const double sg = (myu >= 0.0) ? inv : E * inv;  // sigmoid(u)
    const double2 c01 = ptab[lig], c23 = ptab[32 + lig];
    const double lp_lane = fma(c23.y, E, fma(c23.x, sp, fma(c01.y, myu, c01.x)));
    const double gp_lane = fma(c23.y, E, fma(c23.x, sg, c01.y));
    const double q = __shfl_sync(gmask, sg, 0, GW);
    const double log1mq = -__shfl_sync(gmask, sp, 0, GW);
    const double delta = __shfl_sync(gmask, E, D - 1, GW);
    double A = 0.0, c = 0.0;
    if (MODEL == 0) {
        A = __shfl_sync(gmask, sg, 1, GW);
        c = __shfl_sync(gmask, sg, 2, GW);
    }
    const double phi = delta + phi_min;

    // --- positions: rolled loop over the slots -----------------------------------------------------
    double s_ll = lp_lane, s_dD = 0.0, s_dDw = 0.0, s_dDxw = 0.0, s_dphi = 0.0;
    double lgphi = 0.0, dgphi = 0.0, lga0 = 0.0, dga0 = 0.0, lgb0 = 0.0, dgb0 = 0.0;
    bool bad = !in_range;
#pragma unroll 1
    for (int s = 0; s < n_slots; ++s) {
        const double2 d = kn[s * 32 + lane];  // {k, N}; {0, 0} for the spare and the padding
        const int j = s * GW + lig - 1;
        int xi = (mask == 0 && j >= P) ? j - P : j;
        xi = ((unsigned)j < (unsigned)n_obs) ? xi : 0;  // spare / padding: position 0 (never adds an invalid D)
        const double x = (double)xi;
        double w = 1.0, Dv = q;
        if (MODEL == 0) {
            w = exp_nonpos(x * log1mq);
            Dv = fma(A, w, c);
        }
        const bool ok = (Dv > 0.0) && (Dv < 1.0);  // clip(Dz, 0, 1) reached (fits.py:50): NaN in the reference
        bad |= !ok;
        Dv = ok ? Dv : 0.5;
        const double al = Dv * phi, be = (1.0 - Dv) * phi;
        double lls, ga, gb;
        if (MODEL == 0) {
            const double xs[5] = {d.x + al, d.y - d.x + be, d.y + phi, al, be};
            double d14, d25, l3v, d5[5];
            pmd_special(xs, d14, d25, l3v, d5);
            if (s == 0) {  // the spare (index 0, k = N = 0) has just evaluated lgamma(phi), digamma(phi)
                lgphi = __shfl_sync(gmask, l3v, 0, GW);
                dgphi = __shfl_sync(gmask, d5[2], 0, GW);
            }
            // differences first: the terms of an index with k = N = 0 vanish (to 1e-16: the shared logarithm of
            // d14 sees P(x3) / P(x0) = 1 up to rounding), so the spare and the padding need no masking
            lls = d14 + d25 - (l3v - lgphi);
            const double dgN = d5[2] - dgphi;
            ga = (d5[0] - d5[3]) - dgN;
            gb = (d5[1] - d5[4]) - dgN;
        } else {
            const double xs[3] = {d.x + al, d.y - d.x + be, d.y + phi};
            double l3[3], d3[3];
            lgam_digam_batch<3>(xs, gmask, l3, d3);
            if (s == 0) {  // spare: lgamma/digamma of alpha, beta, phi (position independent in the null model)
                lga0 = __shfl_sync(gmask, l3[0], 0, GW); dga0 = __shfl_sync(gmask, d3[0], 0, GW);
                lgb0 = __shfl_sync(gmask, l3[1], 0, GW); dgb0 = __shfl_sync(gmask, d3[1], 0, GW);
                lgphi = __shfl_sync(gmask, l3[2], 0, GW); dgphi = __shfl_sync(gmask, d3[2], 0, GW);
            }
            lls = (l3[0] - lga0) + (l3[1] - lgb0) - (l3[2] - lgphi);
            const double dgN = d3[2] - dgphi;
            ga = (d3[0] - dga0) - dgN;
            gb = (d3[1] - dgb0) - dgN;
        }
        llw[s * 32 + lane] = lls;
        const double dD = phi * (ga - gb);
        s_ll += lls;
        s_dD += dD;
        s_dphi += fma(Dv, ga - gb, gb);  // D*ga + (1-D)*gb
        if (MODEL == 0) {
            const double dw = dD * w;
            s_dDw += dw;
            s_dDxw = fma(dw, x, s_dDxw);
        }
    }
    s_ll = group_sum<GW>(s_ll, gmask);
    s_dD = group_sum<GW>(s_dD, gmask);
    s_dphi = group_sum<GW>(s_dphi, gmask);
    if (MODEL == 0) {
        s_dDw = group_sum<GW>(s_dDw, gmask);
        s_dDxw = group_sum<GW>(s_dDxw, gmask);
    }

    // --- chain rule to the unconstrained parameters: component jc of the gradient ---------------------
    logp = s_ll;
    double dlogp_dtheta, dtheta_du;
    if (MODEL == 0) {
        dtheta_du = jc == 0 ? -A * q : (jc == 1 ? A * (1.0 - A) : (jc == 2 ? c * (1.0 - c) : delta));
        dlogp_dtheta = jc == 0 ? s_dDxw : (jc == 1 ? s_dDw : (jc == 2 ? s_dD : s_dphi));
    } else {
        dtheta_du = jc == 0 ? q * (1.0 - q) : delta;
        dlogp_dtheta = jc == 0 ? s_dD : s_dphi;
    }
    grad = fma(dtheta_du, dlogp_dtheta, __shfl_sync(gmask, gp_lane, jc, GW));
    // a lane >= D mirrors component 0, so a vote over the whole group sees every component once
    const bool any_bad = (__ballot_sync(gmask, bad || !isfinite(grad)) & gmask) != 0u;
    valid = isfinite(logp) && !any_bad;
}

// ---- the cold paths of nuts_group_kernel, out of line ----------------------------------------------------------
// Once per chain (start, initial point, end), once per adaptation window, the step-size heuristic, fallbacks that
// never run at the default configuration, and the optional stores. Called from the loop body, they leave a call
// there instead of their code, so the warm code (leapfrog, leaf, subtree end, transition end, transition start,
// doubling) is one contiguous block of SASS (tools/sass_layout.py; profiles/r06_nuts_code_layout.md). Each does the
// operations the inlined code did on the same operands in the same order; a call passes values exactly. They read
// the launch's parameters in place (`p` is a __grid_constant__ kernel parameter).
template <int D>  // layout: cold
__device__ MDG_COLD void reset_dual_averaging(GroupShared<D>& sh) {
    sh.da_x = 0.0; sh.da_xavg = 0.0; sh.da_gavg = 0.0; sh.da_t = 0; sh.da_prox = log_cold(10.0 * sh.eps);
}

// the next (TaxID, run) item of a group: {k, N} of the run into the warp's slots, the WAIC accumulators and the chain
// state in shared memory cleared; returns {TaxID index, run mask, Philox key}. Inlined: as a call (in either form,
// with or without the key) it made ptxas spill the phase across the whole leapfrog loop (4 B stored and loaded per
// trip in the PMD kernel); inlined, its code still lies ahead of the loop, outside the warm block.
template <int MODEL, int GW, int D>
__device__ __forceinline__ int4 chain_start(const FitLaunch& p, GroupShared<D>& sh, unsigned item, double2* kn, double* wacc, int lane,
                                     int lig, unsigned gmask) {
    const int P = p.P, NS = p.n_slots;
    const size_t wstride = (size_t)NS * 32;
    int tax, mask;
    {
        const unsigned prio = 2u * (unsigned)p.n_prio, n_all = (unsigned)p.n_items_all;
        const bool is_all = item >= prio && item < prio + n_all;
        const unsigned w = is_all ? item - prio : (item < prio ? item : item - n_all);  // half runs: 2 * position + strand
        const unsigned q = is_all ? w : (w >> 1);  // queue position of the TaxID
        tax = p.order != nullptr ? __ldg(p.order + q) : (int)q;
        mask = is_all ? 0 : 1 + (int)(w & 1u);
    }
    const int run_kind = mask * 2 + MODEL;
    const int n_obs = mask == 0 ? 2 * P : P;
    const uint2 key = make_key(p.cfg.seed, p.tax_id[tax]);
    if (p.chain_clock != nullptr && lig == 0) p.chain_clock[((size_t)tax * MDG_NUM_RUNS + run_kind) * 2] = global_timer_ns();
    const uint32_t* kk = p.k + (size_t)tax * 2 * P + (mask == 2 ? P : 0);
    const uint32_t* NN = p.N + (size_t)tax * 2 * P + (mask == 2 ? P : 0);
#pragma unroll 1
    for (int s = 0; s < NS; ++s) {
        const int j = s * GW + lig - 1;
        const bool a = (unsigned)j < (unsigned)n_obs;
        kn[s * 32 + lane] = make_double2(a ? (double)__ldg(kk + j) : 0.0, a ? (double)__ldg(NN + j) : 0.0);
        wacc[0 * wstride + s * 32] = -INFINITY;  // running max of the streaming log-sum-exp
        wacc[1 * wstride + s * 32] = 0.0;        // its sum
        wacc[2 * wstride + s * 32] = 0.0;        // Welford mean
        wacc[3 * wstride + s * 32] = 0.0;        // Welford M2
    }
    __syncwarp(gmask);
    if (lig < D) { sh.imm[lig] = 1.0; sh.isd[lig] = 1.0; sh.wf_mean[lig] = 0.0; sh.wf_m2[lig] = 0.0; }
    sh.E0 = 0.0; sh.s_weight = 0.0; sh.s_sum_acc = 0.0;
    sh.eps = p.cfg.init_step_size; sh.pe_cur = 0.0;
    sh.da_x = 0.0; sh.da_xavg = 0.0; sh.da_gavg = 0.0; sh.da_prox = 0.0; sh.da_t = 0; sh.wf_n = 0; sh.window_idx = 0;
    sh.mean_accept = 0.0; sh.n_div = 0u;
    sh.m_weight = 0.0; sh.m_sum_acc = 0.0; sh.m_pe_p = 0.0; sh.u_main = 0.0; sh.m_nprop = 0; sh.s_pe_p = 0.0;
    sh.h_step = 0.0; sh.h_Er = 0.0; sh.h_last = 0; sh.h_dir = 0; sh.h_att = 0u; sh.h_call = 0u; sh.init_attempt = 0u;
    if (lig == 0) {
#pragma unroll
        for (int j = 0; j < 5; ++j) { sh.acc_mean[j] = 0.0; sh.acc_m2[j] = 0.0; }
    }
    __syncwarp(gmask);
    return make_int4(tax, mask, (int)key.x, (int)key.y);
}

// init_to_uniform(radius): component jc of the initial-point candidate number `attempt` (component j is the (j % 2)-th
// uniform of the Philox block j / 2)
__device__ MDG_COLD double init_position(const FitLaunch& p, uint2 key, int jc, uint32_t attempt, int run_kind) {
    double u0, u1;
    uniform2(philox4x32(key, (uint32_t)(jc >> 1), attempt, c2word(run_kind, P_INIT), 0u), u0, u1);
    return p.cfg.init_radius * (2.0 * ((jc & 1) ? u1 : u0) - 1.0);
}

// sqrt(t) and t^-0.75 of the dual averaging past the launch's tables
__device__ MDG_COLD double da_sqrt_cold(int t) { return sqrt((double)t); }
__device__ MDG_COLD double da_pow_cold(int t) { return exp_cold(-0.75 * log_cold((double)t)); }

// end of a middle adaptation window: the regularised variance of the window's draws becomes the mass matrix diagonal
// (warmup_adapter); returns whether the step-size heuristic runs next (else dual averaging restarts here)
template <int D>
__device__ MDG_COLD bool window_end(const FitLaunch& p, GroupShared<D>& sh, int lig, unsigned gmask) {
    __syncwarp(gmask);
    if (lig < D) {
        const int wf_n = sh.wf_n;
        const double cov = sh.wf_m2[lig] / (wf_n - 1);
        const double v = ((double)wf_n / (wf_n + 5.0)) * cov + 1e-3 * (5.0 / (wf_n + 5.0));
        sh.imm[lig] = v;
        sh.isd[lig] = 1.0 / sqrt(v);
        sh.wf_mean[lig] = 0.0; sh.wf_m2[lig] = 0.0;
    }
    __syncwarp(gmask);
    sh.wf_n = 0;
    const bool want_heur = p.cfg.find_heuristic_step_size != 0;
    if (!want_heur) reset_dual_averaging(sh);
    return want_heur;
}

// hmc_util.find_reasonable_step_size. heur_record: the direction of the trial just evaluated. heur_next (at `begin`:
// first sets up the search at eps): its next trial, returned as {momentum component jc, 1} (the leapfrog starts from
// the chain state with step h_step), or its end, {0, 0}, with eps = the step found.
template <int D, int GW>
__device__ MDG_COLD void heur_record(GroupShared<D>& sh, int jc, double rn, double pen, unsigned gmask) {
    const double log_target_heur = -0.22314355131420976;  // log(0.8)
    const double delta = (kinetic<D, GW>(sh.imm[jc], rn, gmask) + pen) - sh.h_Er;
    const int dir_new = (log_target_heur < -delta) ? 1 : -1;  // NaN -> -1
    sh.h_last = sh.h_dir;
    sh.h_dir = dir_new;
}

template <int D, int GW>
__device__ MDG_COLD double2 heur_next(GroupShared<D>& sh, bool begin, uint2 key, int run_kind, int jc, unsigned gmask) {
    if (begin) { sh.h_step = sh.eps; sh.h_last = 0; sh.h_dir = 0; sh.h_att = 0; }
    const double h_step = sh.h_step;
    const int h_dir = sh.h_dir, h_last = sh.h_last;
    const bool small_ok = (h_step > 2.2250738585072014e-308) || (h_dir >= 0);
    const bool large_ok = (h_step < 1.7976931348623157e308) || (h_dir <= 0);
    if (small_ok && large_ok && (h_last == 0 || h_dir == h_last)) {
        sh.h_step = h_step * (h_dir > 0 ? 2.0 : (h_dir < 0 ? 0.5 : 1.0));
        const double rf = draw_normal_lane_cold<D>(key, sh.h_call, c2word(run_kind, P_HEUR), sh.h_att, jc) * sh.isd[jc];
        ++sh.h_att;
        sh.h_Er = kinetic<D, GW>(sh.imm[jc], rf, gmask) + sh.pe_cur;
        return make_double2(rf, 1.0);
    }
    sh.eps = h_step;
    return make_double2(0.0, 0.0);
}

// the optional outputs: the chain's trace (one value per lane < 4) and the kept constrained draw
__device__ MDG_COLD void store_trace(const FitLaunch& p, int tax, int run_kind, int t, int lig, double v) {
    p.trace[(((size_t)tax * MDG_NUM_RUNS + run_kind) * (p.cfg.num_warmup + p.cfg.num_samples) + t) * 4 + lig] = v;
}

__device__ MDG_COLD void store_sample(const FitLaunch& p, int tax, int slot, int si, double th0, double th1, double th2, double th3) {
    double* dst = p.samples + (((size_t)tax * p.sample_runs + slot) * p.cfg.num_samples + si) * 4;
    dst[0] = th0; dst[1] = th1; dst[2] = th2; dst[3] = th3;
}

// a finished chain: per-position lppd / pWAIC (with log C(N,k)) and the run record
template <int GW, int D>
__device__ MDG_COLD void chain_end(const FitLaunch& p, GroupShared<D>& sh, const double2* kn, const double* wacc, int tax, int run_kind,
                                   int mask, int n_obs, int ns, int failed, uint32_t n_grad, int lane, int lig, unsigned gmask) {
    const int P = p.P, S = p.cfg.num_samples;
    const size_t wstride = (size_t)p.n_slots * 32;
    double waic_sum = 0.0, lppd_sum = 0.0;
    const size_t R = 2 * (size_t)P;
    double* wout = p.waic + ((size_t)tax * MDG_NUM_RUNS + run_kind) * 2 * R;
#pragma unroll 1
    for (int s = 0; s < ns; ++s) {
        const int j = s * GW + lig - 1;
        if ((unsigned)j < (unsigned)n_obs && !failed && S > 0) {
            const double2 d = kn[s * 32 + lane];
            const double logC = lgam(d.y + 1.0) - lgam(d.x + 1.0) - lgam(d.y - d.x + 1.0);  // log C(N,k)
            const int dense = (mask == 2 ? P : 0) + j;
            const double lppd_i = logC + wacc[0 * wstride + s * 32] + log_cold(wacc[1 * wstride + s * 32]) - log_cold((double)S);
            const double pw_i = wacc[3 * wstride + s * 32] / (double)S;
            wout[dense] = lppd_i;
            wout[R + dense] = pw_i;
            lppd_sum += lppd_i;
            waic_sum += -2.0 * (lppd_i - pw_i);
        }
    }
    waic_sum = group_sum<GW>(waic_sum, gmask);
    lppd_sum = group_sum<GW>(lppd_sum, gmask);
    __syncwarp(gmask);
    if (lig == 0) {
        RunRecord& r = p.rec[(size_t)tax * MDG_NUM_RUNS + run_kind];
        r.step_size = sh.eps;
        r.mean_accept = sh.mean_accept;
        r.n_leapfrog = n_grad;
        r.n_divergent = sh.n_div;
        r.waic = waic_sum;
        r.lppd = lppd_sum;
#pragma unroll
        for (int j = 0; j < 5; ++j) { r.mean[j] = sh.acc_mean[j]; r.sd[j] = S > 0 ? sqrt(sh.acc_m2[j] / (double)S) : 0.0; }
        r.failed = (uint32_t)failed;
        r.pad = 0;
        if (p.chain_clock != nullptr) p.chain_clock[((size_t)tax * MDG_NUM_RUNS + run_kind) * 2 + 1] = global_timer_ns();
    }
    __syncwarp(gmask);
}

#ifndef MDG_NUTS_MINBLOCKS
#define MDG_NUTS_MINBLOCKS 4  // CTAs of four warps per SM: 128 registers per thread, 16 warps per SM (3 / 5 / 6 were measured slower: profiles/r01_nuts_tuning.md)
#endif
template <int MODEL, int GW, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, MDG_NUTS_MINBLOCKS * 4 / WARPS) nuts_group_kernel(__grid_constant__ const FitLaunch p) {  // layout: setup
    constexpr int D = ModelDim<MODEL>::value;
    constexpr int GROUPS = 32 / GW;
    // one lane per component (the lane-order sums of kinetic / is_turning) and one per trace column
    static_assert(GW >= D && GW >= 4, "a group needs a lane for each of the D parameters and each of the 4 trace columns");
    __shared__ GroupShared<D> sh_all[WARPS * GROUPS];
    __shared__ double2 sh_prior[64];
    extern __shared__ __align__(16) unsigned char sh_dyn[];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane / GW, lig = lane % GW;
    // The chain's D-vectors are held one component per lane: lane lig < D of the group owns component lig; a lane
    // lig >= D mirrors component 0 (the evaluation needs a valid parameter on every lane) and never stores it.
    const bool own = lig < D;
    const int jc = own ? lig : 0;
    const unsigned gmask = group_mask<GW>();
    GroupShared<D>& sh = sh_all[warp * GROUPS + grp];
    const int NS = p.n_slots;
    unsigned char* wbase = sh_dyn + (size_t)warp * nuts_warp_smem_bytes(NS);
    double2* const kn = reinterpret_cast<double2*>(wbase);                        // [NS][32]
    double* const llb = reinterpret_cast<double*>(wbase + (size_t)NS * 32 * 16);  // [4][NS][32]
    // WAIC accumulators of this lane (touched once per kept draw): global scratch, [4][NS][32] per warp
    // (the address is recomputed where it is used — chain start, kept draw, chain end — instead of being carried
    // through the leapfrog loop in two registers)
    auto wacc_of_lane = [&]() { return p.waic_acc + ((size_t)blockIdx.x * WARPS + warp) * 4 * (size_t)NS * 32 + lane; };
    const size_t wstride = (size_t)NS * 32;

    const int W = p.cfg.num_warmup, S = p.cfg.num_samples, P = p.P;
    const int max_depth = p.cfg.max_tree_depth < kMaxTreeDepth ? p.cfg.max_tree_depth : kMaxTreeDepth;
    const uint32_t budget = p.cfg.max_leapfrogs_per_run > 0 ? (uint32_t)p.cfg.max_leapfrogs_per_run : 0u;
    log_table_init();
    prior_table_init<MODEL>(sh_prior, p.pr, 1);
    const double phi_min = p.pr.phi_min;

    // ---- per-chain state in registers (group-uniform) ----
    int phase = GP_FETCH;
    int tax = 0, mask = 0, run_kind = 0, n_obs = 0;
    int ns = 0;  // rounds of the position loop of THIS chain (<= NS, the launch's layout)
    uint2 key = make_uint2(0u, 0u);
    LlRoles roles;
    roles.v = 0xE4u;  // identity: role f -> buffer f
    bool m_is_c = true;
    uint32_t n_grad = 0;
    int failed = 0;
    int m_depth = 0;
    bool m_turning = false, m_div = false, going_right = true;
    int s_nprop = 0;
    bool s_div = false;
    uint32_t leaf_counter = 0;
    double zf = 0.0, rf = 0.0, gf = 0.0, e = 0.0;  // leapfrog source (component jc)
    int t = 0;

    // ---- cold chain state: references into shared memory (scalars: single writer or all lanes writing the same
    // value at a converged point, reads are broadcasts; D-vectors: lane j < D writes component j) ----
    double& E0 = sh.E0; double& s_weight = sh.s_weight; double& s_sum_acc = sh.s_sum_acc;
    double& eps = sh.eps; double& pe_cur = sh.pe_cur;
    double& da_x = sh.da_x; double& da_xavg = sh.da_xavg; double& da_gavg = sh.da_gavg; double& da_prox = sh.da_prox;
    int& da_t = sh.da_t; int& wf_n = sh.wf_n; int& window_idx = sh.window_idx;
    double& mean_accept = sh.mean_accept; uint32_t& n_div = sh.n_div;
    double& m_weight = sh.m_weight; double& m_sum_acc = sh.m_sum_acc; double& m_pe_p = sh.m_pe_p; double& u_main = sh.u_main;
    int& m_nprop = sh.m_nprop; double& s_pe_p = sh.s_pe_p;
    double& h_step = sh.h_step; uint32_t& h_call = sh.h_call; uint32_t& init_attempt = sh.init_attempt;

    for (;;) {  // layout: head
        // ================= a group without a chain pulls the next (TaxID, run) item =================
        if (phase == GP_FETCH) {  // layout: fetch
            unsigned item = 0u;
            if (lig == 0) item = atomicAdd(p.work_counter, 1u);
            item = __shfl_sync(gmask, item, 0, GW);
            if (item >= (unsigned)p.n_items) {
                phase = GP_IDLE;
            } else {
                const int4 c = chain_start<MODEL, GW, D>(p, sh, item, kn, wacc_of_lane(), lane, lig, gmask);
                tax = c.x;
                mask = c.y;
                key = make_uint2((uint32_t)c.z, (uint32_t)c.w);
                run_kind = mask * 2 + MODEL;
                n_obs = mask == 0 ? 2 * P : P;
                ns = (n_obs + GW) / GW;  // index 0 is the spare
                roles.v = 0xE4u;
                m_is_c = true;
                n_grad = 0; failed = 0; m_depth = 0; m_turning = false; m_div = false; going_right = true;
                s_nprop = 0; s_div = false; leaf_counter = 0; t = 0;
                zf = init_position(p, key, jc, 0u, run_kind);
                rf = 0.0; gf = 0.0; e = 0.0;
                phase = GP_INIT;
            }
        }
        // layout: head
        if (__all_sync(0xffffffffu, phase == GP_IDLE)) break;
        if (phase == GP_IDLE) continue;

        // =========================== one leapfrog ===========================
        bool done = false;
        {
            int pend = PS_NONE;
            const double imm = sh.imm[jc];
            const double rh = fma(-0.5 * e, gf, rf);
            const double zn = fma(e * imm, rh, zf);
            double logp, grad;
            bool valid;
            eval_group<MODEL, GW>(kn, llb + (size_t)roles.get(LL_X) * wstride, ns, lane, lig, jc, gmask, P, mask, n_obs, zn, sh_prior,
                                  phi_min, logp, grad, valid);
            ++n_grad;
            const double pen = valid ? -logp : nan("");
            const double gn = valid ? -grad : nan("");
            const double rn = fma(-0.5 * e, gn, rh);

            if (budget != 0u && n_grad > budget) {
                // bounded work per run: the analogue of the reference's per-fit timeout (fits.py:472-474)
                failed = 2;
                done = true;
            } else if (phase == GP_LEAF) {  // layout: leaf
                // ---- hmc_util._build_basetree ----
                double dE = pen + kinetic<D, GW>(sh.imm[jc], rn, gmask) - E0;
                if (isnan(dE)) dE = INFINITY;
                const double leaf_w = -dE;
                const bool leaf_div = dE > p.cfg.max_delta_energy;
                const double leaf_acc = dE <= 0.0 ? 1.0 : exp_nonpos(-dE);  // min(1, e^-dE); dE is never NaN here
                const int leaf_idx = s_nprop;
                bool take;
                double s_rsum;  // component jc of the subtree's momentum sum
                if (leaf_idx == 0) {
                    take = true;
                    s_weight = leaf_w;
                    s_sum_acc = leaf_acc;
                    s_rsum = rn;
                } else {
                    // ---- _combine_tree(..., biased_transition=False) ----
                    double us, unused;
                    uniform2(philox4x32(key, leaf_counter, (uint32_t)t, c2word(run_kind, P_SUB), 0u), us, unused);
                    // expit(d) and logaddexp share one exponential: e = exp(-|d|)
                    const double dlt = leaf_w - s_weight;
                    const double ed = exp_nonpos(-fabs(dlt));  // NaN -> ~0 -> take = false
                    const double inv = rcp_pos(1.0 + ed);
                    const double prob = dlt >= 0.0 ? inv : ed * inv;
                    take = us < prob;  // NaN -> false
                    s_weight = isnan(dlt) ? -INFINITY : fmax(s_weight, leaf_w) + log_pos(1.0 + ed);
                    s_sum_acc += leaf_acc;
                    s_rsum = sh.s_rsum[jc] + rn;
                }
                s_div = leaf_div;
                s_nprop = leaf_idx + 1;
                ++leaf_counter;
                if (take) {
                    s_pe_p = pen;
                    roles.swap(LL_X, LL_SUB);  // the leaf's log-likelihoods become the subtree proposal's
                }
                // checkpoint indices (_leaf_idx_to_ckpt_idxs)
                const int idx_max = __popc((unsigned)leaf_idx >> 1);
                const int n_trail = __ffs(~(unsigned)leaf_idx) - 1;
                const int idx_min = idx_max - n_trail + 1;
                __syncwarp(gmask);
                if (own) {
                    sh.s_rsum[lig] = s_rsum;
                    if (take) { sh.szp[lig] = zn; sh.sgp[lig] = gn; }
                    if ((leaf_idx & 1) == 0) { sh.rck[idx_max][lig] = rn; sh.rsck[idx_max][lig] = s_rsum; }
                }
                __syncwarp(gmask);
                bool turning = false;
                if (leaf_idx & 1) {
                    // ---- _is_iterative_turning ----
                    for (int i = idx_max; i >= idx_min && !turning; --i) {
                        const double rc = sh.rck[i][jc];
                        turning = is_turning<D, GW>(sh.imm[jc], rc, rn, s_rsum - sh.rsck[i][jc] + rc, gmask);
                    }
                }
                if (s_nprop < (1 << m_depth) && !turning && !s_div) {
                    // keep extending the subtree from the leaf just built
                    zf = zn; rf = rn; gf = gn;
                } else {  // layout: subtree_end
                    // ---- subtree finished: _combine_tree(..., biased_transition=True) ----
                    const double dlt_m = s_weight - m_weight;
                    // min(1, e^d) and logaddexp share one exponential e^-|d| (u_main < 1, so a
                    // probability above 1 acts as 1; NaN -> ~0 -> false)
                    const double em = exp_nonpos(-fabs(dlt_m));
                    const double prob = (turning || s_div) ? 0.0 : (dlt_m >= 0.0 ? 1.0 : em);
                    const bool take_main = u_main < prob;
                    const double m_rsum = sh.m_rsum[jc] + s_rsum;
                    __syncwarp(gmask);
                    if (own) {
                        if (going_right) { sh.zr[lig] = zn; sh.rr[lig] = rn; sh.gr[lig] = gn; }
                        else { sh.zl[lig] = zn; sh.rl[lig] = rn; sh.gl[lig] = gn; }
                        if (take_main) { sh.zp[lig] = sh.szp[lig]; sh.gp[lig] = sh.sgp[lig]; }
                        sh.m_rsum[lig] = m_rsum;
                    }
                    __syncwarp(gmask);  // the owners are back before anybody reads the tree edges
                    m_turning = turning || is_turning<D, GW>(sh.imm[jc], sh.rl[jc], sh.rr[jc], m_rsum, gmask);
                    if (take_main) {
                        m_pe_p = s_pe_p;
                        roles.swap(LL_SUB, LL_MAIN);
                        m_is_c = false;
                    }
                    m_depth += 1;
                    // logaddexp(m_weight, s_weight) = max + log(1 + e^-|d|)
                    m_weight = isnan(dlt_m) ? -INFINITY : fmax(m_weight, s_weight) + log_pos(1.0 + em);
                    m_div = s_div;
                    m_sum_acc += s_sum_acc;
                    m_nprop += s_nprop;
                    if (m_depth < max_depth && !m_turning && !m_div) {
                        pend = PS_DOUBLING;
                    } else {  // layout: transition_end
                        // ================= transition finished (hmc.py sample_kernel) =================
                        const double accept_prob = m_sum_acc * rcp_pos((double)m_nprop);
                        pe_cur = m_pe_p;
                        if (!m_is_c) roles.swap(LL_MAIN, LL_CUR);
                        __syncwarp(gmask);
                        const double zc = sh.zp[jc];
                        bool want_heur = false;
                        if (t < W) {  // layout: adapt
                            // ---- warmup_adapter.update_fn ----
                            da_t += 1;
                            const double inv_t10 = rcp_pos((double)(da_t + 10));
                            da_gavg = (1.0 - inv_t10) * da_gavg + (p.cfg.target_accept - accept_prob) * inv_t10;
                            // sqrt(t) / gamma and t^-kappa (gamma = 0.05, kappa = 0.75) from the launch's tables (host libm)
                            const bool tab = da_t < kDaTable;
                            const double sq_t = tab ? __ldg(p.da_sqrt + da_t) : da_sqrt_cold(da_t);
                            da_x = da_prox - sq_t * 20.0 * da_gavg;
                            const double wt = tab ? __ldg(p.da_pow + da_t) : da_pow_cold(da_t);
                            da_xavg = (1.0 - wt) * da_xavg + wt * da_x;
                            eps = exp_cold((t == W - 1) ? da_xavg : da_x);
                            eps = fmax(eps, 2.2250738585072014e-308);
                            const bool is_middle = (0 < window_idx) && (window_idx < p.n_windows - 1);
                            if (is_middle) {
                                wf_n += 1;
                                if (own) {
                                    const double inv_wf = rcp_pos((double)wf_n);
                                    const double dpre = zc - sh.wf_mean[lig];
                                    const double mn = sh.wf_mean[lig] + dpre * inv_wf;
                                    sh.wf_mean[lig] = mn;
                                    sh.wf_m2[lig] += dpre * (zc - mn);
                                }
                                __syncwarp(gmask);
                            }
                            const bool at_end = (t == p.win_end[window_idx]);
                            __syncwarp(gmask);  // every lane has read window_idx before it moves
                            if (at_end) window_idx += 1;
                            if (at_end && is_middle) want_heur = window_end(p, sh, lig, gmask);
                        } else {  // layout: kept_draw
                            // ---- after warm-up: keep the draw ----
                            const int si = t - W;
                            const double inv_n = rcp_pos((double)(si + 1));
                            mean_accept += (accept_prob - mean_accept) * inv_n;
                            if (m_div) ++n_div;
                            // constrained draw (q, A, c, phi): lane j < D transforms parameter j, then a broadcast
                            double th[4];
                            {
                                const double myu = zc;
                                const double Ev = exp_fast_split(lig == D - 1 ? myu : -fabs(myu));
                                const double iv = rcp_pos(1.0 + Ev);
                                const double val = (lig == D - 1) ? Ev + p.pr.phi_min : (myu >= 0.0 ? iv : Ev * iv);
                                th[0] = __shfl_sync(gmask, val, 0, GW);
                                th[1] = MODEL == 0 ? __shfl_sync(gmask, val, 1, GW) : nan("");
                                th[2] = MODEL == 0 ? __shfl_sync(gmask, val, 2, GW) : nan("");
                                th[3] = __shfl_sync(gmask, val, D - 1, GW);
                            }
                            if (lig == 0) {
                                const double v[5] = {th[0], th[3], MODEL == 0 ? th[1] + th[2] : th[0], th[1], th[2]};
#pragma unroll
                                for (int j = 0; j < 5; ++j) {
                                    double dpre = v[j] - sh.acc_mean[j];
                                    double mn = sh.acc_mean[j] + dpre * inv_n;
                                    sh.acc_mean[j] = mn;
                                    sh.acc_m2[j] += dpre * (v[j] - mn);
                                }
                                const int slot = p.sample_slot[run_kind];
                                if (p.samples != nullptr && slot >= 0) store_sample(p, tax, slot, si, th[0], th[1], th[2], th[3]);
                            }
                            __syncwarp(gmask);
                            // WAIC: streaming logsumexp + Welford of this lane's log-likelihoods (fits.py:147-165)
                            const double* llc = llb + (size_t)roles.get(LL_CUR) * wstride + lane;
                            double* const wacc = wacc_of_lane();
#pragma unroll 1
                            for (int s = 0; s < ns; ++s) {
                                const double v = llc[s * 32];
                                double wmax = wacc[0 * wstride + s * 32], wsum = wacc[1 * wstride + s * 32];
                                double wmean = wacc[2 * wstride + s * 32], wm2 = wacc[3 * wstride + s * 32];
                                const double ed = exp_nonpos(-fabs(v - wmax));  // first draw: wmax = -inf, ed is ~1e-305 and multiplies wsum = 0
                                if (v > wmax) { wsum = fma(wsum, ed, 1.0); wmax = v; }
                                else wsum += ed;
                                const double dpre = v - wmean;
                                wmean += dpre * inv_n;
                                wm2 += dpre * (v - wmean);
                                wacc[0 * wstride + s * 32] = wmax; wacc[1 * wstride + s * 32] = wsum;
                                wacc[2 * wstride + s * 32] = wmean; wacc[3 * wstride + s * 32] = wm2;
                            }
                        }
                        // layout: transition_end
                        if (p.trace != nullptr && lig < 4) store_trace(p, tax, run_kind, t, lig, own ? zc : nan(""));
                        __syncwarp(gmask);
                        t += 1;
                        if (t >= W + S) {
                            done = true;
                        } else if (want_heur) {
                            ++h_call;
                            pend = PS_HEUR_BEGIN;
                        } else {
                            pend = PS_TRANSITION;
                        }
                    }
                }
            } else if (phase == GP_HEUR) {  // layout: heuristic
                heur_record<D, GW>(sh, jc, rn, pen, gmask);
                pend = PS_HEUR;
            } else {  // layout: init
                // ---- GP_INIT: init_to_uniform(radius), retried until finite ----
                if (valid) {
                    pe_cur = pen;
                    roles.swap(LL_X, LL_CUR);
                    __syncwarp(gmask);
                    if (own) { sh.zp[lig] = zn; sh.gp[lig] = gn; }
                    __syncwarp(gmask);
                    if (W + S == 0) {
                        done = true;
                    } else if (p.cfg.find_heuristic_step_size && W > 0) {
                        h_call = 0;
                        pend = PS_HEUR_BEGIN;
                    } else {
                        pend = PS_RESET;
                    }
                } else {
                    ++init_attempt;
                    if (init_attempt >= 100u) {
                        failed = 1; done = true;
                    } else {
                        zf = init_position(p, key, jc, init_attempt, run_kind);
                        rf = 0.0; gf = 0.0; e = 0.0;
                        phase = GP_INIT;
                    }
                }
            }

            // ---- what the bookkeeping asked for: aim the next leapfrog ----
            if (pend == PS_HEUR_BEGIN || pend == PS_HEUR) {  // layout: heuristic
                const double2 trial = heur_next<D, GW>(sh, pend == PS_HEUR_BEGIN, key, run_kind, jc, gmask);
                if (trial.y != 0.0) {
                    rf = trial.x;
                    __syncwarp(gmask);
                    zf = sh.zp[jc]; gf = sh.gp[jc];
                    e = h_step;
                    phase = GP_HEUR;
                    pend = PS_HEUR;
                } else {
                    pend = PS_RESET;
                }
            }
            if (pend == PS_RESET) {
                reset_dual_averaging(sh);
                pend = PS_TRANSITION;
            }
            if (pend == PS_TRANSITION) {  // layout: transition_start
                const double r0 = draw_normal_lane_cold<D>(key, (uint32_t)t, c2word(run_kind, P_MOM), 0u, jc) * sh.isd[jc];
                E0 = pe_cur + kinetic<D, GW>(sh.imm[jc], r0, gmask);
                __syncwarp(gmask);
                if (own) {
                    const double zj = sh.zp[lig], gj = sh.gp[lig];
                    sh.zl[lig] = zj; sh.zr[lig] = zj; sh.gl[lig] = gj; sh.gr[lig] = gj;
                    sh.rl[lig] = r0; sh.rr[lig] = r0;
                    sh.m_rsum[lig] = r0;
                }
                m_weight = 0.0; m_sum_acc = 0.0; m_nprop = 0; m_depth = 0; m_turning = false; m_div = false;
                m_pe_p = pe_cur;
                m_is_c = true;  // the tree's proposal is the current state until a subtree's proposal is taken
                leaf_counter = 0;
                pend = PS_DOUBLING;
            }
            if (pend == PS_DOUBLING) {  // layout: doubling
                double u_dir;
                uniform2(philox4x32(key, (uint32_t)m_depth, (uint32_t)t, c2word(run_kind, P_DIR), 0u), u_dir, u_main);
                going_right = u_dir < 0.5;
                s_nprop = 0;
                __syncwarp(gmask);
                zf = going_right ? sh.zr[jc] : sh.zl[jc];
                rf = going_right ? sh.rr[jc] : sh.rl[jc];
                gf = going_right ? sh.gr[jc] : sh.gl[jc];
                e = going_right ? eps : -eps;
                phase = GP_LEAF;
            }
        }

        // ================= chain finished: per-run outputs, then fetch the next item =================
        if (done) {  // layout: chain_end
            chain_end<GW, D>(p, sh, kn, wacc_of_lane(), tax, run_kind, mask, n_obs, ns, failed, n_grad, lane, lig, gmask);
            // the leapfrog source is dead here; saying so keeps the compiler from carrying its old value across the
            // evaluation (in registers, which the evaluation needs) for the paths that end a chain without overwriting it
            zf = 0.0; rf = 0.0; gf = 0.0;
            phase = GP_FETCH;
        }
    }
}

}  // namespace mdg
