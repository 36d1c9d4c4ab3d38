// mdg_common.cuh — device helpers shared by the sm_100a kernels: error plumbing, Philox4x32-10
// streams, warp/sub-warp reductions and the FP64 special functions (lgamma + digamma in one pass).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "mdg.h"

// Kernel tuning switches kept for A/B measurements (profiles/r01_nuts_tuning.md). Defaults = shipped.
#ifndef MDG_LOGFN
#define MDG_LOGFN 1          // 1: table-driven log_pos; 0: CUDA log()
#endif
#ifndef MDG_COLD_INLINE
#define MDG_COLD_INLINE 0    // 0: one out-of-line copy of Philox, Box-Muller, logaddexp, cold exp/log (the hot loop is
                             // instruction-fetch sensitive: -9 % NUTS time); 1: everything inlined
#endif
#if MDG_COLD_INLINE
#define MDG_COLD __forceinline__
#else
#define MDG_COLD __noinline__
#endif

namespace mdg {

// ---------------------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define MDG_CUDA_TRY(expr)                                                                     \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            mdg::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,                \
                           cudaGetErrorString(_e));                                            \
            return MDG_ERR_CUDA;                                                               \
        }                                                                                      \
    } while (0)

// ---------------------------------------------------------------------------------------------
// Philox4x32-10, keyed by (seed, tax_id); counter layout (c0 draw index, c1 iteration,
// c2 run_kind | purpose << 8, c3 aux) — see DESIGN.md "Random streams"
// ---------------------------------------------------------------------------------------------
enum Purpose : uint32_t { P_INIT = 1, P_MOM = 2, P_DIR = 3, P_SUB = 4, P_HEUR = 5, P_PPC = 6 };

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__host__ __device__ __forceinline__ uint2 make_key(uint64_t seed, int64_t tax_id) {
    uint64_t k = splitmix64(seed ^ splitmix64((uint64_t)tax_id));
    return make_uint2((uint32_t)k, (uint32_t)(k >> 32));
}

__device__ MDG_COLD uint4 philox4x32(uint2 key, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
    uint32_t k0 = key.x, k1 = key.y;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint32_t c2word(int run_kind, uint32_t purpose) {
    return (uint32_t)run_kind | (purpose << 8);
}

// two uniforms in (0,1): 53 random bits + half an ulp
__device__ __forceinline__ void uniform2(uint4 o, double& u0, double& u1) {
    u0 = ((double)(o.x >> 5) * 67108864.0 + (double)(o.y >> 6) + 0.5) * (1.0 / 9007199254740992.0);
    u1 = ((double)(o.z >> 5) * 67108864.0 + (double)(o.w >> 6) + 0.5) * (1.0 / 9007199254740992.0);
}

// ---------------------------------------------------------------------------------------------
// sub-warp butterflies: every lane of a GW-wide group ends with the bit-identical sum
// ---------------------------------------------------------------------------------------------
template <int GW>
__device__ __forceinline__ double group_sum(double v, unsigned mask) {
#pragma unroll
    for (int o = GW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
}

template <int GW>
__device__ __forceinline__ unsigned group_mask() {
    if constexpr (GW == 32) {
        return 0xffffffffu;
    } else {
        unsigned lane = threadIdx.x & 31u;
        return ((1u << GW) - 1u) << (lane & ~(unsigned)(GW - 1));
    }
}

// ---------------------------------------------------------------------------------------------
// FP64 special functions of the fit kernels.
//
// sm_100a FP64 instructions take no constant-bank operand: a full-precision literal costs two
// register moves (or an LDC) per use, and ptxas, hoisting them, spilled live chain state to make
// room (round-1 ncu: of ~95 instructions per lgamma/digamma pair only 45 were FP64). A double whose
// low 32 bits are zero, however, is encoded as an IMMEDIATE. So every polynomial coefficient whose
// term tolerates a 2^-21 relative perturbation is written as such a 21-significant-bit value
// (hex-float literals below; the perturbation of the result is stated next to each), exact
// constants (0.5, 0.25, small integers) are used where the series allows, ln2 is split into
// immediate pieces, and only four constants (1/12, 1/360, 1/120, ln2_lo) stay full precision.
// ---------------------------------------------------------------------------------------------
// Stirling series of lgamma  t/12 - t^3/360 + t^5/1260 - t^7/1680 + t^9/1188      (t = 1/y)
// and of digamma  log y - t/2 - t^2/12 + t^4/120 - t^6/252 + t^8/240 - t^10/132,  y >= 10:
// truncation 1.9e-14 / 2.1e-14 absolute; the three trailing coefficients of each are immediates
// (perturbation < 5e-16).
#define MDG_K_LG2 0x1.a01a0p-11   /* 1/1260 */
#define MDG_K_LG3 0x1.38138p-11   /* 1/1680 */
#define MDG_K_LG4 0x1.b951ep-11   /* 1/1188 */
#define MDG_K_DG2 0x1.04104p-8    /* 1/252 */
#define MDG_K_DG3 0x1.11111p-8    /* 1/240 */
#define MDG_K_DG4 0x1.f07c2p-8    /* 1/132 */

// ---------------------------------------------------------------------------------------------
// Division-free natural log of a positive, normal, finite double.
//   x = 2^e * m, m in [1, 2);  i = top 8 mantissa bits;  c_i = 1 + (i + 1/2) / 256
//   r = m / c_i - 1  (|r| <= 2^-9, one fma with the tabulated 1/c_i)
//   log x = e ln2 + log c_i + (r - r^2/2 + r^3/3 - r^4/4 + r^5/5)        (r^6/6 < 1e-17)
// 1/3 and 1/5 are immediates (perturbation < 1.2e-15 absolute); e*ln2_hi is exact (21 x 11 bits).
// The 4 KB table {1/c_i, log c_i} lives in shared memory (one copy per CTA); every kernel that
// evaluates logs calls log_table_init() once before use.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double2* log_table() {
    __shared__ double2 tab[256];
    return tab;
}

__device__ __forceinline__ double* exp_table() {
    __shared__ double tab[128];  // 2^(j/128)
    return tab;
}

__device__ __forceinline__ void log_table_init() {
    double2* tab = log_table();
    double* et = exp_table();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const double c = 1.0 + ((double)i + 0.5) / 256.0;
        const double ic = 1.0 / c;
        tab[i] = make_double2(ic, -log(ic));   // the log that matches the ROUNDED reciprocal
        if (i < 128) et[i] = exp2((double)i / 128.0);
    }
    __syncthreads();
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// 1/x for positive normal x: hardware seed (MUFU.RCP64H, ~2^-21) + two Newton steps (<= 2 ulp)
__device__ __forceinline__ double rcp_pos(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

// e^x for finite |x| <= 708, no range or NaN handling (callers guard):
//   n = rint(128 x / ln2) by the 1.5*2^52 trick (its low mantissa word IS the integer),
//   r = x - n ln2/128 with ln2/128 in three immediate pieces (n * piece exact), |r| <= 2.8e-3,
//   e^x = 2^(n >> 7) * 2^((n & 127)/128) * (1 + r + r^2/2 + r^3/6 + r^4/24 + r^5/120);
// 1/6, 1/24, 1/120 are immediates (perturbation < 1e-15 relative); the power of two is added
// straight into the exponent field. ~3 ulp.
__device__ __forceinline__ double exp_core(double x) {
    const double nm = fma(x, 0x1.71547p+7, 6755399441055744.0);
    const int ni = __double2loint(nm);
    const double n = nm - 6755399441055744.0;
    double r = fma(n, -0x1.62e42p-8, x);
    r = fma(n, -0x1.fdf47p-29, r);
    r = fma(n, -0x1.ef358p-52, r);
    const double tj = exp_table()[ni & 127];
    double q = fma(r, 0x1.11111p-7, 0x1.55555p-5);
    q = fma(r, q, 0x1.55555p-3);
    q = fma(r, q, 0.5);
    q = fma(r, q, 1.0);
    q = fma(r, q, 1.0);
    const double y = tj * q;  // in [0.99, 2)
    return __hiloint2double(__double2hiint(y) + ((ni >> 7) << 20), __double2loint(y));
}

// e^x for x <= 0 (sign bit set or +0; -inf and NaN-with-sign allowed): arguments below -700 act
// as -700.99 (one integer min on the high word), i.e. the result is ~1e-305 instead of 0.
__device__ __forceinline__ double exp_nonpos(double x) {
    const unsigned hi = (unsigned)__double2hiint(x);
    return exp_core(__hiloint2double((int)min(hi, 0xc085e000u), __double2loint(x)));
}

// e^x for any double (tests, cold callers): exact limits, NaN propagates
__device__ __forceinline__ double exp_fast(double x) {
    const double xc = fmin(fmax(x, -700.0), 700.0);
    const double y = exp_core(xc);
    return x != x ? x : (x < -700.0 ? (x < -745.2 ? 0.0 : exp(x)) : (x > 700.0 ? exp(x) : y));
}

__device__ __forceinline__ double log_pos(double x) {
    const int hi = __double2hiint(x), lo = __double2loint(x);
    const double2 t = log_table()[(hi >> 12) & 255];
    const double de = (double)((hi >> 20) - 1023);
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, lo);
    const double r = fma(m, t.x, -1.0);
    double q = fma(r, 0x1.9999ap-3, -0.25);
    q = fma(r, q, 0x1.55555p-2);
    q = fma(r, q, -0.5);
    q = fma(r, q, 1.0);
    // ln2 = 0x1.62e43p-1 - 1.904654299957768e-09
    return fma(de, 0x1.62e43p-1, t.y) + fma(de, -1.904654299957768e-09, r * q);
}

// two standard normals (Box-Muller); sincospi needs no large-argument reduction
__device__ __forceinline__ void normal2(uint4 o, double& n0, double& n1) {
    double u0, u1;
    uniform2(o, u0, u1);
    const double rad = sqrt(-2.0 * log_pos(u0));
    double s, c;
    sincospi(2.0 * u1, &s, &c);
    n0 = rad * c;
    n1 = rad * s;
}

// Out-of-line copies of the transcendental functions for the COLD parts of the kernels (once per
// transition or rarer). The NUTS kernel was instruction-fetch bound (ncu: stall_no_instruction
// 45 % of all stalls with 12.4k SASS instructions); one shared copy of each keeps the hot loop
// (one gradient evaluation + leaf bookkeeping) inside the instruction caches.
// They use the kernels' own table-driven exp / log (a few ulp; the CUDA library versions are 2-4x as many
// instructions and every one of them is issued for ONE chain): the library call only backs up arguments
// outside the fast paths' domain.
__device__ MDG_COLD double exp_cold(double x) { return exp_fast(x); }
// exp_fast with its library branches out of line: the same value for every x, for callers that run once per
// transition and want only exp_core's instructions inline
__device__ MDG_COLD double exp_fast_outside(double x) { return x != x ? x : (x < -700.0 ? (x < -745.2 ? 0.0 : exp(x)) : exp(x)); }
__device__ __forceinline__ double exp_fast_split(double x) { return (x >= -700.0 && x <= 700.0) ? exp_core(x) : exp_fast_outside(x); }
__device__ MDG_COLD double log_cold(double x) { return (x >= 2.2250738585072014e-308 && x < INFINITY) ? log_pos(x) : log(x); }
__device__ MDG_COLD double sigmoid_cold(double x) {
    const double e = exp_fast(-fabs(x));  // in (0, 1]
    const double inv = rcp_pos(1.0 + e);
    return x != x ? x : (x >= 0.0 ? inv : e * inv);
}

// st = lgamma(y) - 0.5 log(2 pi) and dg = digamma(y) for y >= 10, t = 1/y (5 Bernoulli terms each)
__device__ __forceinline__ double log_sel(double x) {
#if MDG_LOGFN
    return log_pos(x);
#else
    return log(x);
#endif
}

__device__ __forceinline__ void stirling(double y, double t, double& st, double& dg) {
    const double L = log_sel(y);
    const double t2 = t * t;
    double sl = fma(t2, -MDG_K_LG4, MDG_K_LG3);
    sl = fma(t2, -sl, MDG_K_LG2);
    sl = fma(t2, -sl, 1.0 / 360.0);
    sl = fma(t2, -sl, 1.0 / 12.0);
    double sd = fma(t2, -MDG_K_DG4, MDG_K_DG3);
    sd = fma(t2, -sd, MDG_K_DG2);
    sd = fma(t2, -sd, 1.0 / 120.0);
    sd = fma(t2, -sd, 1.0 / 12.0);
    st = fma(t, sl, fma(y - 0.5, L, -y));
    dg = fma(-t2, sd, fma(-0.5, t, L));
}

// P(x) = x (x+1) ... (x+9) and P'(x) by Horner on the expanded polynomials: every coefficient is an
// integer below 2^22 with at most 21 significant bits, i.e. an exact immediate; all terms are
// positive for x > 0, so there is no cancellation (two independent chains of 10 and 9 operations
// instead of the 27 of the running product).
__device__ __forceinline__ void shift_poly10(double x, double& P, double& dP) {
    double p = x + 45.0;
    p = fma(x, p, 870.0);
    p = fma(x, p, 9450.0);
    p = fma(x, p, 63273.0);
    p = fma(x, p, 269325.0);
    p = fma(x, p, 723680.0);
    p = fma(x, p, 1172700.0);
    p = fma(x, p, 1026576.0);
    p = fma(x, p, 362880.0);
    P = x * p;
    double q = fma(x, 10.0, 405.0);
    q = fma(x, q, 6960.0);
    q = fma(x, q, 66150.0);
    q = fma(x, q, 379638.0);
    q = fma(x, q, 1346625.0);
    q = fma(x, q, 2894720.0);
    q = fma(x, q, 3518100.0);
    q = fma(x, q, 2053152.0);
    dP = fma(x, q, 362880.0);
}

// lgamma(x) - 0.5 log(2 pi) and digamma(x), x > 0, in one pass. x < 10 is shifted to y = x + 10
// with P = x (x+1) ... (x+9) and its derivative (lgamma(x) = lgamma(y) - log P, digamma(x) =
// digamma(y) - P'/P: one log and one reciprocal instead of ten); y >= 10 uses the Stirling /
// asymptotic series. The constant 0.5 log(2 pi) is left out: it cancels in the beta-binomial
// log-likelihood (three lgammas enter with +, three with -).
__device__ __forceinline__ void lgam_digam_u(double x, unsigned gmask, double& lg, double& dg) {
    double y = x, logP = 0.0, dP = 0.0;
    const bool small = x < 10.0;
    double t;
    if (small) {
        double P, Q;
        shift_poly10(x, P, Q);
        logP = log_sel(P);
        y = x + 10.0;
        const double r = rcp_pos(y * P);  // one reciprocal serves 1/y and Q/P
        t = r * P;
        dP = Q * (r * y);
    } else {
        t = rcp_pos(y);
    }
    double st, d;
    stirling(y, t, st, d);
    lg = st - logP;
    dg = d - dP;
}

// K independent evaluations at once, phased so that the (branch-free) reciprocal / log / Stirling
// chains of all K arguments sit in one basic block and can be interleaved by the scheduler; the
// x < 10 corrections (-log P, -P'/P) follow under per-argument branches. ncu on the one-at-a-time
// form: `stall_wait` (dependent FP64 chains, 4 warps per scheduler) was the top stall reason.
#ifndef MDG_PHASED
#define MDG_PHASED 1
#endif
template <int K>
__device__ __forceinline__ void lgam_digam_batch(const double (&x)[K], unsigned gmask, double (&lg)[K], double (&dg)[K]) {
#if MDG_PHASED
    bool small[K];
    double y[K], t[K];
#pragma unroll
    for (int i = 0; i < K; ++i) {
        small[i] = x[i] < 10.0;
        y[i] = x[i] + (small[i] ? 10.0 : 0.0);
        t[i] = rcp_pos(y[i]);
    }
#pragma unroll
    for (int i = 0; i < K; ++i) stirling(y[i], t[i], lg[i], dg[i]);
#pragma unroll
    for (int i = 0; i < K; ++i) {
        if (small[i]) {
            double P, Q;
            shift_poly10(x[i], P, Q);
            lg[i] -= log_sel(P);
            dg[i] = fma(-Q, rcp_pos(P), dg[i]);
        }
    }
#else
#pragma unroll
    for (int i = 0; i < K; ++i) lgam_digam_u(x[i], gmask, lg[i], dg[i]);
#endif
}

// single-thread forms (log C(N,k), the predictive's BTRS sampler, the special-function test hook)
__device__ __forceinline__ void lgam_digam(double x, double& lg, double& dg) {
    double a, b;
    lgam_digam_u(x, 0xffffffffu, a, b);
    lg = a + 0.91893853320467274178;
    dg = b;
}

__device__ __forceinline__ double lgam(double x) {
    double lg, dg;
    lgam_digam(x, lg, dg);
    return lg;
}

// softplus(u) = log(1 + e^u), sigmoid(u), both from one exp + one log1p
__device__ __forceinline__ void softplus_sigmoid(double u, double& sp, double& sg) {
    double e = exp(-fabs(u));
    double l = log1p(e);
    double inv = 1.0 / (1.0 + e);
    sp = fmax(u, 0.0) + l;
    sg = (u >= 0.0) ? inv : e * inv;
}

// log(e^a + e^b) = max + log(1 + e^-|a-b|); out of line (used twice per leaf, never in the gradient)
__device__ MDG_COLD double logaddexp(double a, double b) {
    if (a == -INFINITY && b == -INFINITY) return -INFINITY;
    const double m = fmax(a, b), d = -fabs(a - b);
    return isnan(d) ? (a + b) : m + log_pos(1.0 + exp(d));
}

}  // namespace mdg
