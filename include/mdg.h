/*
 * mdg.h — C-ABI of libmdgb200.so: the B200-native per-TaxID damage-fitting hot path.
 *
 * This is the drop-in boundary for metadamage's hot path. The reference has no FFI of its
 * own (it is pure Python); the two Python seams that bind to these entry points are
 *
 *   counts.compute_counts_with_dask(cfg)          /root/reference/metadamage/counts.py:212-273
 *       -> mdg_counts_reduce()        (replaces counts.py:237-256: reference sums, error
 *                                      rates, signed 1-indexed z, per-TaxID y_sum_total, cuts)
 *   fits.compute_fits(df_counts, cfg, mcmc_kwargs) /root/reference/metadamage/fits.py:709-730
 *       -> mdg_fit_batch()            (replaces fits.py:428-469 per TaxID: 6 NUTS runs
 *                                      fits.py:438-439,311-337, WAIC fits.py:147-227,
 *                                      posterior predictive fits.py:89-120, noise
 *                                      fits.py:359-376, result row fits.py:230-295;
 *                                      plus the new MAP fit the north star asks for)
 *
 * Conventions
 *   - plain pointers and sizes only; every buffer is caller-owned; nothing is retained
 *     after a call returns (mdg_fit_batch_submit: after the matching mdg_fit_batch_wait returns).
 *   - every function returns MDG_OK (0) or a negative error code; mdg_last_error() gives a
 *     thread-local human-readable message.
 *   - a ctx is bound to one GPU and one CUDA stream and is NOT thread-safe; distinct ctxs
 *     are independent (one host thread or one process per GPU).
 *   - `mem` says where ALL data pointers of that call live: MDG_HOST (pageable or pinned
 *     host memory; the call does H2D, compute, D2H and synchronises) or MDG_DEVICE (device
 *     memory on the ctx's GPU). mdg_fit_batch_submit only enqueues work, for either memory
 *     space (ordered after everything already on the ctx stream); mdg_fit_batch_wait,
 *     mdg_fit_batch (= submit + wait) and calls with scalar host outputs such as out_n_tax
 *     synchronise with the host.
 *   - results are a pure function of (tax_id, k, N, cfg): Philox4x32-10 streams are keyed by
 *     (cfg.seed, tax_id) and counted by (run kind, purpose, iteration, draw), so any
 *     partition of a batch over GPUs / calls gives bit-identical per-TaxID results.
 */
#ifndef MDG_H
#define MDG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
#define MDG_STATIC_ASSERT(cond, msg) static_assert(cond, msg)
#else
#define MDG_STATIC_ASSERT(cond, msg) _Static_assert(cond, msg)
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MDG_VERSION 200 /* 0.2.0 */

enum mdg_status {
    MDG_OK = 0,
    MDG_ERR_INVALID = -1,          /* bad argument */
    MDG_ERR_CUDA = -2,             /* CUDA runtime error (message has the detail) */
    MDG_ERR_NOMEM = -3,            /* allocation failed */
    MDG_ERR_SEGMENT_TOO_LONG = -4, /* a TaxID has more rows than MDG_MAX_SEGMENT_ROWS */
    MDG_ERR_OVERFLOW = -5,         /* a reference-base row sum exceeds uint32 (utils.py:338-339) */
    MDG_ERR_BUSY = -6              /* mdg_fit_batch_submit: MDG_MAX_INFLIGHT batches are already in flight on this ctx */
};

enum mdg_memspace { MDG_HOST = 0, MDG_DEVICE = 1 };

/* the six NUTS runs of one TaxID (fits.py:438-439, 312-313, 334-335) */
enum mdg_run_kind {
    MDG_RUN_PMD_ALL = 0,
    MDG_RUN_NULL_ALL = 1,
    MDG_RUN_PMD_FWD = 2,
    MDG_RUN_NULL_FWD = 3,
    MDG_RUN_PMD_REV = 4,
    MDG_RUN_NULL_REV = 5,
    MDG_NUM_RUNS = 6
};

/* per-TaxID status bits in mdg_fit_result.status (0 = clean fit). A TaxID with
 * MDG_FIT_FAILED set is dropped by the host, like a timed-out fit (fits.py:520-521). */
#define MDG_FIT_FAILED 0x1u        /* no finite initial point found / non-finite summary */
#define MDG_FIT_MAP_NOT_CONVERGED 0x2u
#define MDG_FIT_HAS_DIVERGENCES 0x4u /* >=1 divergent transition after warm-up (informational) */
#define MDG_FIT_BUDGET_EXCEEDED 0x8u /* a run needed more than cfg.max_leapfrogs_per_run gradient evaluations:
                                      * the bounded-work analogue of the reference's per-fit timeout
                                      * (fits.py:37-38, 472-474); always set together with MDG_FIT_FAILED */
#define MDG_FIT_COV_INVALID 0x10u    /* mdg_map_batch: no Laplace covariance (the MAP fit did not converge, or the
                                      * Hessian at the mode is not positive definite); the standard deviations are NaN */

#ifndef MDG_MAX_INFLIGHT
#define MDG_MAX_INFLIGHT 2         /* batches one ctx keeps in flight between mdg_fit_batch_submit and _wait */
#endif
#define MDG_MAX_POSITION 64        /* max_position supported by the fit kernels */
#define MDG_MAX_SEGMENT_ROWS 2048  /* rows of one TaxID the counts kernel can hold in one tile */

typedef struct mdg_ctx mdg_ctx;

/* NUTS / model configuration. mdg_fit_config_default() fills the reference's values:
 * fits.py:43-67 (priors), fits.py:792-799 (500 warm-up + 1000 samples, 1 chain) and the
 * numpyro 0.4.1 NUTS defaults (step_size 1, target_accept 0.8, max_tree_depth 10,
 * diagonal mass adaptation, init_to_uniform(radius=2)). */
typedef struct mdg_fit_config {
    int32_t num_warmup;
    int32_t num_samples;
    int32_t max_tree_depth;
    int32_t do_map;                   /* 1: also run the MAP fit (new deliverable) */
    int32_t do_fwd_rev;               /* 1: the four forward-/reverse-only runs (fits.py:298-356) */
    int32_t find_heuristic_step_size; /* numpyro's HMC/NUTS(find_heuristic_step_size=...): 1 runs find_reasonable_step_size
                                       * at initialisation and at every adaptation-window end. Default 0 = numpyro 0.4.1's
                                       * default (False), which fits.py:382-387 does not override */
    int32_t reference_quirks;         /* 1: D_max_reverse predictive uses the forward N (fits.py:343-348) */
    int32_t pack_half_warps;          /* ignored since 0.2.0 (every run is a group of 8 lanes now); kept for layout compatibility */
    double target_accept;
    double init_step_size;
    double max_delta_energy;
    double init_radius;
    double hpdi_prob;                 /* 0.68 (fits.py:119) */
    uint64_t seed;
    double q_prior_a, q_prior_b;      /* Beta(2,3)  fits.py:46,63 */
    double A_prior_a, A_prior_b;      /* Beta(2,3)  fits.py:47 */
    double c_prior_a, c_prior_b;      /* Beta(1,9)  fits.py:48 */
    double phi_prior_rate;            /* Exponential(rate=1/1000) on delta = phi - phi_min  fits.py:53,65 */
    double phi_min;                   /* 2  fits.py:54,66 */
    int32_t max_leapfrogs_per_run;    /* 0 = unlimited (default). > 0: a NUTS run that needs more gradient evaluations is
                                       * abandoned and its TaxID gets MDG_FIT_FAILED | MDG_FIT_BUDGET_EXCEEDED */
    int32_t reserved0;
} mdg_fit_config;

/* per-run sampler diagnostics */
typedef struct mdg_run_diag {
    double step_size;        /* final adapted step size */
    double mean_accept;      /* mean tree acceptance statistic after warm-up */
    uint32_t n_leapfrog;     /* log-density-gradient evaluations of this run (all phases) */
    uint32_t n_divergent;    /* divergent transitions after warm-up */
    double waic;             /* WAIC of this run (fits.py:164-168) */
    double lppd;             /* fits.py:152-156 */
} mdg_run_diag;

/* One row per TaxID. The first block mirrors the reference's fit_result dict
 * (fits.py:242-293, 317-356, 374-376), in FP64; the host down-casts (fits.py:673-676). */
typedef struct mdg_fit_result {
    int64_t tax_id;
    uint32_t status;
    uint32_t map_iters;
    /* reference fit_result fields */
    double D_max;                    /* median_s(y_rep(z=1)/N(z=1))           fits.py:249-250 */
    double n_sigma;                  /* fits.py:252, 194-201 */
    double D_max_lower_hpdi;         /* fits.py:260 */
    double D_max_upper_hpdi;         /* fits.py:261 */
    double q_mean;                   /* fits.py:266 */
    double concentration_mean;       /* mean phi  fits.py:268 */
    double D_max_marginalized_mean;  /* mean A+c  fits.py:270 */
    double n_sigma_forward;          /* fits.py:317 */
    double D_max_forward;            /* fits.py:322 */
    double q_mean_forward;           /* fits.py:329 */
    double n_sigma_reverse;          /* fits.py:339 */
    double D_max_reverse;            /* fits.py:343 (quirk: forward N) */
    double q_mean_reverse;           /* fits.py:350 */
    double asymmetry;                /* fits.py:352, 204-227 */
    double normalized_noise;         /* fits.py:374 */
    double normalized_noise_forward; /* fits.py:375 */
    double normalized_noise_reverse; /* fits.py:376 */
    uint64_t N_z1_forward;           /* fits.py:274 */
    uint64_t N_z1_reverse;           /* fits.py:275 */
    uint64_t N_sum_forward;          /* fits.py:277 */
    uint64_t N_sum_reverse;          /* fits.py:278 */
    uint64_t N_sum_total;            /* fits.py:279 */
    uint64_t y_sum_forward;          /* fits.py:281 */
    uint64_t y_sum_reverse;          /* fits.py:282 */
    uint64_t y_sum_total;            /* fits.py:283 */
    /* new: MAP fit of the PMD model on all positions (constrained-space posterior mode) */
    double map_A, map_q, map_c, map_phi, map_D_max, map_logp;
    /* new: MAP of the null model on all positions */
    double map_null_q, map_null_phi, map_null_logp;
    /* new: posterior spreads of the PMD/all run (needed for the 3xMCSE parity gate) */
    double A_mean, c_mean;
    double D_max_marginalized_std, q_std, concentration_std;
    mdg_run_diag run[MDG_NUM_RUNS];
} mdg_fit_result;

/* device timings of the last call on a ctx, measured with CUDA events on the ctx stream */
typedef struct mdg_timings {
    float counts_ms;      /* counts_reduce kernel (K1); for mdg_tsv_parse: the parse kernels (K0) */
    float map_ms;         /* MAP kernel (K3) */
    float nuts_ms;        /* all NUTS kernels (K4), summed over chunks */
    float ppc_ms;         /* posterior predictive + sort + HPDI (K6) */
    float assemble_ms;    /* WAIC -> n_sigma/asymmetry, noise, row assembly (K5/K7) */
    float total_ms;       /* whole call on the stream, incl. copies for MDG_HOST */
    uint32_t n_launches;  /* kernels launched by the last call */
    uint32_t reserved;
    uint64_t leapfrogs[MDG_NUM_RUNS]; /* gradient evaluations per run kind, summed over TaxIDs */
    /* Batches in flight together run their NUTS launches concurrently, so their nuts_ms overlap. nuts_union_ms is
     * this batch's contribution to the union of all NUTS intervals of the ctx (batches waited for in submission
     * order): summed over batches it is the time during which at least one NUTS kernel was running.
     * nuts_begin_ms / nuts_end_ms: first NUTS start / last NUTS end of the batch, in ms since mdg_ctx_create. */
    float nuts_union_ms;
    float nuts_begin_ms;
    float nuts_end_ms;
    float reserved1;
} mdg_timings;

/*
 * MAP-only screening (mdg_map_batch). A MAP fit is the mode of the constrained-space posterior
 * (likelihood x priors, no Jacobian term), found in the unconstrained coordinates u by LM-damped
 * Newton; it is the same fit as mdg_fit_result.map_*. It is made for the six run kinds of
 * enum mdg_run_kind (cfg.do_fwd_rev = 0: the two all-position ones only).
 *
 * Laplace covariance at the converged u*: H_u is the symmetrised central-difference Hessian of the
 * analytic gradient of f = -log p (steps h_j = 1e-4 (1 + |u_j|), as in the Newton loop),
 * Sigma_u = H_u^-1, and Sigma_theta = J Sigma_u J with J = diag(d theta_j / d u_j): theta (1 - theta)
 * for q, A, c and exp(u_delta) for phi. f has no Jacobian term, so grad_u f = J grad_theta f and the
 * second-order term of the change of variables vanishes at a stationary point: J H_u^-1 J is the
 * inverse Hessian of f in theta.
 */
typedef struct mdg_map_run {
    double q, A, c, phi;                 /* mode; null runs: A = c = NaN */
    double q_std, A_std, c_std, phi_std; /* Laplace standard deviations; NaN with MDG_FIT_COV_INVALID (null: A, c NaN) */
    double cov_Ac;                       /* Laplace covariance of A and c (PMD runs) */
    double logp;                         /* log posterior at the mode incl. log C(N,k), no Jacobian (= map_logp) */
    double loglik;                       /* sum over the run's positions of log BetaBinomial(k | N, alpha, beta) at the
                                          * mode, incl. log C(N,k) */
    uint32_t iters;                      /* Newton iterations */
    uint32_t n_eval;                     /* gradient evaluations: Newton loop, log-likelihood and Laplace Hessian */
    uint32_t flags;                      /* MDG_FIT_FAILED (no finite starting point), MDG_FIT_MAP_NOT_CONVERGED,
                                          * MDG_FIT_COV_INVALID of this run; 0 = clean. A run that was not made
                                          * (do_fwd_rev = 0) is all NaN with flags = n_eval = 0 */
    uint32_t reserved;
} mdg_map_run;

/* One row per TaxID. D_max is A + c at the PMD mode, NOT the posterior predictive median that
 * mdg_fit_result.D_max holds. lambda_LR = 2 (loglik_PMD - loglik_null) of the all-position fits,
 * lambda_LR_P = exp(-max(lambda_LR, 0) / 2) (chi-square tail, 4 - 2 = 2 degrees of freedom),
 * lambda_LR_z = -Phi^-1(lambda_LR_P) evaluated from log P (finite where P underflows). The null model
 * is A = 0, a boundary point of the PMD model at which q is unidentified, so the chi-square
 * reference does not hold: P and z are a screening scale, not calibrated p-values. */
typedef struct mdg_map_result {
    int64_t tax_id;
    uint32_t status;       /* MDG_FIT_FAILED / MDG_FIT_MAP_NOT_CONVERGED / MDG_FIT_COV_INVALID of the two all-position runs */
    uint32_t reserved;
    double D_max;          /* A + c at the PMD mode */
    double D_max_std;      /* sqrt(Sigma_AA + Sigma_cc + 2 Sigma_Ac) */
    double significance;   /* D_max / D_max_std */
    double rho_Ac;         /* Sigma_Ac / sqrt(Sigma_AA Sigma_cc) */
    double lambda_LR, lambda_LR_P, lambda_LR_z;
    double forward_D_max, forward_D_max_std, forward_lambda_LR;  /* same from the forward-only pair of fits */
    double reverse_D_max, reverse_D_max_std, reverse_lambda_LR;  /* same from the reverse-only pair of fits */
    double normalized_noise, normalized_noise_forward, normalized_noise_reverse;  /* as mdg_fit_result */
    uint64_t N_z1_forward, N_z1_reverse, N_sum_forward, N_sum_reverse, N_sum_total;
    uint64_t y_sum_forward, y_sum_reverse, y_sum_total;
    mdg_map_run run[MDG_NUM_RUNS];
} mdg_map_result;

MDG_STATIC_ASSERT(sizeof(mdg_map_run) == 104, "mdg_map_run layout");
MDG_STATIC_ASSERT(offsetof(mdg_map_run, loglik) == 80 && offsetof(mdg_map_run, flags) == 96, "mdg_map_run layout");
MDG_STATIC_ASSERT(sizeof(mdg_map_result) == 832, "mdg_map_result layout");
MDG_STATIC_ASSERT(offsetof(mdg_map_result, D_max) == 16 && offsetof(mdg_map_result, normalized_noise) == 120 &&
                  offsetof(mdg_map_result, N_z1_forward) == 144 && offsetof(mdg_map_result, run) == 208,
                  "mdg_map_result layout");

/*
 * Profile intervals of D_max = A + c for the MAP-only rows (mdg_map_profile). For one PMD run (all positions,
 * forward only, reverse only) with mode logp^ at D^ = A + c, the profile of the constrained-space log posterior
 * (the density the MAP fit maximises: no Jacobian term, log C(N,k) included) is
 *     pl(D) = max over (q, A, c, phi) with A + c = D of log p(q, A, c, phi | k, N),
 * and the interval at level alpha is {D : 2 (logp^ - pl(D)) <= t}, t = (Phi^-1((1 + alpha) / 2))^2, the
 * chi-square(1) quantile. Each end is the root of h(D) = 2 (logp^ - pl(D)) - t on its side of D^. It is a profile
 * interval of the posterior mode, not an HPDI of the posterior; it respects 0 < D < 1 and may be asymmetric.
 */
#define MDG_PROFILE_AT_BOUND 0x20u /* no crossing up to D = 0 / D = 1: the end is that bound */
#define MDG_PROFILE_FAILED 0x40u   /* root search or an inner fit failed: D is NaN */

typedef struct mdg_profile_end {
    double D;               /* the interval end */
    double q, A, c, phi;    /* maximiser of log p on A + c = D (at a bound: of the last point solved, within 1e-9 of it) */
    double logp;            /* pl(D) */
    uint32_t n_eval, flags; /* gradient evaluations spent on this end; MDG_PROFILE_* / MDG_FIT_FAILED (run unusable) */
} mdg_profile_end;

typedef struct mdg_map_interval {
    int64_t tax_id;
    uint32_t status;           /* OR of the flags of the two all-position ends */
    uint32_t reserved;
    double level, threshold;   /* alpha, t */
    mdg_profile_end end[3][2]; /* [all, forward, reverse][lower, upper] */
} mdg_map_interval;

MDG_STATIC_ASSERT(sizeof(mdg_profile_end) == 56 && offsetof(mdg_profile_end, n_eval) == 48, "mdg_profile_end layout");
MDG_STATIC_ASSERT(sizeof(mdg_map_interval) == 368 && offsetof(mdg_map_interval, end) == 32, "mdg_map_interval layout");

int mdg_version(void);
const char* mdg_last_error(void);
int mdg_device_count(void);

int mdg_ctx_create(int device, mdg_ctx** out);
void mdg_ctx_destroy(mdg_ctx* ctx);
/* use an externally owned CUDA stream (e.g. torch.cuda.current_stream().cuda_stream); NULL = ctx's own */
int mdg_ctx_set_stream(mdg_ctx* ctx, void* cuda_stream);
int mdg_ctx_synchronize(mdg_ctx* ctx);
int mdg_ctx_get_timings(mdg_ctx* ctx, mdg_timings* out);

void mdg_fit_config_default(mdg_fit_config* cfg);

/*
 * K1 — counts_reduce. Replaces counts.py:237-256 (+ the dense k/N extraction of
 * fits.py:398-419 and, optionally, the noise statistic of fits.py:359-376).
 *
 * Input: SoA columns of the mismatch matrix, rows grouped by tax_id (all rows of a TaxID
 * contiguous, as in the reference's input files). counts16 is [16][counts_stride] with
 * column index ref*4+obs over A,C,G,T (counts.py:26-31). pos0 is the 0-indexed position
 * as in the file; is_reverse is (strand != "5'") (utils.py:254-255).
 *
 * Per-row outputs (length n_rows): the reference-base sums (counts.py:86-89), the error
 * rates as float32(double(k)/double(N)) with 0/0 -> 0 (counts.py:109-114, 254), the signed
 * 1-indexed position z (counts.py:117-129), y_sum_total broadcast to the TaxID's rows
 * (counts.py:179-204) and the cut flag (counts.py:207-209; rows with |z| > max_position are
 * not kept and do not contribute to y_sum_total).
 * Per-TaxID outputs (the caller provides room for out_capacity TaxIDs; the number of runs of
 * equal tax_id in the input is always enough; kept TaxIDs come out in input order; a too small
 * capacity is an MDG_ERR_INVALID error, nothing is written past it):
 * tax id, N_alignments, first row index, dense k(z)/N(z) as [n_tax][2*max_position] with
 * slot z-1 for z>0 and max_position+|z|-1 for z<0, summed over the TaxID's rows at that z;
 * optional out_noise [n_tax][3] (normalized_noise, _forward, _reverse of fits.py:359-376, over the
 * TaxID's rows with |z| <= max_position: CT blanked on forward rows, GA on reverse rows; pass
 * NULL to skip).
 * Any output pointer may be NULL to skip that column.
 */
int mdg_counts_reduce(mdg_ctx* ctx, int mem, int64_t n_rows,
                      const int64_t* tax_id, const uint32_t* n_alignments,
                      const uint8_t* is_reverse, const uint8_t* pos0,
                      const uint32_t* counts16, int64_t counts_stride,
                      int fwd_ref, int fwd_obs, int rev_ref, int rev_obs,
                      int max_position, uint32_t min_alignments, uint64_t min_y_sum,
                      uint32_t* n_fwd_ref_row, uint32_t* n_rev_ref_row,
                      float* f_fwd_row, float* f_rev_row,
                      int8_t* z_row, uint64_t* y_sum_total_row, uint8_t* keep_row,
                      int64_t* out_tax_id, uint32_t* out_n_alignments, int64_t* out_first_row,
                      uint32_t* out_k, uint32_t* out_N, double* out_noise,
                      int64_t out_capacity, int64_t* out_n_tax /* host pointer */);

/*
 * K1d — counts_order: the row order of df_counts (counts.py:167-172 sort_by_alignments; C8 of SURVEY.md 8a).
 * The reference sorts ROWS by (N_alignments desc, tax_id desc, 1/z for z > 0 else z desc). Rows of a TaxID
 * are contiguous and share N_alignments and tax_id, so the caller sorts the n_tax per-TaxID keys
 * (`tax_order[i]` = index into the per-TaxID arrays of mdg_counts_reduce of the TaxID that comes i-th) and this
 * call produces the row-level permutation: out_perm[j] = input row of output row j, over the kept rows only
 * (keep_row NULL = all rows), z = +1..+P then -1..-P inside a TaxID, ties in input order (stable).
 * *out_n_rows (host pointer) = number of kept rows written (<= perm_capacity, else MDG_ERR_INVALID).
 */
int mdg_counts_order(mdg_ctx* ctx, int mem, int64_t n_rows,
                     const int64_t* tax_id_row, const int8_t* z_row, const uint8_t* keep_row,
                     int64_t n_tax, const int64_t* first_row, const int64_t* tax_order,
                     int64_t* out_perm, int64_t perm_capacity, int64_t* out_n_rows /* host pointer */);

/*
 * K3-K7 — fit a dense batch of TaxIDs. Replaces fits.py:428-469 for every TaxID.
 * k, N: [n_tax][2*max_position] (layout above). mism12: optional [n_tax][2*max_position][12]
 * raw off-diagonal counts in column order AC,AG,AT,CA,CG,CT,GA,GC,GT,TA,TC,TG for the noise
 * estimate (fits.py:359-376); noise3: optional precomputed [n_tax][3] from mdg_counts_reduce
 * (used when mism12 is NULL); both NULL -> noise fields are NaN.
 * out: [n_tax]. out_median / out_hpdi_lo / out_hpdi_hi: [n_tax][2*max_position] posterior
 * predictive summary of the PMD/all run (fits.py:442-446; df_fit_predictions fits.py:632-665).
 * Optional diagnostics (NULL to skip):
 *   out_samples [n_tax][6][num_samples][4]  constrained draws (q, A, c, phi); null runs fill A=c=NaN
 *   out_trace   [n_tax][6][num_warmup+num_samples][4] unconstrained state after every transition
 *   out_waic    [n_tax][6][2][2*max_position]  lppd_i and pWAIC_i (fits.py:152-158), 0 where unused
 */
int mdg_fit_batch(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position,
                  const int64_t* tax_id, const uint32_t* k, const uint32_t* N,
                  const uint32_t* mism12, const double* noise3,
                  const mdg_fit_config* cfg,
                  mdg_fit_result* out,
                  float* out_median, float* out_hpdi_lo, float* out_hpdi_hi,
                  double* out_samples, double* out_trace, double* out_waic);

/*
 * K3m — MAP-only screening of a dense batch: the six MAP fits of every TaxID (mdg_map_run), their Laplace
 * covariances and the likelihood-ratio statistic, with no NUTS run and no NUTS scratch. Synchronous; the
 * arguments and layouts are those of mdg_fit_batch (k, N: [n_tax][2*max_position]; mism12 / noise3 optional,
 * both NULL -> noise NaN). From cfg only the priors, phi_min and do_fwd_rev are read. No random numbers: the
 * result is a pure function of (k, N, cfg), so any partition of a batch is bit-identical, and the
 * all-position fits equal mdg_fit_batch's map_* fields bit for bit. Any n_tax is taken in one call (the work
 * is cut into pieces internally). Scratch is the ctx's own, apart from that of batches in flight through
 * mdg_fit_batch_submit. mdg_ctx_get_timings afterwards: map_ms, assemble_ms, total_ms, n_launches, and
 * leapfrogs[run] = gradient evaluations of that run kind summed over TaxIDs; the NUTS fields are 0.
 */
int mdg_map_batch(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position,
                  const int64_t* tax_id, const uint32_t* k, const uint32_t* N,
                  const uint32_t* mism12, const double* noise3,
                  const mdg_fit_config* cfg, mdg_map_result* out);

/*
 * K3p — profile intervals of D_max for rows of mdg_map_batch (see mdg_map_interval). `map` holds the rows
 * mdg_map_batch returned for the same k, N and cfg; every end of every PMD run it made (run kinds 0, 2, 4) is
 * profiled, at `level` (0 < level < 1; 0.68 is fit_results' HPDI level). Inner fits at fixed D are LM-damped
 * Newton over (logit q, logit(A / D), log(phi - phi_min)), warm-started from the nearest point already solved;
 * each end is bracketed by expanding from D^ +- 2 D_max_std towards the bound and refined by the Illinois method
 * to a bracket of 1e-9 or |h| <= 1e-7. A run with MDG_FIT_FAILED or MDG_FIT_MAP_NOT_CONVERGED gives NaN ends with
 * MDG_FIT_FAILED; a run not made (n_eval = 0, all NaN) gives NaN ends with flags = n_eval = 0. Synchronous; `mem` as for
 * mdg_map_batch; any n_tax in one call; no random numbers, so the result is a pure function of (k, N, cfg, map,
 * level). mdg_ctx_get_timings afterwards: map_ms (the profile kernel), total_ms, n_launches, and leapfrogs[0/2/4] =
 * the gradient evaluations spent on the ends of that run kind; the other fields are 0.
 */
int mdg_map_profile(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position,
                    const uint32_t* k, const uint32_t* N, const mdg_fit_config* cfg,
                    const mdg_map_result* map, double level, mdg_map_interval* out);

/*
 * K0 — tsv_parse: the step before the hot path (SURVEY.md 8f N2). Tokenises a mismatch-matrix
 * text file held in host memory into the SoA columns mdg_counts_reduce takes; replaces the
 * parsing half of dd.read_csv(..., sep="\t", header=None, names=columns) (counts.py:229-235).
 * Layouts: 22 tab-separated columns (counts.py:37-45: tax_id, tax_name, tax_rank, N_alignments,
 * strand, position, AA..TT) or the legacy 20 columns without tax_name / tax_rank that the shipped
 * data/input files use; a first line that does not start with a digit or '-' is a header and is
 * skipped. `mem` says where the OUTPUT columns live (the text is always a host pointer).
 * counts16 is [16][counts_stride]. name_span / rank_span (22-column layout, optional) receive
 * (byte offset, length) pairs into `text` so that the host can build the two string columns.
 * Errors: malformed line / number / value out of range -> MDG_ERR_INVALID with the line number
 * in the message; more data lines than `capacity` -> MDG_ERR_INVALID.
 */
int mdg_tsv_parse(mdg_ctx* ctx, int mem, const char* text, int64_t n_bytes, int64_t capacity,
                  int64_t* tax_id, uint32_t* n_alignments, uint8_t* is_reverse, uint8_t* pos0,
                  uint32_t* counts16, int64_t counts_stride, int64_t* name_span, int64_t* rank_span,
                  int64_t* out_n_rows /* host */, int32_t* out_n_cols /* host: 20 or 22 */);

/*
 * K8 — select_top: `--max-fits` on the device (SURVEY.md 8f N3). Replaces fits.extract_top_max_fits
 * (fits.py:736-744: df_counts.groupby("tax_id")["N_alignments"].sum().nlargest(max_fits), then the
 * rows of those TaxIDs in df_counts order) for the arrays mdg_counts_reduce produces.
 * Per-row inputs [n_rows]: tax_id_row, n_alignments_row, keep_row (the cut flags of
 * mdg_counts_reduce; NULL = every row counts). Per-TaxID inputs [n_tax]: tax_id, first_row (as
 * returned by mdg_counts_reduce; rows of a TaxID are contiguous). weight(t) = sum of
 * n_alignments_row over the kept rows of TaxID t. The min(n_top, n_tax) TaxIDs with the largest
 * weight are selected; ties at the cut go to the smaller tax id (pandas nlargest keep="first" on
 * the tax_id-sorted groupby index). out_index receives their positions in the per-TaxID arrays in
 * ascending order (= df_counts order), out_weight (optional, [n_tax]) all weights, *out_n (host
 * pointer) the number selected. tax ids must be unique (MDG_ERR_INVALID otherwise).
 */
int mdg_select_top(mdg_ctx* ctx, int mem, int64_t n_rows,
                   const int64_t* tax_id_row, const uint32_t* n_alignments_row, const uint8_t* keep_row,
                   int64_t n_tax, const int64_t* tax_id, const int64_t* first_row, int64_t n_top,
                   uint64_t* out_weight, int64_t* out_index, int64_t* out_n /* host pointer */);

/*
 * Asynchronous form of mdg_fit_batch: _submit enqueues the whole batch (H2D staging for MDG_HOST, kernels, D2H of
 * the results) and returns a ticket without waiting for the GPU; _wait blocks until that batch is complete, fills
 * `out_timings` (optional) and orders later work on the ctx stream after the batch. Up to MDG_MAX_INFLIGHT batches
 * per ctx may be in flight (MDG_ERR_BUSY otherwise); they run on separate internal streams with separate scratch, so
 * the next batch starts while the previous one is still finishing its longest chains: a NUTS chain is sequential, and
 * the tail of a batch is a handful of chains on an otherwise idle GPU. The same overlap is used between the chunks
 * of one large batch. All buffers (host or device) must stay valid and unmodified until _wait returns; for MDG_HOST
 * the copies overlap with compute only if the host buffers are pinned. Tickets should be waited for in submission
 * order. The caller drives one stream of batches per ctx, e.g. the per-file loop of main.py:43-66 or bench steps:
 *     submit(batch i+1); wait(batch i); consume(batch i); ...
 */
int mdg_fit_batch_submit(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position,
                         const int64_t* tax_id, const uint32_t* k, const uint32_t* N,
                         const uint32_t* mism12, const double* noise3,
                         const mdg_fit_config* cfg,
                         mdg_fit_result* out,
                         float* out_median, float* out_hpdi_lo, float* out_hpdi_hi,
                         double* out_samples, double* out_trace, double* out_waic,
                         int64_t* out_ticket /* host */);
int mdg_fit_batch_wait(mdg_ctx* ctx, int64_t ticket, mdg_timings* out_timings /* host, optional */);

/* building blocks exported for the parity tests (device evaluation of single functions) */

/* evaluate lgamma and digamma of x[0..n) on the GPU with the fit kernels' own routines */
int mdg_test_lgamma_digamma(mdg_ctx* ctx, int64_t n, const double* x /* host */,
                            double* out_lgamma /* host */, double* out_digamma /* host */);

/* log-joint (likelihood + priors [+ Jacobian]) and its gradient w.r.t. the unconstrained
 * parameters u (PMD: u_q,u_A,u_c,u_delta; null: u_q,u_delta), for n_eval parameter vectors of
 * ONE TaxID. model: 0 = PMD, 1 = null. lane_mask: 0 all, 1 forward only, 2 reverse only.
 * out_logp [n_eval], out_grad [n_eval][4], out_ll [n_eval][2*max_position] per-position
 * log-likelihood incl. log C(N,k). All pointers are host pointers. */
int mdg_test_logp_grad(mdg_ctx* ctx, int max_position, const uint32_t* k, const uint32_t* N,
                       const mdg_fit_config* cfg, int model, int lane_mask, int with_jacobian,
                       int64_t n_eval, const double* u,
                       double* out_logp, double* out_grad, double* out_ll);

/* the fit kernels' own table-driven exp and log at x[0..n) (log only where x > 0); host pointers */
int mdg_test_exp_log(mdg_ctx* ctx, int64_t n, const double* x, double* out_exp, double* out_log);

/* Philox4x32-10 block for (key, counter), 4 words out; n blocks; host pointers */
int mdg_test_philox(mdg_ctx* ctx, int64_t n, const uint32_t* key2, const uint32_t* ctr4,
                    uint32_t* out4);

/* n_draws BetaBinomial(alpha, beta, n) variates from the posterior predictive's own samplers (a Beta variate from two
 * Marsaglia-Tsang gammas, then Binomial by BINV / BTRS), draw i on the Philox stream keyed by (seed, tax id 12345) at
 * counter (0, i, MDG_RUN_PMD_ALL | purpose 6 << 8, i >> 32). Needs alpha > 0, beta > 0, n >= 0; out: host [n_draws] */
int mdg_test_betabinom_draws(mdg_ctx* ctx, uint64_t seed, int64_t n_draws, double alpha, double beta, double n,
                             double* out);

/* measured FP64 FMA peak of this GPU (dependent-free DFMA loop), in TFLOP/s */
int mdg_measure_fp64_peak(mdg_ctx* ctx, double* out_tflops);

#ifdef __cplusplus
}
#endif
#endif /* MDG_H */
