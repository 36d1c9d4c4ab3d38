/*
 * ppc_replay.c — CPU replay (plain C, FP64) of the posterior-predictive kernel K6 (ppc_kernel in
 * metadamage_b200/csrc/mdg_post_kernels.cuh). Test infrastructure only: compiled as one translation unit with
 * oracle/mdg_oracle.c, whose Philox streams (orc_make_key, c2word) and samplers (beta_variate, binomial_variate) it
 * uses unchanged. Its input is what mdg_fit_batch returns: the constrained draws (q, A, c, phi) of out_samples, so the
 * replay redraws each kernel item from the same parameter values and the same stream. It returns the integer draws;
 * the order statistics (median, HPDI) are taken in Python, independently of both C implementations.
 */
#include "../oracle/mdg_oracle.c"

/*
 * K6's item map, per TaxID: items j < 2P are the PMD/all run at dense position j; item 2P is the forward run at
 * dense 0 (D_max_forward); item 2P + 1 the reverse run at dense 0, or at dense P with reference_quirks = 0
 * (D_max_reverse, fits.py:343-348). Returns the run kind and sets the dense position.
 */
static int ppc_item(int P, int quirks, int j, int* dense) {
    if (j < 2 * P) { *dense = j; return MDG_RUN_PMD_ALL; }
    if (j == 2 * P) { *dense = 0; return MDG_RUN_PMD_FWD; }
    *dense = quirks ? 0 : P;
    return MDG_RUN_PMD_REV;
}

/* the items of TaxID t; returns the flat index of the first draw the samplers cannot take, or -1 */
static int64_t ppc_replay_tax(int64_t t, int P, int items, const int64_t* tax_id, const uint32_t* N,
                              const mdg_fit_config* cfg, const double* samples, uint32_t* y) {
    const int S = cfg->num_samples, R = 2 * P;
    for (int j = 0; j < items; ++j) {
        int dense;
        const int run = ppc_item(P, cfg->reference_quirks, j, &dense);
        const double n = (double)N[t * R + dense], x = (double)(dense < P ? dense : dense - P);
        if (!(n > 0)) continue;
        const double* smp = samples + ((size_t)t * MDG_NUM_RUNS + run) * (size_t)S * 4;
        for (int s = 0; s < S; ++s) {
            const double q = smp[s * 4], A = smp[s * 4 + 1], c = smp[s * 4 + 2], phi = smp[s * 4 + 3];
            double Dz = A * exp(x * log1p(-q)) + c;
            if (Dz > 1) Dz = 1;
            if (Dz < 0) Dz = 0;
            const double a = Dz * phi, b = (1 - Dz) * phi;
            /* q == 1 gives Dz = NaN at x = 0, and a NaN or infinite shape parameter never leaves the gamma loop */
            if (!(q > 0 && q < 1) || !isfinite(a) || !isfinite(b)) return (t * items + j) * S + s;
            orc_stream st;
            orc_make_key(cfg->seed, tax_id[t], st.key);
            st.c0 = 0; st.c1 = (uint32_t)s; st.c2 = c2word(run, P_PPC); st.c3 = (uint32_t)dense; st.have = 0;
            const double p = beta_variate(&st, a, b);
            y[(t * items + j) * S + s] = (uint32_t)binomial_variate(&st, n, p);
        }
    }
    return -1;
}

/*
 * y[t][j][s] (integer draws as uint32, like the kernel's sort keys) for the n_tax TaxIDs, items_per_tax = 2P (+ 2
 * with do_fwd_rev) items and S = num_samples draws. samples: [n_tax][6][S][4] constrained draws. TaxIDs whose
 * status has MDG_FIT_FAILED and items with N = 0 are skipped (y left as it was): the kernel and the assembly write
 * NaN there. Returns 0, or -1 with *bad = the flat index t * items_per_tax * S + j * S + s of the first draw whose q
 * is outside (0, 1) or whose Beta parameters are not finite.
 */
int orc_ppc_replay(int64_t n_tax, int P, const int64_t* tax_id, const uint32_t* N, const mdg_fit_config* cfg,
                   const uint32_t* status, const double* samples, uint32_t* y, int64_t* bad, int n_threads) {
    const int items = 2 * P + (cfg->do_fwd_rev ? 2 : 0);
    int64_t first = INT64_MAX;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#else
    (void)n_threads;
#endif
#pragma omp parallel for schedule(dynamic, 1) reduction(min : first)
    for (int64_t t = 0; t < n_tax; ++t) {
        if (status[t] & MDG_FIT_FAILED) continue;
        const int64_t b = ppc_replay_tax(t, P, items, tax_id, N, cfg, samples, y);
        if (b >= 0 && b < first) first = b;
    }
    *bad = first == INT64_MAX ? -1 : first;
    return first == INT64_MAX ? 0 : -1;
}
