// mdg_api.cu — the C-ABI of libmdgb200.so (include/mdg.h): context management, host<->device
// staging, kernel launches and CUDA-event timing for the counts (K1) and fit (K3-K7) paths.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <vector>
#include <algorithm>

#include "mdg_counts_kernel.cuh"
#include "mdg_counts_stream.cuh"
#include "mdg_tsv_kernel.cuh"
#include "mdg_select_kernel.cuh"
#include "mdg_post_kernels.cuh"
#include "mdg_map_batch_kernel.cuh"
#include "mdg_nuts_kernel.cuh"

namespace mdg {

static thread_local char g_error[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
}

// grow-only device buffer
struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return MDG_OK;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&ptr, bytes);
        if (e != cudaSuccess) {
            set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
            (void)cudaGetLastError();
            return MDG_ERR_NOMEM;
        }
        cap = bytes;
        return MDG_OK;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

constexpr int kNumBufs = 24;
constexpr int kNumEvents = 16;

}  // namespace mdg

// One fit lane = the streams, events and scratch of one chunk in flight. Two lanes per ctx: chunk c+1 (of the
// same batch or of the next submitted batch) starts under the tail of chunk c, which is a handful of long
// sequential chains on an otherwise idle GPU.
struct mdg_fit_lane {
    cudaStream_t main = nullptr, side[4] = {nullptr, nullptr, nullptr, nullptr};  // main: high priority; side: the four NUTS launches
    cudaEvent_t ev[5] = {};  // chunk begin, MAP end, NUTS end, predictive end, done (after assembly + D2H)
    cudaEvent_t fork_ev = nullptr, join_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    mdg::DevBuf rec, map, pred, counters, samples, waic, waic_acc[4];
    mdg::DevBuf chain_clock;  // development switch MDG_CHAIN_CLOCK=<file>
    mdg::DevBuf order;        // queue order of the chunk's TaxIDs: [chunk] int order, [chunk] bucket bytes, 3 x kOrderBuckets counters
    int clock_items = 0;
    unsigned long long* h_leap = nullptr;  // pinned [MDG_NUM_RUNS]
    bool busy = false;
    int owner = -1;          // ticket slot of the chunk in flight
    uint32_t launches = 0;
};

// One submitted batch (mdg_fit_batch_submit): staging buffers for MDG_HOST and the accumulated timings.
struct mdg_fit_ticket_slot {
    bool active = false;
    int64_t id = 0;
    cudaEvent_t ev_begin = nullptr;
    mdg::DevBuf in_tax, in_k, in_N, in_m12, in_noise, out_res, out_med, smp, trace, waic;
    mdg_timings t = {};
    double nuts_begin_ms = 0, nuts_end_ms = 0;
    bool have_nuts = false;
};

constexpr int kFitLanes = MDG_MAX_INFLIGHT;
constexpr int kFitTickets = MDG_MAX_INFLIGHT;

struct mdg_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[mdg::kNumEvents] = {};
    cudaEvent_t epoch = nullptr;       // time zero of mdg_timings.nuts_begin_ms / nuts_end_ms
    cudaEvent_t inputs_ready = nullptr;
    mdg::DevBuf buf[mdg::kNumBufs];
    mdg::DevBuf da_tables;             // sqrt(t) and t^-0.75 for t < kDaTable (dual averaging), filled at the first fit
    mdg_fit_lane lane[kFitLanes];
    mdg_fit_ticket_slot ticket[kFitTickets];
    int next_lane = 0;
    int64_t next_ticket_id = 1;
    double nuts_covered_until_ms = 0;  // union of NUTS intervals harvested so far ends here
    mdg_timings timings = {};
    // mdg_map_batch: staged inputs / outputs (MDG_HOST), per-run records, counters; apart from the fit lanes' scratch
    mdg::DevBuf map_in_tax, map_in_k, map_in_N, map_in_m12, map_in_noise, map_out, map_rec, map_counters;
};

using namespace mdg;

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

Priors make_priors(const mdg_fit_config& c) {
    Priors p;
    p.qa = c.q_prior_a; p.qb = c.q_prior_b;
    p.Aa = c.A_prior_a; p.Ab = c.A_prior_b;
    p.ca = c.c_prior_a; p.cb = c.c_prior_b;
    p.rate = c.phi_prior_rate; p.phi_min = c.phi_min;
    p.nlb_q = -(lgamma(p.qa) + lgamma(p.qb) - lgamma(p.qa + p.qb));
    p.nlb_A = -(lgamma(p.Aa) + lgamma(p.Ab) - lgamma(p.Aa + p.Ab));
    p.nlb_c = -(lgamma(p.ca) + lgamma(p.cb) - lgamma(p.ca + p.cb));
    p.log_rate = log(p.rate);
    return p;
}

// numpyro 0.4.1 hmc_util.build_adaptation_schedule: last index of every window
int adaptation_window_ends(int num_steps, int* ends) {
    int n = 0;
    if (num_steps < 20) { ends[n++] = num_steps - 1; return n; }
    int start_buffer = 75, end_buffer = 50, init_window = 25;
    if (start_buffer + end_buffer + init_window > num_steps) {
        start_buffer = (int)(0.15 * num_steps);
        end_buffer = (int)(0.1 * num_steps);
        init_window = num_steps - start_buffer - end_buffer;
    }
    ends[n++] = start_buffer - 1;
    const int end_window_start = num_steps - end_buffer;
    int next_size = init_window, next_start = start_buffer;
    while (next_start < end_window_start && n < kMaxWindows - 1) {
        int cur_start = next_start, cur_size = next_size;
        if (3 * cur_size <= end_window_start - cur_start) next_size = 2 * cur_size;
        else cur_size = end_window_start - cur_start;
        next_start = cur_start + cur_size;
        ends[n++] = next_start - 1;
    }
    ends[n++] = num_steps - 1;
    return n;
}

template <typename K>
int persistent_grid(K kernel, int threads, size_t smem, int num_sms, long long items, int items_per_block) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    if (per_sm < 1) per_sm = 1;
    if (const char* cap_env = getenv("MDG_MAX_CTAS_PER_SM")) {  // occupancy experiments
        int c = atoi(cap_env);
        if (c >= 1 && c < per_sm) per_sm = c;
    }
    long long want = (items + items_per_block - 1) / items_per_block;
    long long cap = (long long)per_sm * num_sms;
    return (int)std::max<long long>(1, std::min(want, cap));
}

constexpr int kNutsWarps = 4;
constexpr int kOrderMinChunk = 32768;  // TaxIDs per chunk from which the NUTS queue is ordered by coverage
constexpr int kMapWarps = 4;
constexpr int kPpcWarps = 4;

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

// K4, group layout: GW lanes per chain, rolled position loop (mdg_nuts_kernel.cuh)
template <int MODEL, int GW, int WARPS>
int launch_nuts_group(mdg_ctx* ctx, cudaStream_t st, FitLaunch fl, DevBuf& acc) {
    auto kern = nuts_group_kernel<MODEL, GW, WARPS>;
    const int n_obs = fl.n_items_all > 0 ? 2 * fl.P : fl.P;  // the launch's longest run
    fl.n_slots = (n_obs + 1 + GW - 1) / GW;  // index 0 is the spare
    size_t smem = (size_t)WARPS * nuts_warp_smem_bytes(fl.n_slots);
    // The NUTS launches of a chunk take over each other's CTA slots as CTAs retire. Shared memory is allocated
    // contiguously, so a retiring CTA's hole must fit the next launch's CTA: every launch asks for the same footprint
    // (static + dynamic), the largest one (PMD with all-position runs). Otherwise the SMs end up with three resident
    // CTAs instead of four (profiles/r02_chain_timeline.md: 8 016 live chains instead of 9 472).
    if (env_int("MDG_NUTS_UNIFORM_SMEM", 1)) {
        cudaFuncAttributes mine, big;
        MDG_CUDA_TRY(cudaFuncGetAttributes(&mine, kern));
        MDG_CUDA_TRY(cudaFuncGetAttributes(&big, nuts_group_kernel<0, GW, WARPS>));
        const size_t want = big.sharedSizeBytes + (size_t)WARPS * nuts_warp_smem_bytes((2 * fl.P + 1 + GW - 1) / GW);
        if (want > mine.sharedSizeBytes + smem) smem = want - mine.sharedSizeBytes;
    }
    MDG_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // One group slot per item up to the whole GPU. (Smaller grids that leave every group several items were measured:
    // 3 / 6 / 12 items per group cost 14 / 21 / 39 % at 10 000 TaxIDs per batch and 0 / 9 / 35 % at 40 000 — fewer
    // resident chains, and different kernels sharing an SM's instruction cache; profiles/r02_nuts_tuning.md.)
    const int per_group = std::max(1, env_int("MDG_ITEMS_PER_GROUP", 1));
    const int grid = persistent_grid(kern, WARPS * 32, smem, ctx->num_sms, fl.n_items, WARPS * (32 / GW) * per_group);
    int rc = acc.ensure((size_t)grid * WARPS * 4 * fl.n_slots * 32 * sizeof(double));
    if (rc) return rc;
    fl.waic_acc = acc.as<double>();
    kern<<<grid, WARPS * 32, smem, st>>>(fl);
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

template <int MODEL>
int launch_nuts_group_dispatch(mdg_ctx* ctx, cudaStream_t st, const FitLaunch& fl, DevBuf& acc, int gw) {
    if (gw == 16) return launch_nuts_group<MODEL, 16, kNutsWarps>(ctx, st, fl, acc);
    if (env_int("MDG_NUTS_WARPS", kNutsWarps) == 2) return launch_nuts_group<MODEL, 8, 2>(ctx, st, fl, acc);  // A/B: CTAs of two warps
    return launch_nuts_group<MODEL, 8, kNutsWarps>(ctx, st, fl, acc);
}

int launch_map(mdg_ctx* ctx, cudaStream_t st, const MapLaunch& ml, int npl) {
    const long long items = 2ll * ml.n_tax;
    if (npl == 1) {
        int grid = persistent_grid(map_kernel<1, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_kernel<1, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    } else if (npl == 2) {
        int grid = persistent_grid(map_kernel<2, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_kernel<2, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    } else {
        int grid = persistent_grid(map_kernel<4, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_kernel<4, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    }
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

int launch_map_batch(mdg_ctx* ctx, cudaStream_t st, const MapBatchLaunch& ml, int npl) {
    const long long items = (long long)ml.n_runs * ml.n_tax;
    if (npl == 1) {
        int grid = persistent_grid(map_batch_kernel<1, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_batch_kernel<1, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    } else if (npl == 2) {
        int grid = persistent_grid(map_batch_kernel<2, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_batch_kernel<2, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    } else {
        int grid = persistent_grid(map_batch_kernel<4, kMapWarps>, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        map_batch_kernel<4, kMapWarps><<<grid, kMapWarps * 32, 0, st>>>(ml);
    }
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

int npl_for(int n_obs, int gw) {
    int npl = (n_obs + gw - 1) / gw;
    return npl <= 1 ? 1 : (npl <= 2 ? 2 : 4);
}

float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

}  // namespace

extern "C" {

void mdg_ctx_destroy(mdg_ctx* ctx);

int mdg_version(void) { return MDG_VERSION; }

const char* mdg_last_error(void) { return g_error; }

int mdg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

void mdg_fit_config_default(mdg_fit_config* c) {
    memset(c, 0, sizeof *c);
    c->num_warmup = 500;
    c->num_samples = 1000;
    c->max_tree_depth = 10;
    c->do_map = 1;
    c->do_fwd_rev = 1;
    c->find_heuristic_step_size = 0;  // numpyro 0.4.1 default (HMC/NUTS(find_heuristic_step_size=False)); fits.py:382-387 passes no override
    c->reference_quirks = 1;
    c->pack_half_warps = 1;
    c->target_accept = 0.8;
    c->init_step_size = 1.0;
    c->max_delta_energy = 1000.0;
    c->init_radius = 2.0;
    c->hpdi_prob = 0.68;
    c->seed = 0;
    c->q_prior_a = 2; c->q_prior_b = 3;
    c->A_prior_a = 2; c->A_prior_b = 3;
    c->c_prior_a = 1; c->c_prior_b = 9;
    c->phi_prior_rate = 1.0 / 1000.0;
    c->phi_min = 2.0;
}

int mdg_ctx_create(int device, mdg_ctx** out) {
    if (!out) { set_error("mdg_ctx_create: out is NULL"); return MDG_ERR_INVALID; }
    int n = mdg_device_count();
    if (device < 0 || device >= n) {
        set_error("mdg_ctx_create: device %d not available (%d CUDA devices visible)", device, n);
        return MDG_ERR_CUDA;
    }
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    MDG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("mdg_ctx_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                  prop.major, prop.minor);
        return MDG_ERR_CUDA;
    }
    *out = nullptr;
    mdg_ctx* ctx = new mdg_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    // any failure below releases what was created so far (mdg_ctx_destroy tolerates null members)
    auto fail = [&](cudaError_t e, const char* what) {
        set_error("mdg_ctx_create: %s failed: %s", what, cudaGetErrorString(e));
        mdg_ctx_destroy(ctx);
        return MDG_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
    ctx->stream = ctx->own_stream;
    for (int i = 0; i < kNumEvents; ++i)
        if ((e = cudaEventCreate(&ctx->ev[i])) != cudaSuccess) return fail(e, "cudaEventCreate");
    if ((e = cudaEventCreate(&ctx->epoch)) != cudaSuccess) return fail(e, "cudaEventCreate");
    if ((e = cudaEventCreateWithFlags(&ctx->inputs_ready, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
    // The NUTS launches are persistent and fill every CTA slot of the GPU; the short kernels around them (MAP,
    // posterior predictive, assembly) of the OTHER batch in flight must not queue behind the NUTS CTAs that are
    // still waiting for a slot, or a batch could not complete (and the next one not be submitted) before the
    // following batch's NUTS launches are through: the lane's main stream gets the highest priority, the NUTS
    // streams the lowest.
    int prio_low = 0, prio_high = 0;
    if ((e = cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high)) != cudaSuccess) return fail(e, "cudaDeviceGetStreamPriorityRange");
    for (auto& ln : ctx->lane) {
        if ((e = cudaStreamCreateWithPriority(&ln.main, cudaStreamNonBlocking, prio_high)) != cudaSuccess) return fail(e, "cudaStreamCreate");
        for (int i = 0; i < 4; ++i)
            if ((e = cudaStreamCreateWithPriority(&ln.side[i], cudaStreamNonBlocking, prio_low)) != cudaSuccess) return fail(e, "cudaStreamCreate");
        for (int i = 0; i < 5; ++i)
            if ((e = cudaEventCreate(&ln.ev[i])) != cudaSuccess) return fail(e, "cudaEventCreate");
        if ((e = cudaEventCreateWithFlags(&ln.fork_ev, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
        for (int i = 0; i < 4; ++i)
            if ((e = cudaEventCreateWithFlags(&ln.join_ev[i], cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
        if ((e = cudaHostAlloc((void**)&ln.h_leap, MDG_NUM_RUNS * sizeof(unsigned long long), cudaHostAllocDefault)) != cudaSuccess)
            return fail(e, "cudaHostAlloc");
    }
    for (auto& tk : ctx->ticket)
        if ((e = cudaEventCreate(&tk.ev_begin)) != cudaSuccess) return fail(e, "cudaEventCreate");
    if ((e = cudaEventRecord(ctx->epoch, ctx->own_stream)) != cudaSuccess) return fail(e, "cudaEventRecord");
    if ((e = cudaEventSynchronize(ctx->epoch)) != cudaSuccess) return fail(e, "cudaEventSynchronize");
    *out = ctx;
    return MDG_OK;
}

void mdg_ctx_destroy(mdg_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    for (auto& ln : ctx->lane) {
        if (ln.main) cudaStreamSynchronize(ln.main);
        for (int i = 0; i < 4; ++i) if (ln.side[i]) cudaStreamSynchronize(ln.side[i]);
    }
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->buf) b.release();
    ctx->da_tables.release();
    for (int i = 0; i < kNumEvents; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->epoch) cudaEventDestroy(ctx->epoch);
    if (ctx->inputs_ready) cudaEventDestroy(ctx->inputs_ready);
    for (auto& ln : ctx->lane) {
        for (mdg::DevBuf* b : {&ln.rec, &ln.map, &ln.pred, &ln.counters, &ln.samples, &ln.waic, &ln.waic_acc[0], &ln.waic_acc[1],
                               &ln.waic_acc[2], &ln.waic_acc[3], &ln.chain_clock, &ln.order})
            b->release();
        for (int i = 0; i < 5; ++i) if (ln.ev[i]) cudaEventDestroy(ln.ev[i]);
        if (ln.fork_ev) cudaEventDestroy(ln.fork_ev);
        for (int i = 0; i < 4; ++i) {
            if (ln.join_ev[i]) cudaEventDestroy(ln.join_ev[i]);
            if (ln.side[i]) cudaStreamDestroy(ln.side[i]);
        }
        if (ln.main) cudaStreamDestroy(ln.main);
        if (ln.h_leap) cudaFreeHost(ln.h_leap);
    }
    for (mdg::DevBuf* b : {&ctx->map_in_tax, &ctx->map_in_k, &ctx->map_in_N, &ctx->map_in_m12, &ctx->map_in_noise, &ctx->map_out,
                           &ctx->map_rec, &ctx->map_counters})
        b->release();
    for (auto& tk : ctx->ticket) {
        for (mdg::DevBuf* b : {&tk.in_tax, &tk.in_k, &tk.in_N, &tk.in_m12, &tk.in_noise, &tk.out_res, &tk.out_med, &tk.smp, &tk.trace, &tk.waic})
            b->release();
        if (tk.ev_begin) cudaEventDestroy(tk.ev_begin);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int mdg_ctx_set_stream(mdg_ctx* ctx, void* cuda_stream) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    ctx->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return MDG_OK;
}

int mdg_ctx_synchronize(mdg_ctx* ctx) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    DeviceGuard guard(ctx->device);
    for (auto& ln : ctx->lane) MDG_CUDA_TRY(cudaStreamSynchronize(ln.main));
    MDG_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return MDG_OK;
}

int mdg_ctx_get_timings(mdg_ctx* ctx, mdg_timings* out) {
    if (!ctx || !out) { set_error("ctx/out is NULL"); return MDG_ERR_INVALID; }
    *out = ctx->timings;
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// K1
// ---------------------------------------------------------------------------------------------
int mdg_counts_reduce(mdg_ctx* ctx, int mem, int64_t n_rows, const int64_t* tax_id, const uint32_t* n_alignments,
                      const uint8_t* is_reverse, const uint8_t* pos0, const uint32_t* counts16,
                      int64_t counts_stride, int fwd_ref, int fwd_obs, int rev_ref, int rev_obs, int max_position,
                      uint32_t min_alignments, uint64_t min_y_sum, uint32_t* n_fwd_ref_row, uint32_t* n_rev_ref_row,
                      float* f_fwd_row, float* f_rev_row, int8_t* z_row, uint64_t* y_sum_total_row,
                      uint8_t* keep_row, int64_t* out_tax_id, uint32_t* out_n_alignments, int64_t* out_first_row,
                      uint32_t* out_k, uint32_t* out_N, double* out_noise, int64_t out_capacity, int64_t* out_n_tax) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (n_rows < 0 || !out_n_tax || out_capacity < 0 || max_position < 1 || max_position > MDG_MAX_POSITION || fwd_ref < 0 || fwd_ref > 3 ||
        fwd_obs < 0 || fwd_obs > 3 || rev_ref < 0 || rev_ref > 3 || rev_obs < 0 || rev_obs > 3 ||
        (mem != MDG_HOST && mem != MDG_DEVICE) || counts_stride < n_rows) {
        set_error("mdg_counts_reduce: invalid argument");
        return MDG_ERR_INVALID;
    }
    if (n_rows > 0 && (!tax_id || !n_alignments || !is_reverse || !pos0 || !counts16)) {
        set_error("mdg_counts_reduce: NULL input column");
        return MDG_ERR_INVALID;
    }
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    ctx->timings = mdg_timings{};
    *out_n_tax = 0;
    if (n_rows == 0) return MDG_OK;
    const int P = max_position, R = 2 * P;
    const size_t n = (size_t)n_rows;
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[0], st));

    // ---- stage inputs / outputs on the device for MDG_HOST ----
    CountsLaunch cl = {};
    const bool host = (mem == MDG_HOST);
    struct OutCopy { void* host_ptr; const void* dev_ptr; size_t elem; bool per_tax; };
    std::vector<OutCopy> copies;
    if (host) {
        // one arena for inputs, one for outputs
        size_t in_bytes = n * (8 + 4 + 1 + 1) + 256 * 5 + 16 * ((n * 4 + 255) & ~(size_t)255);
        int rc = ctx->buf[0].ensure(in_bytes);
        if (rc) return rc;
        unsigned char* base = ctx->buf[0].as<unsigned char>();
        size_t off = 0;
        auto put = [&](const void* src, size_t bytes) -> void* {
            void* d = base + off;
            cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st);
            off += (bytes + 255) & ~(size_t)255;
            return d;
        };
        cl.tax_id = (const long long*)put(tax_id, n * 8);
        cl.n_align = (const uint32_t*)put(n_alignments, n * 4);
        cl.is_rev = (const uint8_t*)put(is_reverse, n);
        cl.pos0 = (const uint8_t*)put(pos0, n);
        const size_t col_stride = ((n * 4 + 255) & ~(size_t)255) / 4;
        uint32_t* dcounts = (uint32_t*)(base + off);
        for (int c = 0; c < 16; ++c)
            cudaMemcpyAsync(dcounts + (size_t)c * col_stride, counts16 + (size_t)c * counts_stride, n * 4, cudaMemcpyHostToDevice, st);
        cl.counts16 = dcounts;
        cl.stride = (long long)col_stride;
        MDG_CUDA_TRY(cudaGetLastError());
        const size_t ncap = (size_t)out_capacity;
        size_t out_bytes = n * (4 + 4 + 4 + 4 + 1 + 8 + 1) + ncap * (8 + 4 + 8) + ncap * (size_t)R * 8 + ncap * 24 + 256 * 16;
        rc = ctx->buf[1].ensure(out_bytes);
        if (rc) return rc;
        unsigned char* ob = ctx->buf[1].as<unsigned char>();
        size_t oo = 0;
        auto take = [&](void* host_ptr, size_t elem, size_t count, bool per_tax) -> void* {
            if (!host_ptr) return nullptr;
            void* d = ob + oo;
            oo += (elem * count + 255) & ~(size_t)255;
            copies.push_back({host_ptr, d, elem, per_tax});
            return d;
        };
        cl.n_fwd_row = (uint32_t*)take(n_fwd_ref_row, 4, n, false);
        cl.n_rev_row = (uint32_t*)take(n_rev_ref_row, 4, n, false);
        cl.f_fwd_row = (float*)take(f_fwd_row, 4, n, false);
        cl.f_rev_row = (float*)take(f_rev_row, 4, n, false);
        cl.z_row = (int8_t*)take(z_row, 1, n, false);
        cl.y_row = (unsigned long long*)take(y_sum_total_row, 8, n, false);
        cl.keep_row = (uint8_t*)take(keep_row, 1, n, false);
        cl.out_tax = (long long*)take(out_tax_id, 8, ncap, true);
        cl.out_nal = (uint32_t*)take(out_n_alignments, 4, ncap, true);
        cl.out_first = (long long*)take(out_first_row, 8, ncap, true);
        cl.out_k = (uint32_t*)take(out_k, 4 * (size_t)R, ncap, true);
        cl.out_N = (uint32_t*)take(out_N, 4 * (size_t)R, ncap, true);
        cl.out_noise = (double*)take(out_noise, 24, ncap, true);
    } else {
        cl.tax_id = (const long long*)tax_id; cl.n_align = n_alignments; cl.is_rev = is_reverse; cl.pos0 = pos0;
        cl.counts16 = counts16; cl.stride = counts_stride;
        cl.n_fwd_row = n_fwd_ref_row; cl.n_rev_row = n_rev_ref_row; cl.f_fwd_row = f_fwd_row; cl.f_rev_row = f_rev_row;
        cl.z_row = z_row; cl.y_row = (unsigned long long*)y_sum_total_row; cl.keep_row = keep_row;
        cl.out_tax = (long long*)out_tax_id; cl.out_nal = out_n_alignments; cl.out_first = (long long*)out_first_row;
        cl.out_k = out_k; cl.out_N = out_N; cl.out_noise = out_noise;
    }
    cl.n_rows = n_rows;
    cl.fwd_ref = fwd_ref; cl.fwd_obs = fwd_obs; cl.rev_ref = rev_ref; cl.rev_obs = rev_obs;
    cl.P = P; cl.min_align = min_alignments; cl.min_y = min_y_sum;
    // staged columns: the reference-base rows of the two substitutions (+ all off-diagonals for noise)
    bool need[16] = {};
    for (int o = 0; o < 4; ++o) { need[fwd_ref * 4 + o] = true; need[rev_ref * 4 + o] = true; }
    if (cl.out_noise) for (int r = 0; r < 4; ++r) for (int o = 0; o < 4; ++o) if (r != o) need[r * 4 + o] = true;
    cl.ncols = 0;
    for (int c = 0; c < 16; ++c) {
        cl.col_slot[c] = -1;
        if (need[c]) { cl.col_slot[c] = cl.ncols; cl.col_id[cl.ncols++] = c; }
    }
    auto aligned16 = [](const void* p) { return ((uintptr_t)p & 15u) == 0; };
    cl.use_tma = aligned16(cl.tax_id) && aligned16(cl.n_align) && aligned16(cl.is_rev) && aligned16(cl.pos0) &&
                 aligned16(cl.counts16) && (cl.stride % 4 == 0);

    // output bases 16-byte aligned -> 128-bit stores
    cl.vec_out = aligned16(cl.n_fwd_row) && aligned16(cl.n_rev_row) && aligned16(cl.f_fwd_row) && aligned16(cl.f_rev_row) &&
                 aligned16(cl.z_row) && aligned16(cl.y_row) && aligned16(cl.keep_row);
    int rc = ctx->buf[2].ensure(64);
    if (rc) return rc;
    long long* d_ntax = ctx->buf[2].as<long long>();
    int* d_err = reinterpret_cast<int*>(d_ntax + 1);
    unsigned int* d_ticket = reinterpret_cast<unsigned int*>(d_ntax + 2);
    int h_err = 0;
    long long h_ntax = 0;
    const bool stream_design = getenv("MDG_COUNTS_TILES") == nullptr;  // the round-1 tile kernel stays selectable for A/B runs
    if (stream_design) {
        // ---- warp-synchronous streaming kernel (mdg_counts_stream.cuh): one warp per 128 rows ----
        const long long n_tiles = (n_rows + kStreamRows - 1) / kStreamRows;
        const size_t ncap_t = (size_t)out_capacity;
        const long long n_chunks_cap = (n_tiles + kScanChunk - 1) / kScanChunk;
        rc = ctx->buf[3].ensure((size_t)n_tiles * (8 + 8 + 4) + (size_t)n_chunks_cap * 8 + 64);
        if (rc) return rc;
        long long* d_tile_base = ctx->buf[3].as<long long>();
        long long* d_final_base = d_tile_base + n_tiles;
        long long* d_chunk = d_final_base + n_tiles;
        int* d_tile_cnt = reinterpret_cast<int*>(d_chunk + n_chunks_cap);
        const size_t tmp_bytes = ncap_t * (8 + 4 + 8 + 8 + (size_t)R * 8) + 256 * 8;
        rc = ctx->buf[21].ensure(tmp_bytes);
        if (rc) return rc;
        unsigned char* tb = ctx->buf[21].as<unsigned char>();
        size_t to = 0;
        auto tmp = [&](size_t bytes) { void* q = tb + to; to += (bytes + 255) & ~(size_t)255; return q; };
        // the noise kernel needs the first rows in final order even if the caller does not want them
        long long* d_first_final = cl.out_first ? cl.out_first : (cl.out_noise ? (long long*)tmp(ncap_t * 8) : nullptr);
        CountsPermute cp = {};
        cp.n_tiles = n_tiles; cp.tile_base = d_tile_base; cp.final_base = d_final_base; cp.tile_cnt = d_tile_cnt; cp.R = R;
        cp.chunk_off = d_chunk;
        cp.out_tax = cl.out_tax; cp.out_nal = cl.out_nal; cp.out_first = d_first_final; cp.out_k = cl.out_k; cp.out_N = cl.out_N;
        cp.out_noise = nullptr;
        CountsLaunch kl = cl;  // the tile kernel writes the per-TaxID rows into the temporaries
        kl.out_noise = nullptr;
        kl.out_first = nullptr;
        if (cl.out_tax) { cp.t_tax = (long long*)tmp(ncap_t * 8); kl.out_tax = (long long*)cp.t_tax; }
        if (cl.out_nal) { cp.t_nal = (uint32_t*)tmp(ncap_t * 4); kl.out_nal = (uint32_t*)cp.t_nal; }
        if (d_first_final) { cp.t_first = (long long*)tmp(ncap_t * 8); kl.out_first = (long long*)cp.t_first; }
        if (cl.out_k) { cp.t_k = (uint32_t*)tmp(ncap_t * R * 4); kl.out_k = (uint32_t*)cp.t_k; }
        if (cl.out_N) { cp.t_N = (uint32_t*)tmp(ncap_t * R * 4); kl.out_N = (uint32_t*)cp.t_N; }
        kl.tile_ticket = d_ticket;
        kl.kept_counter = reinterpret_cast<unsigned long long*>(d_ntax + 3);
        kl.tile_base = d_tile_base;
        kl.tile_cnt = d_tile_cnt;
        kl.capacity = out_capacity;
        kl.error_flag = d_err;
        MDG_CUDA_TRY(cudaMemsetAsync(d_ntax, 0, 64, st));
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
        counts_stream_kernel<<<(unsigned)((n_tiles + kStreamWarps - 1) / kStreamWarps), kStreamWarps * 32, 0, st>>>(kl);
        MDG_CUDA_TRY(cudaGetLastError());
        const long long n_chunks = (n_tiles + kScanChunk - 1) / kScanChunk;
        counts_scan_local_kernel<<<(unsigned)n_chunks, kScanChunk, 0, st>>>(d_tile_cnt, n_tiles, d_final_base, d_chunk);
        counts_scan_chunks_kernel<<<1, 32, 0, st>>>(d_chunk, n_chunks, d_ntax);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches += 1;
        counts_permute_kernel<<<(unsigned)((n_tiles + kPermuteWarps * kPermuteTiles - 1) / (kPermuteWarps * kPermuteTiles)), kPermuteWarps * 32, 0, st>>>(cp);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches += 3;
        if (cl.out_noise) {
            NoiseLaunch nl = {};
            nl.n_rows = n_rows; nl.tax_id = cl.tax_id; nl.is_rev = cl.is_rev; nl.pos0 = cl.pos0; nl.counts16 = cl.counts16;
            nl.stride = cl.stride; nl.P = P; nl.n_tax = d_ntax; nl.first_row = d_first_final; nl.out_noise = cl.out_noise;
            nl.capacity = out_capacity;
            counts_noise_kernel<<<(unsigned)std::max<long long>(1, std::min<long long>((out_capacity + 3) / 4, 16LL * ctx->num_sms)), 128, 0, st>>>(nl);
            MDG_CUDA_TRY(cudaGetLastError());
            ctx->timings.n_launches += 1;
        }
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
        MDG_CUDA_TRY(cudaMemcpyAsync(&h_err, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(&h_ntax, d_ntax, sizeof(long long), cudaMemcpyDeviceToHost, st));
        MDG_CUDA_TRY(cudaStreamSynchronize(st));
    } else {
    static const int ladder_T[3] = {448, 512, 512};
    static const int ladder_L[3] = {64, 512, MDG_MAX_SEGMENT_ROWS};
    const size_t row_bytes = (size_t)kCountsBytesPerRow + 4 * (size_t)cl.ncols;
    const size_t fixed_bytes = 16 + 16 + (size_t)kCountsWarps * 2 * R * 4 + 256;
    for (int step = 0; step < 3; ++step) {
        cl.T = ladder_T[step];
        cl.L = ladder_L[step];
        if (step == 0) if (const char* t_env = getenv("MDG_COUNTS_T")) { int tv = atoi(t_env); if (tv >= 64 && tv % 16 == 0) cl.T = tv; }  // tile-size experiments
        // shrink the tile (never the lookahead) until it fits the 227 KB of shared memory
        while (cl.T > 16 && fixed_bytes + row_bytes * (size_t)(cl.T + cl.L) > 227 * 1024 - 1024) cl.T -= 16;
        const int cap = cl.T + cl.L;
        const size_t smem = fixed_bytes + row_bytes * (size_t)cap;
        if (smem > 227 * 1024 - 1024) {
            set_error("mdg_counts_reduce: a TaxID spans more rows than one shared-memory tile can stage (%d with these options)",
                      (int)((227 * 1024 - 1024 - fixed_bytes) / row_bytes) - 16);
            return MDG_ERR_SEGMENT_TOO_LONG;
        }
        const long long n_tiles = (n_rows + cl.T - 1) / cl.T;
        // per-tile block bookkeeping + temporaries for the (unordered) dense rows
        const size_t ncap_t = (size_t)out_capacity;
        rc = ctx->buf[3].ensure((size_t)n_tiles * (8 + 8 + 4) + 64);
        if (rc) return rc;
        long long* d_tile_base = ctx->buf[3].as<long long>();
        long long* d_final_base = d_tile_base + n_tiles;
        int* d_tile_cnt = reinterpret_cast<int*>(d_final_base + n_tiles);
        const size_t tmp_bytes = ncap_t * (8 + 4 + 8 + 24 + (size_t)R * 8) + 256 * 8;
        rc = ctx->buf[21].ensure(tmp_bytes);
        if (rc) return rc;
        unsigned char* tb = ctx->buf[21].as<unsigned char>();
        size_t to = 0;
        auto tmp = [&](size_t bytes) { void* q = tb + to; to += (bytes + 255) & ~(size_t)255; return q; };
        CountsPermute cp = {};
        cp.n_tiles = n_tiles; cp.tile_base = d_tile_base; cp.final_base = d_final_base; cp.tile_cnt = d_tile_cnt; cp.R = R;
        cp.out_tax = cl.out_tax; cp.out_nal = cl.out_nal; cp.out_first = cl.out_first; cp.out_k = cl.out_k; cp.out_N = cl.out_N;
        cp.out_noise = cl.out_noise;
        CountsLaunch kl = cl;  // the tile kernel writes the per-TaxID rows into the temporaries
        if (cl.out_tax) { cp.t_tax = (long long*)tmp(ncap_t * 8); kl.out_tax = (long long*)cp.t_tax; }
        if (cl.out_nal) { cp.t_nal = (uint32_t*)tmp(ncap_t * 4); kl.out_nal = (uint32_t*)cp.t_nal; }
        if (cl.out_first) { cp.t_first = (long long*)tmp(ncap_t * 8); kl.out_first = (long long*)cp.t_first; }
        if (cl.out_k) { cp.t_k = (uint32_t*)tmp(ncap_t * R * 4); kl.out_k = (uint32_t*)cp.t_k; }
        if (cl.out_N) { cp.t_N = (uint32_t*)tmp(ncap_t * R * 4); kl.out_N = (uint32_t*)cp.t_N; }
        if (cl.out_noise) { cp.t_noise = (double*)tmp(ncap_t * 24); kl.out_noise = (double*)cp.t_noise; }
        kl.tile_ticket = d_ticket;
        kl.kept_counter = reinterpret_cast<unsigned long long*>(d_ntax + 3);
        kl.tile_base = d_tile_base;
        kl.tile_cnt = d_tile_cnt;
        kl.capacity = out_capacity;
        kl.error_flag = d_err;
        MDG_CUDA_TRY(cudaMemsetAsync(d_ntax, 0, 64, st));
        MDG_CUDA_TRY(cudaFuncSetAttribute(counts_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
        counts_reduce_kernel<<<(unsigned)n_tiles, kCountsThreads, smem, st>>>(kl);
        MDG_CUDA_TRY(cudaGetLastError());
        counts_scan_kernel<<<1, 1024, 0, st>>>(d_tile_cnt, n_tiles, d_final_base, d_ntax);
        MDG_CUDA_TRY(cudaGetLastError());
        counts_permute_kernel<<<(unsigned)((n_tiles + kPermuteWarps * kPermuteTiles - 1) / (kPermuteWarps * kPermuteTiles)), kPermuteWarps * 32, 0, st>>>(cp);
        MDG_CUDA_TRY(cudaGetLastError());
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
        ctx->timings.n_launches += 3;
        MDG_CUDA_TRY(cudaMemcpyAsync(&h_err, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(&h_ntax, d_ntax, sizeof(long long), cudaMemcpyDeviceToHost, st));
        MDG_CUDA_TRY(cudaStreamSynchronize(st));
        if (h_err != CE_SEGMENT_TOO_LONG) break;
    }
    }
    if (h_err == CE_SEGMENT_TOO_LONG) {
        set_error("mdg_counts_reduce: a TaxID has more than %d rows (rows must be grouped by tax_id)", MDG_MAX_SEGMENT_ROWS);
        return MDG_ERR_SEGMENT_TOO_LONG;
    }
    if (h_err == CE_CAPACITY) {
        set_error("mdg_counts_reduce: out_capacity (%lld) is smaller than the number of kept TaxIDs (%lld)",
                  (long long)out_capacity, h_ntax);
        return MDG_ERR_INVALID;
    }
    if (h_err == CE_OVERFLOW) {
        set_error("mdg_counts_reduce: a reference-base row sum exceeds uint32 (utils.py:338-339)");
        return MDG_ERR_OVERFLOW;
    }
    *out_n_tax = h_ntax;
    if (host) {
        for (const auto& c : copies) {
            size_t count = c.per_tax ? (size_t)h_ntax : n;
            if (count) MDG_CUDA_TRY(cudaMemcpyAsync(c.host_ptr, c.dev_ptr, c.elem * count, cudaMemcpyDeviceToHost, st));
        }
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->ev[1], ctx->ev[2]);
    ctx->timings.total_ms = elapsed(ctx->ev[0], ctx->ev[3]);
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// K1d: row order of df_counts
// ---------------------------------------------------------------------------------------------
int mdg_counts_order(mdg_ctx* ctx, int mem, int64_t n_rows, const int64_t* tax_id_row, const int8_t* z_row, const uint8_t* keep_row,
                     int64_t n_tax, const int64_t* first_row, const int64_t* tax_order, int64_t* out_perm, int64_t perm_capacity,
                     int64_t* out_n_rows) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (n_rows < 0 || n_tax < 0 || perm_capacity < 0 || !out_n_rows || (mem != MDG_HOST && mem != MDG_DEVICE) ||
        (n_tax > 0 && (!tax_id_row || !z_row || !first_row || !tax_order || !out_perm || n_rows <= 0))) {
        set_error("mdg_counts_order: invalid argument");
        return MDG_ERR_INVALID;
    }
    *out_n_rows = 0;
    ctx->timings = mdg_timings{};
    if (n_tax == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    const bool host = (mem == MDG_HOST);
    const size_t nr = (size_t)n_rows, nt = (size_t)n_tax;
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    int rc;
    OrderLaunch ol = {};
    ol.n_rows = n_rows; ol.n_tax = n_tax;
    ol.tax_id_row = reinterpret_cast<const long long*>(tax_id_row); ol.z_row = z_row; ol.keep_row = keep_row;
    ol.first_row = reinterpret_cast<const long long*>(first_row); ol.tax_order = reinterpret_cast<const long long*>(tax_order);
    ol.perm = reinterpret_cast<long long*>(out_perm);
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[0], st));
    if (host) {
        if ((rc = ctx->buf[22].ensure(up(nr * 8) + up(nr) + up(nr) + 2 * up(nt * 8) + up((size_t)perm_capacity * 8)))) return rc;
        unsigned char* b = ctx->buf[22].as<unsigned char>();
        size_t o = 0;
        auto put = [&](const void* src, size_t bytes) -> void* {
            void* d = b + o; o += up(bytes);
            if (src) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st);
            return d;
        };
        ol.tax_id_row = (const long long*)put(tax_id_row, nr * 8);
        ol.z_row = (const int8_t*)put(z_row, nr);
        void* kp = put(keep_row, nr);
        ol.keep_row = keep_row ? (const uint8_t*)kp : nullptr;
        ol.first_row = (const long long*)put(first_row, nt * 8);
        ol.tax_order = (const long long*)put(tax_order, nt * 8);
        ol.perm = (long long*)put(nullptr, (size_t)perm_capacity * 8);
        MDG_CUDA_TRY(cudaGetLastError());
    }
    if ((rc = ctx->buf[23].ensure(up(nt * 4) + up(nt * 8) + 256))) return rc;
    unsigned char* sb = ctx->buf[23].as<unsigned char>();
    ol.len_sorted = reinterpret_cast<int*>(sb);
    long long* d_start = reinterpret_cast<long long*>(sb + up(nt * 4));
    long long* d_total = reinterpret_cast<long long*>(sb + up(nt * 4) + up(nt * 8));
    ol.out_start = d_start;
    ol.error_flag = reinterpret_cast<int*>(d_total + 1);
    MDG_CUDA_TRY(cudaMemsetAsync(d_total, 0, 16, st));
    const unsigned grid = (unsigned)((n_tax + kOrderWarps - 1) / kOrderWarps);
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
    counts_order_kernel<0><<<grid, kOrderWarps * 32, 0, st>>>(ol);
    counts_scan_kernel<<<1, 1024, 0, st>>>(ol.len_sorted, n_tax, d_start, d_total);
    MDG_CUDA_TRY(cudaGetLastError());
    long long h_total = 0;
    int h_err = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_total, d_total, 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_err, ol.error_flag, 4, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    if (h_err) { set_error("mdg_counts_order: a TaxID has more than %d rows", MDG_MAX_SEGMENT_ROWS); return MDG_ERR_SEGMENT_TOO_LONG; }
    if (h_total > perm_capacity) {
        set_error("mdg_counts_order: %lld kept rows but room for %lld", h_total, (long long)perm_capacity);
        return MDG_ERR_INVALID;
    }
    counts_order_kernel<1><<<grid, kOrderWarps * 32, 0, st>>>(ol);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
    ctx->timings.n_launches = 3;
    if (host && h_total > 0) MDG_CUDA_TRY(cudaMemcpyAsync(out_perm, ol.perm, (size_t)h_total * 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->ev[1], ctx->ev[2]);
    ctx->timings.total_ms = elapsed(ctx->ev[0], ctx->ev[3]);
    *out_n_rows = h_total;
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// K0
// ---------------------------------------------------------------------------------------------
int mdg_tsv_parse(mdg_ctx* ctx, int mem, const char* text, int64_t n_bytes, int64_t capacity, int64_t* tax_id,
                  uint32_t* n_alignments, uint8_t* is_reverse, uint8_t* pos0, uint32_t* counts16, int64_t counts_stride,
                  int64_t* name_span, int64_t* rank_span, int64_t* out_n_rows, int32_t* out_n_cols) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (n_bytes < 0 || capacity < 0 || !out_n_rows || (mem != MDG_HOST && mem != MDG_DEVICE) || counts_stride < capacity ||
        (n_bytes > 0 && !text) || (capacity > 0 && (!tax_id || !n_alignments || !is_reverse || !pos0 || !counts16))) {
        set_error("mdg_tsv_parse: invalid argument");
        return MDG_ERR_INVALID;
    }
    *out_n_rows = 0;
    if (out_n_cols) *out_n_cols = 0;
    ctx->timings = mdg_timings{};
    if (n_bytes > 0) {
        // `text` is read on the host (header / layout detection): a device pointer is an error, not a crash
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, text) == cudaSuccess && attr.type == cudaMemoryTypeDevice) {
            set_error("mdg_tsv_parse: text must be a host pointer (mem only says where the OUTPUT columns live)");
            return MDG_ERR_INVALID;
        }
        (void)cudaGetLastError();
    }
    // blank lines at the end of the file are not rows (pandas.read_csv skips them too)
    while (n_bytes > 0 && (text[n_bytes - 1] == '\n' || text[n_bytes - 1] == '\r')) --n_bytes;
    // header detection and layout from the first line (host)
    int64_t first = 0;
    {
        int64_t e = 0;
        while (e < n_bytes && text[e] != '\n') ++e;
        const bool header = n_bytes > 0 && !((text[0] >= '0' && text[0] <= '9') || text[0] == '-');
        if (header) first = e < n_bytes ? e + 1 : n_bytes;
    }
    int64_t e1 = first;
    int tabs = 0;
    while (e1 < n_bytes && text[e1] != '\n') { tabs += text[e1] == '\t'; ++e1; }
    if (first >= n_bytes) return MDG_OK;  // no data lines
    const int n_cols = tabs + 1;
    if (n_cols != 20 && n_cols != 22) {
        set_error("mdg_tsv_parse: expected 20 or 22 tab-separated columns, got %d", n_cols);
        return MDG_ERR_INVALID;
    }
    if (out_n_cols) *out_n_cols = n_cols;
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[0], st));
    const bool host = (mem == MDG_HOST);
    const size_t cap = (size_t)capacity;
    TsvLaunch tl = {};
    tl.n_bytes = n_bytes; tl.first = first; tl.n_cols = n_cols; tl.capacity = capacity;
    tl.n_blocks = (n_bytes - first + kTsvBlockBytes - 1) / kTsvBlockBytes;
    int rc;
    if ((rc = ctx->buf[22].ensure((size_t)n_bytes + 16))) return rc;
    MDG_CUDA_TRY(cudaMemcpyAsync(ctx->buf[22].ptr, text, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    tl.text = ctx->buf[22].as<char>();
    if ((rc = ctx->buf[23].ensure((size_t)tl.n_blocks * 12 + (cap + 2) * 8 + 256))) return rc;
    tl.block_base = ctx->buf[23].as<long long>();
    tl.line_start = tl.block_base + tl.n_blocks;
    tl.block_cnt = reinterpret_cast<int*>(tl.line_start + cap + 2);
    if ((rc = ctx->buf[2].ensure(64))) return rc;
    long long* d_scal = ctx->buf[2].as<long long>();  // [0] newline total, [1] error flag (int), [2] error line
    tl.n_lines = d_scal; tl.error_flag = reinterpret_cast<int*>(d_scal + 1); tl.error_line = d_scal + 2;
    MDG_CUDA_TRY(cudaMemsetAsync(d_scal, 0, 64, st));
    struct OutCopy { void* host_ptr; const void* dev_ptr; size_t bytes_per_row; };
    std::vector<OutCopy> copies;
    if (host) {
        const size_t stride_dev = (cap + 63) & ~(size_t)63;
        if ((rc = ctx->buf[1].ensure(cap * (8 + 4 + 1 + 1 + 32) + 16 * stride_dev * 4 + 4096))) return rc;
        unsigned char* ob = ctx->buf[1].as<unsigned char>();
        size_t oo = 0;
        auto take = [&](void* hp, size_t elem) -> void* {
            void* d = ob + oo;
            oo += (elem * cap + 255) & ~(size_t)255;
            if (hp) copies.push_back({hp, d, elem});
            return d;
        };
        tl.tax_id = (long long*)take(tax_id, 8);
        tl.n_align = (uint32_t*)take(n_alignments, 4);
        tl.is_rev = (uint8_t*)take(is_reverse, 1);
        tl.pos0 = (uint8_t*)take(pos0, 1);
        tl.name_span = name_span ? (long long*)take(name_span, 16) : nullptr;
        tl.rank_span = rank_span ? (long long*)take(rank_span, 16) : nullptr;
        tl.counts16 = reinterpret_cast<uint32_t*>(ob + oo);
        tl.stride = (long long)stride_dev;
    } else {
        tl.tax_id = (long long*)tax_id; tl.n_align = n_alignments; tl.is_rev = is_reverse; tl.pos0 = pos0;
        tl.counts16 = counts16; tl.stride = counts_stride;
        tl.name_span = (long long*)name_span; tl.rank_span = (long long*)rank_span;
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
    tsv_count_kernel<<<(unsigned)tl.n_blocks, kTsvThreads, 0, st>>>(tl);
    MDG_CUDA_TRY(cudaGetLastError());
    counts_scan_kernel<<<1, 1024, 0, st>>>(tl.block_cnt, tl.n_blocks, tl.block_base, tl.n_lines);
    MDG_CUDA_TRY(cudaGetLastError());
    long long newlines = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(&newlines, tl.n_lines, 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    const long long n_lines = newlines + (text[n_bytes - 1] != '\n' ? 1 : 0);
    if (n_lines > capacity) {
        set_error("mdg_tsv_parse: %lld data lines but room for %lld rows", n_lines, (long long)capacity);
        return MDG_ERR_INVALID;
    }
    tsv_lines_kernel<<<(unsigned)tl.n_blocks, kTsvThreads, 0, st>>>(tl);
    MDG_CUDA_TRY(cudaGetLastError());
    if (n_lines > 0) {
        tsv_parse_kernel<<<(unsigned)((n_lines + kTsvThreads - 1) / kTsvThreads), kTsvThreads, 0, st>>>(tl, n_lines);
        MDG_CUDA_TRY(cudaGetLastError());
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
    ctx->timings.n_launches = 4;
    int h_err[2] = {0, 0};
    long long h_line = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(h_err, tl.error_flag, 4, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_line, tl.error_line, 8, cudaMemcpyDeviceToHost, st));
    if (host && n_lines > 0) {
        for (const auto& c : copies)
            MDG_CUDA_TRY(cudaMemcpyAsync(c.host_ptr, c.dev_ptr, c.bytes_per_row * (size_t)n_lines, cudaMemcpyDeviceToHost, st));
        for (int c = 0; c < 16; ++c)
            MDG_CUDA_TRY(cudaMemcpyAsync(counts16 + (size_t)c * counts_stride, tl.counts16 + (size_t)c * tl.stride,
                                         (size_t)n_lines * 4, cudaMemcpyDeviceToHost, st));
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->ev[1], ctx->ev[2]);
    ctx->timings.total_ms = elapsed(ctx->ev[0], ctx->ev[3]);
    if (h_err[0] != TE_NONE) {
        static const char* what[] = {"", "wrong number of fields", "malformed number", "value out of range", ""};
        set_error("mdg_tsv_parse: %s in data line %lld", what[h_err[0] & 3], h_line + 1);
        return MDG_ERR_INVALID;
    }
    *out_n_rows = n_lines;
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// K8 (N3): --max-fits on the device
// ---------------------------------------------------------------------------------------------
int mdg_select_top(mdg_ctx* ctx, int mem, int64_t n_rows, const int64_t* tax_id_row, const uint32_t* n_alignments_row,
                   const uint8_t* keep_row, int64_t n_tax, const int64_t* tax_id, const int64_t* first_row, int64_t n_top,
                   uint64_t* out_weight, int64_t* out_index, int64_t* out_n) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (n_rows < 0 || n_tax < 0 || n_top < 0 || !out_n || (mem != MDG_HOST && mem != MDG_DEVICE) ||
        (n_tax > 0 && (!tax_id_row || !n_alignments_row || !tax_id || !first_row || !out_index || n_rows <= 0))) {
        set_error("mdg_select_top: invalid argument");
        return MDG_ERR_INVALID;
    }
    MDG_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ctx->timings = mdg_timings{};
    const long long take = std::min<long long>(n_top, n_tax);
    *out_n = take;
    if (n_tax == 0 || (take == 0 && !out_weight)) { *out_n = 0; return MDG_OK; }
    const bool host = (mem == MDG_HOST);
    const size_t nr = (size_t)n_rows, nt = (size_t)n_tax;
    int rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[0], st));
    const long long* d_tax_row = reinterpret_cast<const long long*>(tax_id_row);
    const uint32_t* d_nal_row = n_alignments_row; const uint8_t* d_keep = keep_row;
    const long long* d_tax = reinterpret_cast<const long long*>(tax_id);
    const long long* d_first = reinterpret_cast<const long long*>(first_row);
    unsigned long long* d_weight = reinterpret_cast<unsigned long long*>(out_weight);
    long long* d_index = reinterpret_cast<long long*>(out_index);
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    if (host) {
        const size_t in_bytes = up(nr * 8) + up(nr * 4) + up(nr) + 2 * up(nt * 8);
        if ((rc = ctx->buf[22].ensure(in_bytes))) return rc;
        unsigned char* b = ctx->buf[22].as<unsigned char>();
        size_t o = 0;
        auto put = [&](const void* src, size_t bytes) -> void* {
            void* d = b + o; o += up(bytes);
            if (src) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st);
            return d;
        };
        d_tax_row = (const long long*)put(tax_id_row, nr * 8);
        d_nal_row = (const uint32_t*)put(n_alignments_row, nr * 4);
        void* kp = put(keep_row, nr);
        d_keep = keep_row ? (const uint8_t*)kp : nullptr;
        d_tax = (const long long*)put(tax_id, nt * 8);
        d_first = (const long long*)put(first_row, nt * 8);
        MDG_CUDA_TRY(cudaGetLastError());
    }
    const int n_blocks = (int)((n_tax + kTopThreads - 1) / kTopThreads);
    const size_t scratch = up(kTopPasses * 256 * 4) + up((size_t)n_blocks * 4) + up((size_t)n_blocks * 8) + up(8) +
                           ((host || !out_weight) ? up(nt * 8) : 0) + (host ? up((size_t)take * 8 + 8) : 0);
    if ((rc = ctx->buf[23].ensure(scratch))) return rc;
    unsigned char* sb = ctx->buf[23].as<unsigned char>();
    size_t so = 0;
    auto carve = [&](size_t bytes) { void* q = sb + so; so += up(bytes); return q; };
    TopLaunch tl = {};
    tl.n_tax = n_tax; tl.n_top = take;
    tl.hist = (unsigned int*)carve(kTopPasses * 256 * 4);
    tl.block_cnt = (int*)carve((size_t)n_blocks * 4);
    tl.block_base = (long long*)carve((size_t)n_blocks * 8);
    long long* d_total = (long long*)carve(8);
    if (host || !out_weight) d_weight = (unsigned long long*)carve(nt * 8);
    if (host) d_index = (long long*)carve((size_t)take * 8 + 8);
    tl.weight = d_weight; tl.tax_id = d_tax; tl.out_index = d_index;
    MDG_CUDA_TRY(cudaMemsetAsync(tl.hist, 0, kTopPasses * 256 * 4, st));
    top_weight_kernel<<<(unsigned)((n_tax * 32 + kTopThreads - 1) / kTopThreads), kTopThreads, 0, st>>>(
        n_rows, d_tax_row, d_nal_row, d_keep, n_tax, d_first, d_weight);
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    if (take == 0) {
        MDG_CUDA_TRY(cudaMemsetAsync(d_total, 0, 8, st));  // weights only
    } else if (take < n_tax) {
        const int hist_grid = std::min(n_blocks, 4 * ctx->num_sms);
        for (int pass = 0; pass < kTopPasses; ++pass) top_hist_kernel<<<hist_grid, kTopThreads, 0, st>>>(tl, pass);
        MDG_CUDA_TRY(cudaGetLastError());
        top_emit_kernel<0><<<n_blocks, kTopThreads, 0, st>>>(tl);
        counts_scan_kernel<<<1, 1024, 0, st>>>(tl.block_cnt, n_blocks, tl.block_base, d_total);
        top_emit_kernel<1><<<n_blocks, kTopThreads, 0, st>>>(tl);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches += kTopPasses + 3;
    } else {
        // everything is taken: threshold = smallest possible key (all-zero histograms replay to digit 0)
        top_emit_kernel<0><<<n_blocks, kTopThreads, 0, st>>>(tl);
        counts_scan_kernel<<<1, 1024, 0, st>>>(tl.block_cnt, n_blocks, tl.block_base, d_total);
        top_emit_kernel<1><<<n_blocks, kTopThreads, 0, st>>>(tl);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches += 3;
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[9], st));
    if (host) {
        if (take > 0) MDG_CUDA_TRY(cudaMemcpyAsync(out_index, d_index, (size_t)take * 8, cudaMemcpyDeviceToHost, st));
        if (out_weight) MDG_CUDA_TRY(cudaMemcpyAsync(out_weight, d_weight, nt * 8, cudaMemcpyDeviceToHost, st));
    }
    long long h_total = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_total, d_total, 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[9]);
    ctx->timings.total_ms = ms;
    if (h_total != take) {
        set_error("mdg_select_top: selected %lld of %lld (duplicate tax ids in the per-TaxID arrays?)", h_total, take);
        return MDG_ERR_INVALID;
    }
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// K3-K7
// ---------------------------------------------------------------------------------------------
}  // extern "C"

namespace {

double ms_since_epoch(mdg_ctx* ctx, cudaEvent_t ev) { return (double)elapsed(ctx->epoch, ev); }

// Wait (on the host) for the chunk in flight on a lane and book its CUDA-event times on its ticket.
int harvest_lane(mdg_ctx* ctx, mdg_fit_lane& ln) {
    if (!ln.busy) return MDG_OK;
    MDG_CUDA_TRY(cudaEventSynchronize(ln.ev[4]));
    mdg_fit_ticket_slot& tk = ctx->ticket[ln.owner];
    tk.t.map_ms += elapsed(ln.ev[0], ln.ev[1]);
    tk.t.nuts_ms += elapsed(ln.ev[1], ln.ev[2]);
    tk.t.ppc_ms += elapsed(ln.ev[2], ln.ev[3]);
    tk.t.assemble_ms += elapsed(ln.ev[3], ln.ev[4]);
    tk.t.total_ms = std::max(tk.t.total_ms, elapsed(tk.ev_begin, ln.ev[4]));
    tk.t.n_launches += ln.launches;
    for (int r = 0; r < MDG_NUM_RUNS; ++r) tk.t.leapfrogs[r] += ln.h_leap[r];
    // NUTS-active time as a union of intervals over everything harvested on this ctx (chunks of overlapping
    // batches run their NUTS launches concurrently; chunks are harvested in submission order)
    const double a = ms_since_epoch(ctx, ln.ev[1]), b = ms_since_epoch(ctx, ln.ev[2]);
    tk.t.nuts_union_ms += (float)std::max(0.0, b - std::max(a, ctx->nuts_covered_until_ms));
    ctx->nuts_covered_until_ms = std::max(ctx->nuts_covered_until_ms, b);
    if (!tk.have_nuts) { tk.nuts_begin_ms = a; tk.nuts_end_ms = b; tk.have_nuts = true; }
    tk.nuts_begin_ms = std::min(tk.nuts_begin_ms, a);
    tk.nuts_end_ms = std::max(tk.nuts_end_ms, b);
    if (ln.clock_items > 0) {  // development: append this chunk's per-chain start / end times to the file MDG_CHAIN_CLOCK names
        std::vector<unsigned long long> h((size_t)ln.clock_items * 2);
        MDG_CUDA_TRY(cudaMemcpy(h.data(), ln.chain_clock.ptr, h.size() * 8, cudaMemcpyDeviceToHost));
        const char* path = getenv("MDG_CHAIN_CLOCK");
        if (FILE* f = path ? fopen(path, "ab") : nullptr) { fwrite(h.data(), 8, h.size(), f); fclose(f); }
        ln.clock_items = 0;
    }
    ln.busy = false;
    ln.owner = -1;
    return MDG_OK;
}

}  // namespace

extern "C" {

int mdg_fit_batch_submit(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position, const int64_t* tax_id, const uint32_t* k,
                         const uint32_t* N, const uint32_t* mism12, const double* noise3, const mdg_fit_config* cfg,
                         mdg_fit_result* out, float* out_median, float* out_hpdi_lo, float* out_hpdi_hi,
                         double* out_samples, double* out_trace, double* out_waic, int64_t* out_ticket) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (!cfg || !out_ticket || n_tax < 0 || max_position < 1 || max_position > MDG_MAX_POSITION || (mem != MDG_HOST && mem != MDG_DEVICE)) {
        set_error("mdg_fit_batch: invalid argument");
        return MDG_ERR_INVALID;
    }
    if (cfg->num_samples < 1 || cfg->num_samples > 4096 || cfg->num_warmup < 0 || cfg->max_tree_depth < 1 ||
        cfg->max_tree_depth > kMaxTreeDepth || cfg->max_leapfrogs_per_run < 0) {
        set_error("mdg_fit_batch: need 1 <= num_samples <= 4096, num_warmup >= 0, 1 <= max_tree_depth <= %d, max_leapfrogs_per_run >= 0",
                  kMaxTreeDepth);
        return MDG_ERR_INVALID;
    }
    if (n_tax > 0 && (!tax_id || !k || !N || !out)) { set_error("mdg_fit_batch: NULL tax_id/k/N/out"); return MDG_ERR_INVALID; }
    int slot = -1;
    for (int i = 0; i < kFitTickets; ++i) if (!ctx->ticket[i].active) { slot = i; break; }
    if (slot < 0) {
        set_error("mdg_fit_batch_submit: %d batches are already in flight on this ctx; call mdg_fit_batch_wait first", kFitTickets);
        return MDG_ERR_BUSY;
    }
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    mdg_fit_ticket_slot& tk = ctx->ticket[slot];
    tk.t = mdg_timings{};
    tk.have_nuts = false;
    tk.nuts_begin_ms = tk.nuts_end_ms = 0;
    tk.id = ctx->next_ticket_id++;
    tk.active = true;
    *out_ticket = tk.id;
    MDG_CUDA_TRY(cudaEventRecord(tk.ev_begin, st));
    if (n_tax == 0) return MDG_OK;
    const int P = max_position, R = 2 * P, S = cfg->num_samples, W = cfg->num_warmup;
    const bool host = (mem == MDG_HOST);
    const bool fwd_rev = cfg->do_fwd_rev != 0;
    const Priors pr = make_priors(*cfg);

    const int sample_runs = out_samples ? MDG_NUM_RUNS : (fwd_rev ? 3 : 1);
    const int items_per_tax = R + (fwd_rev ? 2 : 0);
    // TaxIDs per chunk: every chunk ends with the tail of its four NUTS launches (the next chunk starts under
    // it on the other lane), so chunks are as large as ~8 GB of scratch per lane allows (posterior draws
    // dominate: 96 KB per TaxID at S = 1000)
    long long chunk_cap = 65536;
    {
        const size_t per_tax = (size_t)sample_runs * S * 4 * 8 + (size_t)MDG_NUM_RUNS * (sizeof(RunRecord) + 2 * R * 8) +
                               (size_t)items_per_tax * 3 * 8 + 2 * sizeof(MapRecord);
        while (chunk_cap > 4096 && (size_t)chunk_cap * per_tax > ((size_t)8 << 30)) chunk_cap /= 2;
        if (const char* e = getenv("MDG_FIT_CHUNK")) { const long long v = atoll(e); if (v >= 1 && v <= (1 << 20)) chunk_cap = v; }  // tests
    }
    const long long chunk_max = std::min<long long>(n_tax, chunk_cap);

    // ---- staged inputs / outputs for MDG_HOST (whole batch, owned by the ticket) ----
    int rc;
    const int64_t* d_tax = tax_id; const uint32_t* d_k = k; const uint32_t* d_N = N; const uint32_t* d_m12 = mism12;
    const double* d_noise = noise3;
    mdg_fit_result* d_out = out; float* d_med = out_median; float* d_lo = out_hpdi_lo; float* d_hi = out_hpdi_hi;
    double* d_samples = out_samples; double* d_trace = out_trace; double* d_waic_user = out_waic;
    const size_t nt = (size_t)n_tax;
    auto bail = [&](int code) { tk.active = false; return code; };
    if (host) {
        if ((rc = tk.in_tax.ensure(nt * 8))) return bail(rc);
        if ((rc = tk.in_k.ensure(nt * R * 4))) return bail(rc);
        if ((rc = tk.in_N.ensure(nt * R * 4))) return bail(rc);
        MDG_CUDA_TRY(cudaMemcpyAsync(tk.in_tax.ptr, tax_id, nt * 8, cudaMemcpyHostToDevice, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(tk.in_k.ptr, k, nt * R * 4, cudaMemcpyHostToDevice, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(tk.in_N.ptr, N, nt * R * 4, cudaMemcpyHostToDevice, st));
        d_tax = tk.in_tax.as<int64_t>(); d_k = tk.in_k.as<uint32_t>(); d_N = tk.in_N.as<uint32_t>();
        if (mism12) {
            if ((rc = tk.in_m12.ensure(nt * R * 12 * 4))) return bail(rc);
            MDG_CUDA_TRY(cudaMemcpyAsync(tk.in_m12.ptr, mism12, nt * R * 12 * 4, cudaMemcpyHostToDevice, st));
            d_m12 = tk.in_m12.as<uint32_t>();
        }
        if (noise3) {
            if ((rc = tk.in_noise.ensure(nt * 24))) return bail(rc);
            MDG_CUDA_TRY(cudaMemcpyAsync(tk.in_noise.ptr, noise3, nt * 24, cudaMemcpyHostToDevice, st));
            d_noise = tk.in_noise.as<double>();
        }
        if ((rc = tk.out_res.ensure(nt * sizeof(mdg_fit_result)))) return bail(rc);
        d_out = tk.out_res.as<mdg_fit_result>();
        if ((rc = tk.out_med.ensure(nt * R * 4 * 3))) return bail(rc);
        d_med = tk.out_med.as<float>(); d_lo = d_med + nt * R; d_hi = d_lo + nt * R;
        if (out_samples) {
            if ((rc = tk.smp.ensure(nt * MDG_NUM_RUNS * S * 4 * 8))) return bail(rc);
            d_samples = tk.smp.as<double>();
        }
        if (out_trace) {
            if ((rc = tk.trace.ensure(nt * MDG_NUM_RUNS * (size_t)(W + S) * 4 * 8))) return bail(rc);
            d_trace = tk.trace.as<double>();
        }
        if (out_waic) {
            if ((rc = tk.waic.ensure(nt * MDG_NUM_RUNS * 2 * R * 8))) return bail(rc);
            d_waic_user = tk.waic.as<double>();
        }
    } else {
        if (!d_med || !d_lo || !d_hi) {
            if ((rc = tk.out_med.ensure(nt * R * 4 * 3))) return bail(rc);
            float* base = tk.out_med.as<float>();
            if (!d_med) d_med = base;
            if (!d_lo) d_lo = base + nt * R;
            if (!d_hi) d_hi = base + 2 * nt * R;
        }
    }
    if (!ctx->da_tables.ptr) {
        // the same libm calls as the reference arithmetic (t^-0.75 by pow, sqrt), made once on the host
        std::vector<double> tab(2 * kDaTable);
        for (int t = 0; t < kDaTable; ++t) { tab[t] = sqrt((double)t); tab[kDaTable + t] = t ? pow((double)t, -0.75) : 0.0; }
        if ((rc = ctx->da_tables.ensure(tab.size() * sizeof(double)))) return bail(rc);
        MDG_CUDA_TRY(cudaMemcpyAsync(ctx->da_tables.ptr, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        MDG_CUDA_TRY(cudaStreamSynchronize(st));  // `tab` is a stack-lifetime source
    }
    if (d_trace) MDG_CUDA_TRY(cudaMemsetAsync(d_trace, 0xFF, nt * MDG_NUM_RUNS * (size_t)(W + S) * 4 * 8, st));
    if (out_samples) MDG_CUDA_TRY(cudaMemsetAsync(d_samples, 0xFF, nt * MDG_NUM_RUNS * (size_t)S * 4 * 8, st));
    // everything enqueued so far on the ctx stream (the caller's producers of the inputs, the copies above)
    // precedes the chunks, which run on the lanes' own streams
    MDG_CUDA_TRY(cudaEventRecord(ctx->inputs_ready, st));

    for (long long c0 = 0; c0 < n_tax; c0 += chunk_cap) {
        const int nc = (int)std::min<long long>(chunk_cap, n_tax - c0);
        mdg_fit_lane& ln = ctx->lane[ctx->next_lane];
        ctx->next_lane = (ctx->next_lane + 1) % kFitLanes;
        if ((rc = harvest_lane(ctx, ln))) return bail(rc);  // the lane's previous chunk (host wait only if it is still running)
        // ---- per-lane scratch ----
        if ((rc = ln.rec.ensure((size_t)chunk_max * MDG_NUM_RUNS * sizeof(RunRecord)))) return bail(rc);
        if ((rc = ln.map.ensure((size_t)chunk_max * 2 * sizeof(MapRecord)))) return bail(rc);
        if ((rc = ln.pred.ensure((size_t)chunk_max * items_per_tax * 3 * sizeof(double)))) return bail(rc);
        if ((rc = ln.counters.ensure(256))) return bail(rc);  // work counters + leapfrog totals
        if (!out_samples && (rc = ln.samples.ensure((size_t)chunk_max * sample_runs * S * 4 * sizeof(double)))) return bail(rc);
        if (!out_waic && (rc = ln.waic.ensure((size_t)chunk_max * MDG_NUM_RUNS * 2 * R * sizeof(double)))) return bail(rc);
        cudaStream_t ls = ln.main;
        const uint32_t launches_before = ctx->timings.n_launches;
        MDG_CUDA_TRY(cudaStreamWaitEvent(ls, ctx->inputs_ready, 0));
        unsigned int* d_counters = ln.counters.as<unsigned int>();                            // [8]
        unsigned long long* d_leap = reinterpret_cast<unsigned long long*>(d_counters + 16);  // [6]
        RunRecord* d_rec = ln.rec.as<RunRecord>();
        MapRecord* d_map = ln.map.as<MapRecord>();
        double* d_pred = ln.pred.as<double>();
        double* d_waic = d_waic_user ? d_waic_user + (size_t)c0 * MDG_NUM_RUNS * 2 * R : ln.waic.as<double>();
        double* d_smp = out_samples ? d_samples + (size_t)c0 * MDG_NUM_RUNS * S * 4 : ln.samples.as<double>();
        MDG_CUDA_TRY(cudaMemsetAsync(d_counters, 0, 256, ls));
        MDG_CUDA_TRY(cudaMemsetAsync(d_waic, 0, (size_t)nc * MDG_NUM_RUNS * 2 * R * 8, ls));
        MDG_CUDA_TRY(cudaMemsetAsync(d_rec, 0, (size_t)nc * MDG_NUM_RUNS * sizeof(RunRecord), ls));

        // ---- K3 MAP ----
        MDG_CUDA_TRY(cudaEventRecord(ln.ev[0], ls));
        if (cfg->do_map) {
            MapLaunch ml = {};
            ml.tax_id = d_tax + c0; ml.k = d_k + (size_t)c0 * R; ml.N = d_N + (size_t)c0 * R;
            ml.n_tax = nc; ml.P = P; ml.pr = pr; ml.work_counter = d_counters + 0; ml.rec = d_map;
            if ((rc = launch_map(ctx, ls, ml, npl_for(R, 32)))) return bail(rc);
        }
        MDG_CUDA_TRY(cudaEventRecord(ln.ev[1], ls));

        // ---- K4 NUTS: four launches on four streams (they share the SMs as CTAs retire) ----
        FitLaunch fl = {};
        fl.tax_id = d_tax + c0; fl.k = d_k + (size_t)c0 * R; fl.N = d_N + (size_t)c0 * R;
        fl.n_tax = nc; fl.P = P; fl.cfg = *cfg; fl.pr = pr;
        fl.n_windows = adaptation_window_ends(W, fl.win_end);
        fl.rec = d_rec; fl.waic = d_waic; fl.samples = d_smp; fl.sample_runs = sample_runs;
        fl.da_sqrt = ctx->da_tables.as<double>(); fl.da_pow = fl.da_sqrt + kDaTable;
        fl.trace = d_trace ? d_trace + (size_t)c0 * MDG_NUM_RUNS * (W + S) * 4 : nullptr;
        for (int r = 0; r < MDG_NUM_RUNS; ++r) fl.sample_slot[r] = out_samples ? r : ((r & 1) ? -1 : r / 2);
        // queue order: TaxIDs from both ends of the coverage range first (mdg_fit_kernels.cuh), for chunks long enough to
        // hide a chain that starts early (a 10 000-TaxID batch ends with its longest chain whatever the order, and pays
        // 1.3 % for it: NUTS 678 -> 687 ms); MDG_NUTS_ORDER=0: never, 2: always
        const int order_mode = env_int("MDG_NUTS_ORDER", 1);
        if (order_mode == 2 || (order_mode == 1 && nc >= kOrderMinChunk)) {
            const size_t off_bucket = (size_t)chunk_max * sizeof(int), off_cnt = (off_bucket + (size_t)chunk_max + 15) & ~(size_t)15;
            if ((rc = ln.order.ensure(off_cnt + 3 * kOrderBuckets * sizeof(unsigned int)))) return bail(rc);
            int* d_order = ln.order.as<int>();
            unsigned char* d_bucket = ln.order.as<unsigned char>() + off_bucket;
            unsigned int* d_cnt = reinterpret_cast<unsigned int*>(ln.order.as<unsigned char>() + off_cnt);
            MDG_CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 3 * kOrderBuckets * sizeof(unsigned int), ls));
            nuts_order_count_kernel<<<(nc + 255) / 256, 256, 0, ls>>>(fl.N, nc, R, d_bucket, d_cnt);
            nuts_order_offsets_kernel<<<1, 32, 0, ls>>>(d_cnt);
            nuts_order_scatter_kernel<<<(nc + 255) / 256, 256, 0, ls>>>(d_bucket, nc, d_cnt, d_order);
            MDG_CUDA_TRY(cudaGetLastError());
            ctx->timings.n_launches += 3;
            fl.order = d_order;
        }
        // the forward / reverse runs of the first 1/16 of that order go before everything else: the worst stragglers
        // measured (850 585 and 247 182 leapfrogs in one run; mean 9 800) are forward- or reverse-only runs of TaxIDs with
        // 60-110 reads, and a chain that long must start at once to end inside its batch (profiles/r02_chain_timeline.md)
        {
            const int frac = env_int("MDG_NUTS_PRIO_FRAC", 16);
            fl.n_prio = (fwd_rev && fl.order != nullptr && frac > 0) ? nc / frac : 0;
        }
        if (getenv("MDG_CHAIN_CLOCK")) {
            if ((rc = ln.chain_clock.ensure((size_t)chunk_max * MDG_NUM_RUNS * 16))) return bail(rc);
            MDG_CUDA_TRY(cudaMemsetAsync(ln.chain_clock.ptr, 0, (size_t)nc * MDG_NUM_RUNS * 16, ls));
            fl.chain_clock = ln.chain_clock.as<unsigned long long>();
            ln.clock_items = nc * MDG_NUM_RUNS;
        }
        // Overlap with the chunk in flight on another lane is wanted for its TAIL only (a few long chains on an
        // otherwise idle GPU), not for its bulk: two different NUTS kernels sharing the SMs evict each other from
        // the instruction cache (measured: -2..-5 % with unrestricted overlap). So this chunk's NUTS launches wait
        // until the other chunk's first three launches are through and only its last one (null model, all
        // positions: short, uniform chains) is still running.
        for (auto& other : ctx->lane)
            if (&other != &ln && other.busy)
                for (int i = 1; i < 4; ++i) MDG_CUDA_TRY(cudaStreamWaitEvent(ls, other.join_ev[i], 0));
        MDG_CUDA_TRY(cudaEventRecord(ln.fork_ev, ls));
        for (int i = 0; i < 4; ++i) MDG_CUDA_TRY(cudaStreamWaitEvent(ln.side[i], ln.fork_ev, 0));
        {
            // Launch order = dispatch order of the persistent CTAs: the kernels share the SMs as CTAs
            // retire, so the whole step behaves like one list schedule over all (TaxID, run) items.
            // PMD chains are long and heavy-tailed (adapted step size; max ~8x the mean), null chains
            // short and uniform: PMD first, null last fills the tail (profiles/r01_nuts_tuning.md).
            FitLaunch a = fl;  // PMD, all positions
            a.n_items = nc; a.n_items_all = nc; a.n_prio = 0; a.work_counter = d_counters + 1;
            FitLaunch b = a;   // null, all positions
            b.work_counter = d_counters + 2;
            FitLaunch c = fl, d = fl;  // PMD / null, forward-only and reverse-only
            c.work_counter = d_counters + 3; d.work_counter = d_counters + 4;
            c.n_items = 2 * nc; d.n_items = 2 * nc; c.n_items_all = 0; d.n_items_all = 0; c.n_prio = 0; d.n_prio = 0;
            const int gw_all = env_int("MDG_GW_ALL", 8), gw_half = env_int("MDG_GW_HALF", 8);  // lanes per chain (A/B runs: 16)
            if (fwd_rev && env_int("MDG_NUTS_MERGE", 1)) {
                // One launch and ONE queue per model: the all-position runs first (the longest chains), then the
                // forward-only / reverse-only runs. A group that finishes a chain always finds the next item until the
                // model's whole queue is empty, so the only hand-over between launches (CTA slots are released per CTA,
                // i.e. when the last of its 16 chains ends) is PMD -> null.
                a.n_items = 3 * nc; b.n_items = 3 * nc;
                a.n_prio = fl.n_prio; b.n_prio = fl.n_prio;
                if ((rc = launch_nuts_group_dispatch<0>(ctx, ln.side[3], a, ln.waic_acc[0], gw_all))) return bail(rc);
                if ((rc = launch_nuts_group_dispatch<1>(ctx, ln.side[0], b, ln.waic_acc[1], gw_all))) return bail(rc);
            } else if (env_int("MDG_NUTS_A_FIRST", 1)) {
                if ((rc = launch_nuts_group_dispatch<0>(ctx, ln.side[3], a, ln.waic_acc[0], gw_all))) return bail(rc);
                if (fwd_rev && (rc = launch_nuts_group_dispatch<0>(ctx, ln.side[1], c, ln.waic_acc[2], gw_half))) return bail(rc);
                if (fwd_rev && (rc = launch_nuts_group_dispatch<1>(ctx, ln.side[2], d, ln.waic_acc[3], gw_half))) return bail(rc);
                if ((rc = launch_nuts_group_dispatch<1>(ctx, ln.side[0], b, ln.waic_acc[1], gw_all))) return bail(rc);
            } else {
                if (fwd_rev && (rc = launch_nuts_group_dispatch<0>(ctx, ln.side[1], c, ln.waic_acc[2], gw_half))) return bail(rc);
                if ((rc = launch_nuts_group_dispatch<0>(ctx, ln.side[3], a, ln.waic_acc[0], gw_all))) return bail(rc);
                if (fwd_rev && (rc = launch_nuts_group_dispatch<1>(ctx, ln.side[2], d, ln.waic_acc[3], gw_half))) return bail(rc);
                if ((rc = launch_nuts_group_dispatch<1>(ctx, ln.side[0], b, ln.waic_acc[1], gw_all))) return bail(rc);
            }
        }
        for (int i = 0; i < 4; ++i) {
            MDG_CUDA_TRY(cudaEventRecord(ln.join_ev[i], ln.side[i]));
            MDG_CUDA_TRY(cudaStreamWaitEvent(ls, ln.join_ev[i], 0));
        }
        MDG_CUDA_TRY(cudaEventRecord(ln.ev[2], ls));

        // ---- K6 posterior predictive ----
        {
            PpcLaunch pl = {};
            pl.tax_id = d_tax + c0; pl.N = d_N + (size_t)c0 * R; pl.n_tax = nc; pl.P = P; pl.cfg = *cfg; pl.pr = pr;
            pl.samples = d_smp; pl.sample_runs = sample_runs;
            for (int r = 0; r < MDG_NUM_RUNS; ++r) pl.sample_slot[r] = fl.sample_slot[r];
            pl.rec = d_rec; pl.work_counter = d_counters + 5; pl.items_per_tax = items_per_tax;
            int sp = 64;
            while (sp < S) sp <<= 1;
            pl.s_pad = sp;
            pl.pred = d_pred;
            const size_t smem = (size_t)kPpcWarps * sp * 4;
            MDG_CUDA_TRY(cudaFuncSetAttribute(ppc_kernel<kPpcWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int grid = persistent_grid(ppc_kernel<kPpcWarps>, kPpcWarps * 32, smem, ctx->num_sms, (long long)nc * items_per_tax, kPpcWarps);
            ppc_kernel<kPpcWarps><<<grid, kPpcWarps * 32, smem, ls>>>(pl);
            MDG_CUDA_TRY(cudaGetLastError());
            ctx->timings.n_launches++;
        }
        MDG_CUDA_TRY(cudaEventRecord(ln.ev[3], ls));

        // ---- K5/K7 assembly ----
        {
            AssembleLaunch al = {};
            al.tax_id = d_tax + c0; al.k = d_k + (size_t)c0 * R; al.N = d_N + (size_t)c0 * R;
            al.mism12 = d_m12 ? d_m12 + (size_t)c0 * R * 12 : nullptr;
            al.noise3 = d_noise ? d_noise + (size_t)c0 * 3 : nullptr;
            al.n_tax = nc; al.P = P; al.cfg = *cfg; al.rec = d_rec; al.map = cfg->do_map ? d_map : nullptr;
            al.waic = d_waic; al.pred = d_pred; al.items_per_tax = items_per_tax;
            al.out = d_out + c0; al.out_median = d_med + (size_t)c0 * R; al.out_lo = d_lo + (size_t)c0 * R;
            al.out_hi = d_hi + (size_t)c0 * R; al.leapfrog_totals = d_leap;
            assemble_kernel<<<(nc + 127) / 128, 128, 0, ls>>>(al);
            MDG_CUDA_TRY(cudaGetLastError());
            ctx->timings.n_launches++;
        }
        // ---- this chunk's results back to the caller's host buffers ----
        if (host) {
            const size_t o = (size_t)c0, n_ = (size_t)nc;
            MDG_CUDA_TRY(cudaMemcpyAsync(out + o, d_out + o, n_ * sizeof(mdg_fit_result), cudaMemcpyDeviceToHost, ls));
            if (out_median) MDG_CUDA_TRY(cudaMemcpyAsync(out_median + o * R, d_med + o * R, n_ * R * 4, cudaMemcpyDeviceToHost, ls));
            if (out_hpdi_lo) MDG_CUDA_TRY(cudaMemcpyAsync(out_hpdi_lo + o * R, d_lo + o * R, n_ * R * 4, cudaMemcpyDeviceToHost, ls));
            if (out_hpdi_hi) MDG_CUDA_TRY(cudaMemcpyAsync(out_hpdi_hi + o * R, d_hi + o * R, n_ * R * 4, cudaMemcpyDeviceToHost, ls));
            const size_t so = o * MDG_NUM_RUNS * S * 4, to = o * MDG_NUM_RUNS * (size_t)(W + S) * 4, wo = o * MDG_NUM_RUNS * 2 * R;
            if (out_samples) MDG_CUDA_TRY(cudaMemcpyAsync(out_samples + so, d_samples + so, n_ * MDG_NUM_RUNS * S * 4 * 8, cudaMemcpyDeviceToHost, ls));
            if (out_trace) MDG_CUDA_TRY(cudaMemcpyAsync(out_trace + to, d_trace + to, n_ * MDG_NUM_RUNS * (size_t)(W + S) * 4 * 8, cudaMemcpyDeviceToHost, ls));
            if (out_waic) MDG_CUDA_TRY(cudaMemcpyAsync(out_waic + wo, d_waic_user + wo, n_ * MDG_NUM_RUNS * 2 * R * 8, cudaMemcpyDeviceToHost, ls));
        }
        MDG_CUDA_TRY(cudaMemcpyAsync(ln.h_leap, d_leap, MDG_NUM_RUNS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ls));
        MDG_CUDA_TRY(cudaEventRecord(ln.ev[4], ls));
        ln.launches = ctx->timings.n_launches - launches_before;
        ln.busy = true;
        ln.owner = slot;
    }
    return MDG_OK;
}

int mdg_fit_batch_wait(mdg_ctx* ctx, int64_t ticket, mdg_timings* out_timings) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    int slot = -1;
    for (int i = 0; i < kFitTickets; ++i) if (ctx->ticket[i].active && ctx->ticket[i].id == ticket) slot = i;
    if (slot < 0) { set_error("mdg_fit_batch_wait: unknown ticket %lld", (long long)ticket); return MDG_ERR_INVALID; }
    DeviceGuard guard(ctx->device);
    mdg_fit_ticket_slot& tk = ctx->ticket[slot];
    // harvest this ticket's chunks in submission order: the lane after `next_lane - 1` is the older one
    for (int i = 0; i < kFitLanes; ++i) {
        mdg_fit_lane& ln = ctx->lane[(ctx->next_lane + i) % kFitLanes];
        if (ln.busy && ln.owner == slot) {
            // later work on the ctx stream (e.g. the caller's consumers of device-resident results) follows the chunk
            MDG_CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ln.ev[4], 0));
            int rc = harvest_lane(ctx, ln);
            if (rc) return rc;
        }
    }
    tk.t.nuts_begin_ms = (float)tk.nuts_begin_ms;
    tk.t.nuts_end_ms = (float)tk.nuts_end_ms;
    tk.active = false;
    ctx->timings = tk.t;
    if (out_timings) *out_timings = tk.t;
    return MDG_OK;
}

int mdg_fit_batch(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position, const int64_t* tax_id, const uint32_t* k,
                  const uint32_t* N, const uint32_t* mism12, const double* noise3, const mdg_fit_config* cfg,
                  mdg_fit_result* out, float* out_median, float* out_hpdi_lo, float* out_hpdi_hi,
                  double* out_samples, double* out_trace, double* out_waic) {
    int64_t ticket = 0;
    int rc = mdg_fit_batch_submit(ctx, mem, n_tax, max_position, tax_id, k, N, mism12, noise3, cfg, out, out_median, out_hpdi_lo,
                                  out_hpdi_hi, out_samples, out_trace, out_waic, &ticket);
    if (rc) return rc;
    return mdg_fit_batch_wait(ctx, ticket, nullptr);
}

int mdg_map_batch(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position, const int64_t* tax_id, const uint32_t* k,
                  const uint32_t* N, const uint32_t* mism12, const double* noise3, const mdg_fit_config* cfg, mdg_map_result* out) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (!cfg || n_tax < 0 || max_position < 1 || max_position > MDG_MAX_POSITION || (mem != MDG_HOST && mem != MDG_DEVICE)) {
        set_error("mdg_map_batch: invalid argument");
        return MDG_ERR_INVALID;
    }
    if (n_tax > 0 && (!tax_id || !k || !N || !out)) { set_error("mdg_map_batch: NULL tax_id/k/N/out"); return MDG_ERR_INVALID; }
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    ctx->timings = mdg_timings{};
    const int P = max_position, R = 2 * P;
    const int n_runs = cfg->do_fwd_rev ? MDG_NUM_RUNS : 2;
    const bool host = (mem == MDG_HOST);
    const size_t nt = (size_t)n_tax;
    // TaxIDs per piece: bounds the per-run records (624 MB per 2^20 TaxIDs); results go straight to their rows
    const long long piece = 1ll << 20;
    const long long piece_max = std::min<long long>(n_tax, piece);
    int rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[0], st));
    const int64_t* d_tax = tax_id; const uint32_t* d_k = k; const uint32_t* d_N = N; const uint32_t* d_m12 = mism12;
    const double* d_noise = noise3;
    mdg_map_result* d_out = out;
    if (n_tax > 0 && host) {
        if ((rc = ctx->map_in_tax.ensure(nt * 8))) return rc;
        if ((rc = ctx->map_in_k.ensure(nt * R * 4))) return rc;
        if ((rc = ctx->map_in_N.ensure(nt * R * 4))) return rc;
        MDG_CUDA_TRY(cudaMemcpyAsync(ctx->map_in_tax.ptr, tax_id, nt * 8, cudaMemcpyHostToDevice, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(ctx->map_in_k.ptr, k, nt * R * 4, cudaMemcpyHostToDevice, st));
        MDG_CUDA_TRY(cudaMemcpyAsync(ctx->map_in_N.ptr, N, nt * R * 4, cudaMemcpyHostToDevice, st));
        d_tax = ctx->map_in_tax.as<int64_t>(); d_k = ctx->map_in_k.as<uint32_t>(); d_N = ctx->map_in_N.as<uint32_t>();
        if (mism12) {
            if ((rc = ctx->map_in_m12.ensure(nt * R * 12 * 4))) return rc;
            MDG_CUDA_TRY(cudaMemcpyAsync(ctx->map_in_m12.ptr, mism12, nt * R * 12 * 4, cudaMemcpyHostToDevice, st));
            d_m12 = ctx->map_in_m12.as<uint32_t>();
        }
        if (noise3) {
            if ((rc = ctx->map_in_noise.ensure(nt * 24))) return rc;
            MDG_CUDA_TRY(cudaMemcpyAsync(ctx->map_in_noise.ptr, noise3, nt * 24, cudaMemcpyHostToDevice, st));
            d_noise = ctx->map_in_noise.as<double>();
        }
        if ((rc = ctx->map_out.ensure(nt * sizeof(mdg_map_result)))) return rc;
        d_out = ctx->map_out.as<mdg_map_result>();
    }
    if ((rc = ctx->map_counters.ensure(256))) return rc;
    unsigned int* d_counter = ctx->map_counters.as<unsigned int>();                           // [1] work counter
    unsigned long long* d_evals = reinterpret_cast<unsigned long long*>(d_counter + 16);      // [6] gradient evaluations
    MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, st));
    if (n_tax > 0 && (rc = ctx->map_rec.ensure((size_t)piece_max * MDG_NUM_RUNS * sizeof(mdg_map_run)))) return rc;
    const Priors pr = make_priors(*cfg);
    const int npl = npl_for(R, 32);  // map_kernel's layout: the all-position fits are mdg_fit_batch's
    for (long long c0 = 0; c0 < n_tax; c0 += piece) {
        const int nc = (int)std::min<long long>(piece, n_tax - c0);
        if (c0 > 0) MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), st));
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
        MapBatchLaunch ml = {};
        ml.k = d_k + (size_t)c0 * R; ml.N = d_N + (size_t)c0 * R; ml.n_tax = nc; ml.P = P; ml.n_runs = n_runs;
        ml.pr = pr; ml.work_counter = d_counter; ml.rec = ctx->map_rec.as<mdg_map_run>();
        if ((rc = launch_map_batch(ctx, st, ml, npl))) return rc;
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
        MapAssembleLaunch al = {};
        al.tax_id = d_tax + c0; al.k = ml.k; al.N = ml.N;
        al.mism12 = d_m12 ? d_m12 + (size_t)c0 * R * 12 : nullptr;
        al.noise3 = d_noise ? d_noise + (size_t)c0 * 3 : nullptr;
        al.n_tax = nc; al.P = P; al.n_runs = n_runs; al.rec = ml.rec; al.out = d_out + c0; al.eval_totals = d_evals;
        map_assemble_kernel<<<(nc + 127) / 128, 128, 0, st>>>(al);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches++;
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
        MDG_CUDA_TRY(cudaEventSynchronize(ctx->ev[3]));  // the events are reused by the next piece
        ctx->timings.map_ms += elapsed(ctx->ev[1], ctx->ev[2]);
        ctx->timings.assemble_ms += elapsed(ctx->ev[2], ctx->ev[3]);
    }
    if (n_tax > 0 && host) MDG_CUDA_TRY(cudaMemcpyAsync(out, d_out, nt * sizeof(mdg_map_result), cudaMemcpyDeviceToHost, st));
    unsigned long long evals[MDG_NUM_RUNS];
    MDG_CUDA_TRY(cudaMemcpyAsync(evals, d_evals, sizeof evals, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->ev[4], st));
    MDG_CUDA_TRY(cudaEventSynchronize(ctx->ev[4]));
    for (int r = 0; r < MDG_NUM_RUNS; ++r) ctx->timings.leapfrogs[r] = evals[r];
    ctx->timings.total_ms = elapsed(ctx->ev[0], ctx->ev[4]);
    return MDG_OK;
}

// ---------------------------------------------------------------------------------------------
// test / measurement entry points
// ---------------------------------------------------------------------------------------------
}  // extern "C"

namespace {

__global__ void test_lgam_kernel(long long n, const double* x, double* lg, double* dg) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    log_table_init();
    if (i < n) {
        double a, b;
        lgam_digam(x[i], a, b);
        lg[i] = a;
        dg[i] = b;
    }
}

__global__ void test_exp_log_kernel(long long n, const double* x, double* ex, double* lg) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    log_table_init();
    if (i < n) {
        ex[i] = exp_fast(x[i]);
        lg[i] = x[i] > 0.0 ? log_pos(x[i]) : nan("");
    }
}

__global__ void test_philox_kernel(long long n, const uint32_t* key2, const uint32_t* ctr4, uint32_t* out4) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) {
        uint4 o = philox4x32(make_uint2(key2[2 * i], key2[2 * i + 1]), ctr4[4 * i], ctr4[4 * i + 1], ctr4[4 * i + 2], ctr4[4 * i + 3]);
        out4[4 * i] = o.x; out4[4 * i + 1] = o.y; out4[4 * i + 2] = o.z; out4[4 * i + 3] = o.w;
    }
}

template <int MODEL, int NPL>
__global__ void test_logp_kernel(int P, const uint32_t* k, const uint32_t* N, Priors pr, int mask, int jac,
                                 long long n_eval, const double* u, double* out_logp, double* out_grad, double* out_ll) {
    constexpr int D = ModelDim<MODEL>::value;
    const int lane = threadIdx.x & 31;
    const long long e = blockIdx.x;
    __shared__ double2 s_prior[64];
    log_table_init();
    prior_table_init<MODEL>(s_prior, pr, jac);
    if (e >= n_eval) return;
    LaneObs<NPL> ob;
    load_obs<NPL, 32>(ob, k, N, P, mask, lane);
    double logC[NPL];
    log_binom_coeff<NPL>(ob, logC);
    double uu[D];
#pragma unroll
    for (int j = 0; j < D; ++j) uu[j] = u[e * 4 + j];
    double logp, grad[D], ll[NPL];
    bool valid;
    eval_model<MODEL, NPL, 32>(ob, uu, s_prior, pr.phi_min, (mask == 0 ? 2 * P : P) < NPL * 32, 0xffffffffu, lane, logp, grad, ll, valid);
    double sumC = 0.0;
#pragma unroll
    for (int s = 0; s < NPL; ++s) sumC += logC[s];
    sumC = group_sum<32>(sumC, 0xffffffffu);
    if (lane == 0) {
        out_logp[e] = valid ? logp + sumC : nan("");
        for (int j = 0; j < 4; ++j) out_grad[e * 4 + j] = j < D ? grad[j] : 0.0;
    }
    if (out_ll) {
#pragma unroll
        for (int s = 0; s < NPL; ++s)
            if (ob.act[s]) out_ll[e * 2 * P + (mask == 2 ? P : 0) + s * 32 + lane] = ll[s] + logC[s];
    }
}

__global__ void fp64_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678) out[0] = a0;
}

}  // namespace

extern "C" {

int mdg_test_lgamma_digamma(mdg_ctx* ctx, int64_t n, const double* x, double* out_lgamma, double* out_digamma) {
    if (!ctx || n < 0) { set_error("invalid argument"); return MDG_ERR_INVALID; }
    if (n == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    int rc = ctx->buf[20].ensure((size_t)n * 24);
    if (rc) return rc;
    double* d = ctx->buf[20].as<double>();
    MDG_CUDA_TRY(cudaMemcpyAsync(d, x, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    test_lgam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, d, d + n, d + 2 * n);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out_lgamma, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaMemcpyAsync(out_digamma, d + 2 * n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return MDG_OK;
}

int mdg_test_exp_log(mdg_ctx* ctx, int64_t n, const double* x, double* out_exp, double* out_log) {
    if (!ctx || n < 0) { set_error("invalid argument"); return MDG_ERR_INVALID; }
    if (n == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    int rc = ctx->buf[20].ensure((size_t)n * 24);
    if (rc) return rc;
    double* d = ctx->buf[20].as<double>();
    MDG_CUDA_TRY(cudaMemcpyAsync(d, x, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    test_exp_log_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, d, d + n, d + 2 * n);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out_exp, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaMemcpyAsync(out_log, d + 2 * n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return MDG_OK;
}

int mdg_test_philox(mdg_ctx* ctx, int64_t n, const uint32_t* key2, const uint32_t* ctr4, uint32_t* out4) {
    if (!ctx || n < 0) { set_error("invalid argument"); return MDG_ERR_INVALID; }
    if (n == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    int rc = ctx->buf[20].ensure((size_t)n * 40);
    if (rc) return rc;
    uint32_t* d = ctx->buf[20].as<uint32_t>();
    MDG_CUDA_TRY(cudaMemcpyAsync(d, key2, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    MDG_CUDA_TRY(cudaMemcpyAsync(d + 2 * n, ctr4, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    test_philox_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, d, d + 2 * n, d + 6 * n);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out4, d + 6 * n, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return MDG_OK;
}

int mdg_test_logp_grad(mdg_ctx* ctx, int max_position, const uint32_t* k, const uint32_t* N, const mdg_fit_config* cfg,
                       int model, int lane_mask, int with_jacobian, int64_t n_eval, const double* u, double* out_logp,
                       double* out_grad, double* out_ll) {
    if (!ctx || !cfg || max_position < 1 || max_position > MDG_MAX_POSITION || n_eval < 0 || model < 0 || model > 1 ||
        lane_mask < 0 || lane_mask > 2) {
        set_error("invalid argument");
        return MDG_ERR_INVALID;
    }
    if (n_eval == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    const int P = max_position, R = 2 * P;
    const size_t ne = (size_t)n_eval;
    int rc = ctx->buf[20].ensure((size_t)R * 8 + ne * (32 + 8 + 32 + (size_t)R * 8) + 1024);
    if (rc) return rc;
    unsigned char* base = ctx->buf[20].as<unsigned char>();
    uint32_t* dk = (uint32_t*)base;
    uint32_t* dN = dk + R;
    double* du = (double*)(base + (((size_t)R * 8 + 255) & ~(size_t)255));
    double* dlogp = du + ne * 4;
    double* dgrad = dlogp + ne;
    double* dll = dgrad + ne * 4;
    cudaStream_t st = ctx->stream;
    MDG_CUDA_TRY(cudaMemcpyAsync(dk, k, (size_t)R * 4, cudaMemcpyHostToDevice, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(dN, N, (size_t)R * 4, cudaMemcpyHostToDevice, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(du, u, ne * 32, cudaMemcpyHostToDevice, st));
    MDG_CUDA_TRY(cudaMemsetAsync(dll, 0, ne * R * 8, st));
    const Priors pr = make_priors(*cfg);
    const int n_obs = lane_mask == 0 ? R : P;
    const int npl = npl_for(n_obs, 32);
    const unsigned grid = (unsigned)n_eval;
#define MDG_LAUNCH_LOGP(M, NPL_) test_logp_kernel<M, NPL_><<<grid, 32, 0, st>>>(P, dk, dN, pr, lane_mask, with_jacobian, n_eval, du, dlogp, dgrad, out_ll ? dll : nullptr)
    if (model == 0) { if (npl == 1) MDG_LAUNCH_LOGP(0, 1); else if (npl == 2) MDG_LAUNCH_LOGP(0, 2); else MDG_LAUNCH_LOGP(0, 4); }
    else { if (npl == 1) MDG_LAUNCH_LOGP(1, 1); else if (npl == 2) MDG_LAUNCH_LOGP(1, 2); else MDG_LAUNCH_LOGP(1, 4); }
#undef MDG_LAUNCH_LOGP
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out_logp, dlogp, ne * 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(out_grad, dgrad, ne * 32, cudaMemcpyDeviceToHost, st));
    if (out_ll) MDG_CUDA_TRY(cudaMemcpyAsync(out_ll, dll, ne * R * 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    return MDG_OK;
}

int mdg_measure_fp64_peak(mdg_ctx* ctx, double* out_tflops) {
    if (!ctx || !out_tflops) { set_error("invalid argument"); return MDG_ERR_INVALID; }
    DeviceGuard guard(ctx->device);
    int rc = ctx->buf[20].ensure(64);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    const int iters = 20000, threads = 512, blocks = ctx->num_sms * 4;
    fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->buf[20].as<double>(), 1000);  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[10], st));
        fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->buf[20].as<double>(), iters);
        MDG_CUDA_TRY(cudaEventRecord(ctx->ev[11], st));
        MDG_CUDA_TRY(cudaStreamSynchronize(st));
        MDG_CUDA_TRY(cudaGetLastError());
        const double ms = elapsed(ctx->ev[10], ctx->ev[11]);
        const double flops = 2.0 * 8.0 * iters * (double)threads * blocks;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *out_tflops = best;
    return MDG_OK;
}

}  // extern "C"
