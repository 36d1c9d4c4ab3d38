// mdg_api.cu — the C-ABI of libmdgb200.so (include/mdg.h): context management, host<->device
// staging, kernel launches and CUDA-event timing for the counts (K1) and fit (K3-K7) paths.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>
#include <algorithm>

#include "mdg_counts_kernel.cuh"
#include "mdg_counts_stream.cuh"
#include "mdg_tsv_kernel.cuh"
#include "mdg_select_kernel.cuh"
#include "mdg_post_kernels.cuh"
#include "mdg_map_batch_kernel.cuh"
#include "mdg_map_profile_kernel.cuh"
#include "mdg_nuts_kernel.cuh"

namespace mdg {

static thread_local char g_error[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
}

// grow-only device buffer, freed by its destructor
struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (ptr) cudaFree(ptr);
    }
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
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

// owner of a stream, an event or a pinned host allocation, released by its destructor
template <typename H, auto Release>
struct Owned {
    H h = nullptr;
    Owned() = default;
    Owned(const Owned&) = delete;
    Owned& operator=(const Owned&) = delete;
    ~Owned() {
        if (h) Release(h);
    }
    operator H() const { return h; }
};
using CudaStream = Owned<cudaStream_t, cudaStreamDestroy>;
using CudaEvent = Owned<cudaEvent_t, cudaEventDestroy>;

}  // namespace mdg

// One fit lane = the streams, events and scratch of one chunk in flight. Two lanes per ctx: chunk c+1 (of the
// same batch or of the next submitted batch) starts under the tail of chunk c, which is a handful of long
// sequential chains on an otherwise idle GPU.
struct mdg_fit_lane {
    mdg::CudaStream main, side[2];  // main: high priority; side[m]: the NUTS launch of model m (0 PMD, 1 null)
    mdg::CudaEvent begin, map_end, nuts_end, pred_end, done;  // done: after assembly and the copies back
    mdg::CudaEvent nuts_fork, nuts_join[2];  // nuts_join[m]: end of side[m]'s NUTS launch
    mdg::DevBuf rec, map, pred, counters, samples, waic, waic_acc[2];
    mdg::DevBuf chain_clock;  // development switch MDG_CHAIN_CLOCK=<file>
    mdg::DevBuf order;        // queue order of the chunk's TaxIDs: [chunk] int order, [chunk] bucket bytes, 3 x kOrderBuckets counters
    int clock_items = 0;
    mdg::Owned<unsigned long long*, cudaFreeHost> h_leap;  // pinned [MDG_NUM_RUNS]
    bool busy = false;
    int owner = -1;          // ticket slot of the chunk in flight
    uint32_t launches = 0;
};

// One submitted batch (mdg_fit_batch_submit): its staged inputs / outputs and the accumulated timings.
struct mdg_fit_ticket_slot {
    bool active = false;
    int64_t id = 0;
    mdg::CudaEvent ev_begin;
    mdg::DevBuf arena;
    mdg_timings t = {};
    double nuts_begin_ms = 0, nuts_end_ms = 0;
    bool have_nuts = false;
};

constexpr int kFitLanes = MDG_MAX_INFLIGHT;
constexpr int kFitTickets = MDG_MAX_INFLIGHT;

struct mdg_ctx {
    int device = 0;
    int num_sms = 0;
    mdg::CudaStream own_stream;
    cudaStream_t stream = nullptr;  // own_stream, or the caller's (mdg_ctx_set_stream)
    // timing of the synchronous entry points
    mdg::CudaEvent call_begin, work_begin, work_end, call_end;
    mdg::CudaEvent epoch;  // time zero of mdg_timings.nuts_begin_ms / nuts_end_ms
    mdg::CudaEvent inputs_ready;
    // staged buffers and scratch of the synchronous entry points (they never overlap: each synchronises before
    // it returns)
    mdg::DevBuf arena;
    mdg::DevBuf test_scratch;  // mdg_test_*, mdg_measure_fp64_peak
    mdg::DevBuf da_tables;     // sqrt(t) and t^-0.75 for t < kDaTable (dual averaging), filled at the first fit
    mdg_fit_lane lane[kFitLanes];
    mdg_fit_ticket_slot ticket[kFitTickets];
    int next_lane = 0;
    int64_t next_ticket_id = 1;
    double nuts_covered_until_ms = 0;  // union of NUTS intervals harvested so far ends here
    mdg_timings timings = {};
    mdg::DevBuf map_rec, map_counters;  // mdg_map_batch: per-run records, counters; apart from the fit lanes' scratch
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

// The device side of one call's buffers. Callers register requests, each naming the launch-struct field that
// receives the device pointer: inputs (copied in), outputs (copied back by rows) and scratch. commit() lays them
// out in one grow-only arena, each 256-byte aligned (the 128-bit load / store paths of mdg_counts_reduce depend
// on it), and enqueues the host-to-device copies. Under MDG_DEVICE inputs and outputs are the caller's pointers
// and only scratch takes arena space; a NULL input or output stays NULL.
class Stage {
public:
    Stage(DevBuf& arena, bool host, cudaStream_t st) : arena_(arena), host_(host), st_(st) {}
    template <typename T> void in(T*& field, const void* src, size_t bytes) { add(&field, kIn, const_cast<void*>(src), bytes, 0); }
    // `rows` rows of `row_bytes` each; copy_back() copies a range of them
    template <typename T> void out(T*& field, void* dst, size_t row_bytes, size_t rows) { add(&field, kOut, dst, row_bytes * rows, row_bytes); }
    // copied back in full by every copy_back()
    template <typename T> void out_all(T*& field, void* dst, size_t bytes) { add(&field, kOut, dst, bytes, 0); }
    template <typename T> void scratch(T*& field, size_t bytes) { add(&field, kScratch, nullptr, bytes, 0); }

    int commit() {
        size_t total = 0;
        for (const Req& r : reqs_) total += staged(r) ? align(r.bytes) : 0;
        if (int rc = arena_.ensure(total)) return rc;
        unsigned char* p = arena_.as<unsigned char>();
        for (const Req& r : reqs_) {
            void* d = staged(r) ? p : r.user;
            std::memcpy(r.field, &d, sizeof d);
            if (!staged(r)) continue;
            p += align(r.bytes);
            if (r.kind == kIn && r.bytes) MDG_CUDA_TRY(cudaMemcpyAsync(d, r.user, r.bytes, cudaMemcpyHostToDevice, st_));
        }
        return MDG_OK;
    }

    int copy_back(size_t row0, size_t rows, cudaStream_t st) const {
        for (const Req& r : reqs_) {
            if (r.kind != kOut || !staged(r)) continue;
            unsigned char* d;
            std::memcpy(&d, r.field, sizeof d);
            const size_t off = row0 * r.row_bytes, bytes = r.row_bytes ? rows * r.row_bytes : r.bytes;
            if (bytes) MDG_CUDA_TRY(cudaMemcpyAsync((unsigned char*)r.user + off, d + off, bytes, cudaMemcpyDeviceToHost, st));
        }
        return MDG_OK;
    }

private:
    enum Kind { kIn, kOut, kScratch };
    struct Req {
        void* field;  // a T* launch-struct member (or local)
        Kind kind;
        void* user;   // the caller's source / destination
        size_t bytes, row_bytes;
    };
    static size_t align(size_t b) { return (b + 255) & ~(size_t)255; }
    bool staged(const Req& r) const { return r.kind == kScratch || (host_ && r.user); }
    template <typename T> void add(T** field, Kind kind, void* user, size_t bytes, size_t row_bytes) {
        reqs_.push_back({(void*)field, kind, user, bytes, row_bytes});
    }
    DevBuf& arena_;
    const bool host_;
    const cudaStream_t st_;
    std::vector<Req> reqs_;
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
    long long want = (items + items_per_block - 1) / items_per_block;
    long long cap = (long long)per_sm * num_sms;
    return (int)std::max<long long>(1, std::min(want, cap));
}

constexpr int kNutsGroupLanes = 8;  // lanes per chain
constexpr int kNutsWarps = 4;
constexpr int kOrderMinChunk = 32768;  // TaxIDs per chunk from which the NUTS queue is ordered by coverage
constexpr int kMapWarps = 4;
constexpr int kPpcWarps = 4;

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

// K4, group layout: GW lanes per chain, rolled position loop (mdg_nuts_kernel.cuh)
template <int MODEL>
int launch_nuts_group(mdg_ctx* ctx, cudaStream_t st, FitLaunch fl, DevBuf& acc) {
    constexpr int GW = kNutsGroupLanes, WARPS = kNutsWarps;
    auto kern = nuts_group_kernel<MODEL, GW, WARPS>;
    const int n_obs = fl.n_items_all > 0 ? 2 * fl.P : fl.P;  // the launch's longest run
    fl.n_slots = (n_obs + 1 + GW - 1) / GW;  // index 0 is the spare
    size_t smem = (size_t)WARPS * nuts_warp_smem_bytes(fl.n_slots);
    // The NUTS launches of a chunk take over each other's CTA slots as CTAs retire. Shared memory is allocated
    // contiguously, so a retiring CTA's hole must fit the next launch's CTA: every launch asks for the same footprint
    // (static + dynamic), the largest one (PMD with all-position runs). Otherwise the SMs end up with three resident
    // CTAs instead of four (profiles/r02_chain_timeline.md: 8 016 live chains instead of 9 472).
    {
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
    const int grid = persistent_grid(kern, WARPS * 32, smem, ctx->num_sms, fl.n_items, WARPS * (32 / GW));
    int rc = acc.ensure((size_t)grid * WARPS * 4 * fl.n_slots * 32 * sizeof(double));
    if (rc) return rc;
    fl.waic_acc = acc.as<double>();
    kern<<<grid, WARPS * 32, smem, st>>>(fl);
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

int npl_for(int n_obs, int gw) {
    int npl = (n_obs + gw - 1) / gw;
    return npl <= 1 ? 1 : (npl <= 2 ? 2 : 4);
}

// f(std::integral_constant<int, NPL>{}) for the observations per lane of a warp over n_obs positions
template <typename F>
void with_npl(int n_obs, F&& f) {
    const int npl = npl_for(n_obs, 32);
    if (npl == 1) f(std::integral_constant<int, 1>{});
    else if (npl == 2) f(std::integral_constant<int, 2>{});
    else f(std::integral_constant<int, 4>{});
}

// map_kernel / map_batch_kernel fit all 2P positions of a TaxID
int launch_map(mdg_ctx* ctx, cudaStream_t st, const MapLaunch& ml) {
    const long long items = 2ll * ml.n_tax;
    with_npl(2 * ml.P, [&](auto npl) {
        auto kern = map_kernel<decltype(npl)::value, kMapWarps>;
        int grid = persistent_grid(kern, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        kern<<<grid, kMapWarps * 32, 0, st>>>(ml);
    });
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

int launch_map_batch(mdg_ctx* ctx, cudaStream_t st, const MapBatchLaunch& ml) {
    const long long items = (long long)ml.n_runs * ml.n_tax;
    with_npl(2 * ml.P, [&](auto npl) {
        auto kern = map_batch_kernel<decltype(npl)::value, kMapWarps>;
        int grid = persistent_grid(kern, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        kern<<<grid, kMapWarps * 32, 0, st>>>(ml);
    });
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

int launch_map_profile(mdg_ctx* ctx, cudaStream_t st, const MapProfileLaunch& ml) {
    const long long items = 2ll * ml.n_prof * ml.n_tax;
    with_npl(2 * ml.P, [&](auto npl) {
        auto kern = map_profile_kernel<decltype(npl)::value, kMapWarps>;
        int grid = persistent_grid(kern, kMapWarps * 32, 0, ctx->num_sms, items, kMapWarps);
        kern<<<grid, kMapWarps * 32, 0, st>>>(ml);
    });
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches++;
    return MDG_OK;
}

float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

}  // namespace

extern "C" {

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
    std::unique_ptr<mdg_ctx> ctx(new mdg_ctx());  // a failure below releases what was created so far
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    auto fail = [&](cudaError_t e, const char* what) {
        set_error("mdg_ctx_create: %s failed: %s", what, cudaGetErrorString(e));
        return MDG_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream.h, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
    ctx->stream = ctx->own_stream;
    for (CudaEvent* ev : {&ctx->call_begin, &ctx->work_begin, &ctx->work_end, &ctx->call_end, &ctx->epoch})
        if ((e = cudaEventCreate(&ev->h)) != cudaSuccess) return fail(e, "cudaEventCreate");
    if ((e = cudaEventCreateWithFlags(&ctx->inputs_ready.h, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
    // The NUTS launches are persistent and fill every CTA slot of the GPU; the short kernels around them (MAP,
    // posterior predictive, assembly) of the OTHER batch in flight must not queue behind the NUTS CTAs that are
    // still waiting for a slot, or a batch could not complete (and the next one not be submitted) before the
    // following batch's NUTS launches are through: the lane's main stream gets the highest priority, the NUTS
    // streams the lowest.
    int prio_low = 0, prio_high = 0;
    if ((e = cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high)) != cudaSuccess) return fail(e, "cudaDeviceGetStreamPriorityRange");
    for (auto& ln : ctx->lane) {
        if ((e = cudaStreamCreateWithPriority(&ln.main.h, cudaStreamNonBlocking, prio_high)) != cudaSuccess) return fail(e, "cudaStreamCreate");
        for (auto& sd : ln.side)
            if ((e = cudaStreamCreateWithPriority(&sd.h, cudaStreamNonBlocking, prio_low)) != cudaSuccess) return fail(e, "cudaStreamCreate");
        for (CudaEvent* ev : {&ln.begin, &ln.map_end, &ln.nuts_end, &ln.pred_end, &ln.done})
            if ((e = cudaEventCreate(&ev->h)) != cudaSuccess) return fail(e, "cudaEventCreate");
        for (CudaEvent* ev : {&ln.nuts_fork, &ln.nuts_join[0], &ln.nuts_join[1]})
            if ((e = cudaEventCreateWithFlags(&ev->h, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
        if ((e = cudaHostAlloc((void**)&ln.h_leap.h, MDG_NUM_RUNS * sizeof(unsigned long long), cudaHostAllocDefault)) != cudaSuccess)
            return fail(e, "cudaHostAlloc");
    }
    for (auto& tk : ctx->ticket)
        if ((e = cudaEventCreate(&tk.ev_begin.h)) != cudaSuccess) return fail(e, "cudaEventCreate");
    if ((e = cudaEventRecord(ctx->epoch, ctx->own_stream)) != cudaSuccess) return fail(e, "cudaEventRecord");
    if ((e = cudaEventSynchronize(ctx->epoch)) != cudaSuccess) return fail(e, "cudaEventSynchronize");
    *out = ctx.release();
    return MDG_OK;
}

void mdg_ctx_destroy(mdg_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    for (auto& ln : ctx->lane) {
        cudaStreamSynchronize(ln.main);
        for (cudaStream_t sd : ln.side) cudaStreamSynchronize(sd);
    }
    cudaStreamSynchronize(ctx->stream);
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
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));

    // ---- the caller's buffers (MDG_DEVICE) or staged ones (MDG_HOST), and scratch ----
    const bool host = (mem == MDG_HOST);
    const size_t ncap = (size_t)out_capacity;
    CountsLaunch cl = {};
    Stage stage(ctx->arena, host, st);
    stage.in(cl.tax_id, tax_id, n * 8);
    stage.in(cl.n_align, n_alignments, n * 4);
    stage.in(cl.is_rev, is_reverse, n);
    stage.in(cl.pos0, pos0, n);
    // staged counts16 columns start 256 bytes apart, a multiple of 4 rows
    cl.counts16 = counts16;
    cl.stride = host ? (long long)(((n * 4 + 255) & ~(size_t)255) / 4) : counts_stride;
    if (host) stage.scratch(cl.counts16, 16 * (size_t)cl.stride * 4);
    stage.out_all(cl.n_fwd_row, n_fwd_ref_row, n * 4);
    stage.out_all(cl.n_rev_row, n_rev_ref_row, n * 4);
    stage.out_all(cl.f_fwd_row, f_fwd_row, n * 4);
    stage.out_all(cl.f_rev_row, f_rev_row, n * 4);
    stage.out_all(cl.z_row, z_row, n);
    stage.out_all(cl.y_row, y_sum_total_row, n * 8);
    stage.out_all(cl.keep_row, keep_row, n);
    stage.out(cl.out_tax, out_tax_id, 8, ncap);
    stage.out(cl.out_nal, out_n_alignments, 4, ncap);
    // the noise kernel needs the first rows in final order even if the caller does not want them
    if (out_first_row || !out_noise) stage.out(cl.out_first, out_first_row, 8, ncap);
    else stage.scratch(cl.out_first, ncap * 8);
    stage.out(cl.out_k, out_k, 4 * (size_t)R, ncap);
    stage.out(cl.out_N, out_N, 4 * (size_t)R, ncap);
    stage.out(cl.out_noise, out_noise, 24, ncap);
    long long* d_ntax;  // [0] kept TaxIDs, [1] error flag (int), [2] dense rows reserved
    stage.scratch(d_ntax, 64);
    // ---- warp-synchronous streaming kernel (mdg_counts_stream.cuh): one warp per 128 rows ----
    const long long n_tiles = (n_rows + kStreamRows - 1) / kStreamRows;
    const long long n_chunks = (n_tiles + kScanChunk - 1) / kScanChunk;
    CountsPermute cp = {};
    long long *d_tile_base, *d_final_base, *d_chunk;
    int* d_tile_cnt;
    stage.scratch(d_tile_base, (size_t)n_tiles * 8);
    stage.scratch(d_final_base, (size_t)n_tiles * 8);
    stage.scratch(d_chunk, (size_t)n_chunks * 8);
    stage.scratch(d_tile_cnt, (size_t)n_tiles * 4);
    // the stream kernel writes the per-TaxID rows into temporaries, the permute moves them
    if (out_tax_id) stage.scratch(cp.t_tax, ncap * 8);
    if (out_n_alignments) stage.scratch(cp.t_nal, ncap * 4);
    if (out_first_row || out_noise) stage.scratch(cp.t_first, ncap * 8);
    if (out_k) stage.scratch(cp.t_k, ncap * R * 4);
    if (out_N) stage.scratch(cp.t_N, ncap * R * 4);
    if (int rc = stage.commit()) return rc;
    if (host)
        for (int c = 0; c < 16; ++c)
            cudaMemcpyAsync((uint32_t*)cl.counts16 + (size_t)c * cl.stride, counts16 + (size_t)c * counts_stride, n * 4, cudaMemcpyHostToDevice, st);
    MDG_CUDA_TRY(cudaGetLastError());
    cl.n_rows = n_rows;
    cl.fwd_ref = fwd_ref; cl.fwd_obs = fwd_obs; cl.rev_ref = rev_ref; cl.rev_obs = rev_obs;
    cl.P = P; cl.min_align = min_alignments; cl.min_y = min_y_sum;
    auto aligned16 = [](const void* p) { return ((uintptr_t)p & 15u) == 0; };
    cl.vec_in = aligned16(cl.tax_id) && aligned16(cl.n_align) && aligned16(cl.is_rev) && aligned16(cl.pos0) &&
                aligned16(cl.counts16) && (cl.stride % 4 == 0);

    // output bases 16-byte aligned -> 128-bit stores
    cl.vec_out = aligned16(cl.n_fwd_row) && aligned16(cl.n_rev_row) && aligned16(cl.f_fwd_row) && aligned16(cl.f_rev_row) &&
                 aligned16(cl.z_row) && aligned16(cl.y_row) && aligned16(cl.keep_row);
    int* d_err = reinterpret_cast<int*>(d_ntax + 1);
    int h_err = 0;
    long long h_ntax = 0;
    cp.n_tiles = n_tiles; cp.tile_base = d_tile_base; cp.final_base = d_final_base; cp.tile_cnt = d_tile_cnt; cp.R = R;
    cp.chunk_off = d_chunk;
    cp.out_tax = cl.out_tax; cp.out_nal = cl.out_nal; cp.out_first = cl.out_first; cp.out_k = cl.out_k; cp.out_N = cl.out_N;
    CountsLaunch kl = cl;
    kl.out_noise = nullptr;
    kl.out_tax = (long long*)cp.t_tax;
    kl.out_nal = (uint32_t*)cp.t_nal;
    kl.out_first = (long long*)cp.t_first;
    kl.out_k = (uint32_t*)cp.t_k;
    kl.out_N = (uint32_t*)cp.t_N;
    kl.kept_counter = reinterpret_cast<unsigned long long*>(d_ntax + 2);
    kl.tile_base = d_tile_base;
    kl.tile_cnt = d_tile_cnt;
    kl.capacity = out_capacity;
    kl.error_flag = d_err;
    MDG_CUDA_TRY(cudaMemsetAsync(d_ntax, 0, 64, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
    counts_stream_kernel<<<(unsigned)((n_tiles + kStreamWarps - 1) / kStreamWarps), kStreamWarps * 32, 0, st>>>(kl);
    MDG_CUDA_TRY(cudaGetLastError());
    counts_scan_local_kernel<<<(unsigned)n_chunks, kScanChunk, 0, st>>>(d_tile_cnt, n_tiles, d_final_base, d_chunk);
    counts_scan_chunks_kernel<<<1, 32, 0, st>>>(d_chunk, n_chunks, d_ntax);
    MDG_CUDA_TRY(cudaGetLastError());
    counts_permute_kernel<<<(unsigned)((n_tiles + kPermuteWarps * kPermuteTiles - 1) / (kPermuteWarps * kPermuteTiles)), kPermuteWarps * 32, 0, st>>>(cp);
    MDG_CUDA_TRY(cudaGetLastError());
    ctx->timings.n_launches += 4;
    if (cl.out_noise) {
        NoiseLaunch nl = {};
        nl.n_rows = n_rows; nl.tax_id = cl.tax_id; nl.is_rev = cl.is_rev; nl.pos0 = cl.pos0; nl.counts16 = cl.counts16;
        nl.stride = cl.stride; nl.P = P; nl.n_tax = d_ntax; nl.first_row = cl.out_first; nl.out_noise = cl.out_noise;
        nl.capacity = out_capacity;
        counts_noise_kernel<<<(unsigned)std::max<long long>(1, std::min<long long>((out_capacity + 3) / 4, 16LL * ctx->num_sms)), 128, 0, st>>>(nl);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches += 1;
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_err, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_ntax, d_ntax, sizeof(long long), cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
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
    if (int rc = stage.copy_back(0, (size_t)h_ntax, st)) return rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->work_begin, ctx->work_end);
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->call_end);
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
    const size_t nr = (size_t)n_rows, nt = (size_t)n_tax;
    OrderLaunch ol = {};
    ol.n_rows = n_rows; ol.n_tax = n_tax;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));
    Stage stage(ctx->arena, mem == MDG_HOST, st);
    stage.in(ol.tax_id_row, tax_id_row, nr * 8);
    stage.in(ol.z_row, z_row, nr);
    stage.in(ol.keep_row, keep_row, nr);
    stage.in(ol.first_row, first_row, nt * 8);
    stage.in(ol.tax_order, tax_order, nt * 8);
    stage.out(ol.perm, out_perm, 8, (size_t)perm_capacity);
    long long *d_start, *d_total;  // d_total: [0] kept rows, [1] error flag (int)
    stage.scratch(ol.len_sorted, nt * 4);
    stage.scratch(d_start, nt * 8);
    stage.scratch(d_total, 16);
    if (int rc = stage.commit()) return rc;
    ol.out_start = d_start;
    ol.error_flag = reinterpret_cast<int*>(d_total + 1);
    MDG_CUDA_TRY(cudaMemsetAsync(d_total, 0, 16, st));
    const unsigned grid = (unsigned)((n_tax + kOrderWarps - 1) / kOrderWarps);
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
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
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
    ctx->timings.n_launches = 3;
    if (int rc = stage.copy_back(0, (size_t)h_total, st)) return rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->work_begin, ctx->work_end);
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->call_end);
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
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));
    const bool host = (mem == MDG_HOST);
    const size_t cap = (size_t)capacity;
    TsvLaunch tl = {};
    tl.n_bytes = n_bytes; tl.first = first; tl.n_cols = n_cols; tl.capacity = capacity;
    tl.n_blocks = (n_bytes - first + kTsvBlockBytes - 1) / kTsvBlockBytes;
    Stage stage(ctx->arena, host, st);
    stage.scratch(tl.text, (size_t)n_bytes);  // copied below: `text` is a host pointer whatever `mem` says
    stage.scratch(tl.block_base, (size_t)tl.n_blocks * 8);
    stage.scratch(tl.line_start, (cap + 2) * 8);
    stage.scratch(tl.block_cnt, (size_t)tl.n_blocks * 4);
    long long* d_scal;  // [0] newline total, [1] error flag (int), [2] error line
    stage.scratch(d_scal, 64);
    stage.out(tl.tax_id, tax_id, 8, cap);
    stage.out(tl.n_align, n_alignments, 4, cap);
    stage.out(tl.is_rev, is_reverse, 1, cap);
    stage.out(tl.pos0, pos0, 1, cap);
    stage.out(tl.name_span, name_span, 16, cap);
    stage.out(tl.rank_span, rank_span, 16, cap);
    // staged counts16 columns start (cap rounded up to 64 rows) * 4 bytes apart
    tl.counts16 = counts16;
    tl.stride = host ? (long long)((cap + 63) & ~(size_t)63) : counts_stride;
    if (host) stage.scratch(tl.counts16, 16 * (size_t)tl.stride * 4);
    if (int rc = stage.commit()) return rc;
    MDG_CUDA_TRY(cudaMemcpyAsync((char*)tl.text, text, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    tl.n_lines = d_scal; tl.error_flag = reinterpret_cast<int*>(d_scal + 1); tl.error_line = d_scal + 2;
    MDG_CUDA_TRY(cudaMemsetAsync(d_scal, 0, 64, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
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
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
    ctx->timings.n_launches = 4;
    int h_err[2] = {0, 0};
    long long h_line = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(h_err, tl.error_flag, 4, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_line, tl.error_line, 8, cudaMemcpyDeviceToHost, st));
    if (int rc = stage.copy_back(0, (size_t)n_lines, st)) return rc;
    if (host && n_lines > 0) {
        for (int c = 0; c < 16; ++c)
            MDG_CUDA_TRY(cudaMemcpyAsync(counts16 + (size_t)c * counts_stride, tl.counts16 + (size_t)c * tl.stride,
                                         (size_t)n_lines * 4, cudaMemcpyDeviceToHost, st));
    }
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.counts_ms = elapsed(ctx->work_begin, ctx->work_end);
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->call_end);
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
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    ctx->timings = mdg_timings{};
    const long long take = std::min<long long>(n_top, n_tax);
    *out_n = take;
    if (n_tax == 0 || (take == 0 && !out_weight)) { *out_n = 0; return MDG_OK; }
    const size_t nr = (size_t)n_rows, nt = (size_t)n_tax;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));
    const int n_blocks = (int)((n_tax + kTopThreads - 1) / kTopThreads);
    TopLaunch tl = {};
    tl.n_tax = n_tax; tl.n_top = take;
    const long long *d_tax_row, *d_first;
    const uint32_t* d_nal_row;
    const uint8_t* d_keep;
    unsigned long long* d_weight;
    long long* d_total;
    Stage stage(ctx->arena, mem == MDG_HOST, st);
    stage.in(d_tax_row, tax_id_row, nr * 8);
    stage.in(d_nal_row, n_alignments_row, nr * 4);
    stage.in(d_keep, keep_row, nr);
    stage.in(tl.tax_id, tax_id, nt * 8);
    stage.in(d_first, first_row, nt * 8);
    stage.out(tl.out_index, out_index, 8, (size_t)take);
    if (out_weight) stage.out_all(d_weight, out_weight, nt * 8);
    else stage.scratch(d_weight, nt * 8);
    stage.scratch(tl.hist, kTopPasses * 256 * 4);
    stage.scratch(tl.block_cnt, (size_t)n_blocks * 4);
    stage.scratch(tl.block_base, (size_t)n_blocks * 8);
    stage.scratch(d_total, 8);
    if (int rc = stage.commit()) return rc;
    tl.weight = d_weight;
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
    MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
    if (int rc = stage.copy_back(0, (size_t)take, st)) return rc;
    long long h_total = 0;
    MDG_CUDA_TRY(cudaMemcpyAsync(&h_total, d_total, 8, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->work_end);
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
    MDG_CUDA_TRY(cudaEventSynchronize(ln.done));
    mdg_fit_ticket_slot& tk = ctx->ticket[ln.owner];
    tk.t.map_ms += elapsed(ln.begin, ln.map_end);
    tk.t.nuts_ms += elapsed(ln.map_end, ln.nuts_end);
    tk.t.ppc_ms += elapsed(ln.nuts_end, ln.pred_end);
    tk.t.assemble_ms += elapsed(ln.pred_end, ln.done);
    tk.t.total_ms = std::max(tk.t.total_ms, elapsed(tk.ev_begin, ln.done));
    tk.t.n_launches += ln.launches;
    for (int r = 0; r < MDG_NUM_RUNS; ++r) tk.t.leapfrogs[r] += ln.h_leap[r];
    // NUTS-active time as a union of intervals over everything harvested on this ctx (chunks of overlapping
    // batches run their NUTS launches concurrently; chunks are harvested in submission order)
    const double a = ms_since_epoch(ctx, ln.map_end), b = ms_since_epoch(ctx, ln.nuts_end);
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

// Frees the slot of a batch whose submit failed, after waiting for its chunks already enqueued: no lane may keep an
// owner that points at a free slot, and the next batch must not stage into the slot's arena under a running chunk.
void abandon_ticket(mdg_ctx* ctx, int slot) {
    const std::string error = g_error;  // the submit's error, not one of the waits'
    for (auto& ln : ctx->lane)
        if (ln.busy && ln.owner == slot && harvest_lane(ctx, ln) != MDG_OK) {
            ln.busy = false;
            ln.owner = -1;
        }
    ctx->ticket[slot].active = false;
    set_error("%s", error.c_str());
}

// the five per-TaxID inputs of mdg_fit_batch_submit and mdg_map_batch
struct FitInputs {
    const int64_t* tax;
    const uint32_t *k, *N, *m12;
    const double* noise;
};

void stage_fit_inputs(Stage& stage, FitInputs& d, size_t nt, int R, const int64_t* tax_id, const uint32_t* k,
                      const uint32_t* N, const uint32_t* mism12, const double* noise3) {
    stage.in(d.tax, tax_id, nt * 8);
    stage.in(d.k, k, nt * R * 4);
    stage.in(d.N, N, nt * R * 4);
    stage.in(d.m12, mism12, nt * R * 12 * 4);
    stage.in(d.noise, noise3, nt * 24);
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
        cfg->max_tree_depth > kMaxTreeDepth || cfg->max_leapfrogs_per_run < 0 || !(cfg->hpdi_prob > 0.0 && cfg->hpdi_prob <= 1.0)) {
        // K6's HPDI window is buf[i .. i + (int)(hpdi_prob * S)], clamped to S - 1 from above only
        set_error("mdg_fit_batch: need 1 <= num_samples <= 4096, num_warmup >= 0, 1 <= max_tree_depth <= %d, max_leapfrogs_per_run >= 0, "
                  "0 < hpdi_prob <= 1",
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
    // from here on every error return frees the slot again
    struct Abandon {
        mdg_ctx* ctx;
        int slot;
        bool armed = true;
        ~Abandon() {
            if (armed) abandon_ticket(ctx, slot);
        }
    } abandon{ctx, slot};
    MDG_CUDA_TRY(cudaEventRecord(tk.ev_begin, st));
    if (n_tax == 0) {
        abandon.armed = false;
        return MDG_OK;
    }
    const int P = max_position, R = 2 * P, S = cfg->num_samples, W = cfg->num_warmup;
    const bool host = (mem == MDG_HOST);
    const bool fwd_rev = cfg->do_fwd_rev != 0;
    const Priors pr = make_priors(*cfg);

    const int sample_runs = out_samples ? MDG_NUM_RUNS : (fwd_rev ? 3 : 1);
    const int items_per_tax = R + (fwd_rev ? 2 : 0);
    // TaxIDs per chunk: every chunk ends with the tail of its NUTS launches (the next chunk starts under
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

    // ---- the caller's buffers (MDG_DEVICE) or staged ones (MDG_HOST: whole batch, owned by the ticket) ----
    int rc;
    const size_t nt = (size_t)n_tax;
    FitInputs d;
    mdg_fit_result* d_out;
    float *d_med, *d_lo, *d_hi;
    double *d_samples, *d_trace, *d_waic_user;
    Stage stage(tk.arena, host, st);
    stage_fit_inputs(stage, d, nt, R, tax_id, k, N, mism12, noise3);
    stage.out(d_out, out, sizeof(mdg_fit_result), nt);
    // the assembly writes the medians and HPDI bounds whether or not the caller wants them
    for (auto [field, dst] : {std::make_pair(&d_med, out_median), std::make_pair(&d_lo, out_hpdi_lo), std::make_pair(&d_hi, out_hpdi_hi)}) {
        if (dst) stage.out(*field, dst, (size_t)R * 4, nt);
        else stage.scratch(*field, nt * R * 4);
    }
    stage.out(d_samples, out_samples, (size_t)MDG_NUM_RUNS * S * 4 * 8, nt);
    stage.out(d_trace, out_trace, (size_t)MDG_NUM_RUNS * (W + S) * 4 * 8, nt);
    stage.out(d_waic_user, out_waic, (size_t)MDG_NUM_RUNS * 2 * R * 8, nt);
    if ((rc = stage.commit())) return rc;
    if (!ctx->da_tables.ptr) {
        // the same libm calls as the reference arithmetic (t^-0.75 by pow, sqrt), made once on the host
        std::vector<double> tab(2 * kDaTable);
        for (int t = 0; t < kDaTable; ++t) { tab[t] = sqrt((double)t); tab[kDaTable + t] = t ? pow((double)t, -0.75) : 0.0; }
        if ((rc = ctx->da_tables.ensure(tab.size() * sizeof(double)))) return rc;
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
        if ((rc = harvest_lane(ctx, ln))) return rc;  // the lane's previous chunk (host wait only if it is still running)
        // ---- per-lane scratch ----
        if ((rc = ln.rec.ensure((size_t)chunk_max * MDG_NUM_RUNS * sizeof(RunRecord)))) return rc;
        if ((rc = ln.map.ensure((size_t)chunk_max * 2 * sizeof(MapRecord)))) return rc;
        if ((rc = ln.pred.ensure((size_t)chunk_max * items_per_tax * 3 * sizeof(double)))) return rc;
        if ((rc = ln.counters.ensure(256))) return rc;  // work counters + leapfrog totals
        if (!out_samples && (rc = ln.samples.ensure((size_t)chunk_max * sample_runs * S * 4 * sizeof(double)))) return rc;
        if (!out_waic && (rc = ln.waic.ensure((size_t)chunk_max * MDG_NUM_RUNS * 2 * R * sizeof(double)))) return rc;
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
        MDG_CUDA_TRY(cudaEventRecord(ln.begin, ls));
        if (cfg->do_map) {
            MapLaunch ml = {};
            ml.tax_id = d.tax + c0; ml.k = d.k + (size_t)c0 * R; ml.N = d.N + (size_t)c0 * R;
            ml.n_tax = nc; ml.P = P; ml.pr = pr; ml.work_counter = d_counters + 0; ml.rec = d_map;
            if ((rc = launch_map(ctx, ls, ml))) return rc;
        }
        MDG_CUDA_TRY(cudaEventRecord(ln.map_end, ls));

        // ---- K4 NUTS: one launch per model, each on its own stream (they share the SMs as CTAs retire) ----
        FitLaunch fl = {};
        fl.tax_id = d.tax + c0; fl.k = d.k + (size_t)c0 * R; fl.N = d.N + (size_t)c0 * R;
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
            if ((rc = ln.order.ensure(off_cnt + 3 * kOrderBuckets * sizeof(unsigned int)))) return rc;
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
            if ((rc = ln.chain_clock.ensure((size_t)chunk_max * MDG_NUM_RUNS * 16))) return rc;
            MDG_CUDA_TRY(cudaMemsetAsync(ln.chain_clock.ptr, 0, (size_t)nc * MDG_NUM_RUNS * 16, ls));
            fl.chain_clock = ln.chain_clock.as<unsigned long long>();
            ln.clock_items = nc * MDG_NUM_RUNS;
        }
        // Overlap with the chunk in flight on another lane is wanted for its TAIL only (a few long chains on an
        // otherwise idle GPU), not for its bulk: two different NUTS kernels sharing the SMs evict each other from
        // the instruction cache (measured: -2..-5 % with unrestricted overlap). So this chunk's NUTS launches wait
        // until the other chunk's PMD launch is through and only its null launch (short, uniform chains) is still
        // running.
        for (auto& other : ctx->lane)
            if (&other != &ln && other.busy) MDG_CUDA_TRY(cudaStreamWaitEvent(ls, other.nuts_join[0], 0));
        MDG_CUDA_TRY(cudaEventRecord(ln.nuts_fork, ls));
        for (cudaStream_t sd : ln.side) MDG_CUDA_TRY(cudaStreamWaitEvent(sd, ln.nuts_fork, 0));
        {
            // Launch order = dispatch order of the persistent CTAs: the kernels share the SMs as CTAs
            // retire, so the whole step behaves like one list schedule over all (TaxID, run) items.
            // PMD chains are long and heavy-tailed (adapted step size; max ~8x the mean), null chains
            // short and uniform: PMD first, null last fills the tail (profiles/r01_nuts_tuning.md).
            // One launch and ONE queue per model: the all-position runs first (the longest chains), then the
            // forward-only / reverse-only runs. A group that finishes a chain always finds the next item until the
            // model's whole queue is empty, so the only hand-over between launches (CTA slots are released per CTA,
            // i.e. when the last of its 16 chains ends) is PMD -> null.
            FitLaunch a = fl;  // PMD
            a.n_items = fwd_rev ? 3 * nc : nc; a.n_items_all = nc; a.work_counter = d_counters + 1;
            FitLaunch b = a;   // null
            b.work_counter = d_counters + 2;
            if ((rc = launch_nuts_group<0>(ctx, ln.side[0], a, ln.waic_acc[0]))) return rc;
            if ((rc = launch_nuts_group<1>(ctx, ln.side[1], b, ln.waic_acc[1]))) return rc;
        }
        for (int m = 0; m < 2; ++m) {
            MDG_CUDA_TRY(cudaEventRecord(ln.nuts_join[m], ln.side[m]));
            MDG_CUDA_TRY(cudaStreamWaitEvent(ls, ln.nuts_join[m], 0));
        }
        MDG_CUDA_TRY(cudaEventRecord(ln.nuts_end, ls));

        // ---- K6 posterior predictive ----
        {
            PpcLaunch pl = {};
            pl.tax_id = d.tax + c0; pl.N = d.N + (size_t)c0 * R; pl.n_tax = nc; pl.P = P; pl.cfg = *cfg; pl.pr = pr;
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
        MDG_CUDA_TRY(cudaEventRecord(ln.pred_end, ls));

        // ---- K5/K7 assembly ----
        {
            AssembleLaunch al = {};
            al.tax_id = d.tax + c0; al.k = d.k + (size_t)c0 * R; al.N = d.N + (size_t)c0 * R;
            al.mism12 = d.m12 ? d.m12 + (size_t)c0 * R * 12 : nullptr;
            al.noise3 = d.noise ? d.noise + (size_t)c0 * 3 : nullptr;
            al.n_tax = nc; al.P = P; al.cfg = *cfg; al.rec = d_rec; al.map = cfg->do_map ? d_map : nullptr;
            al.waic = d_waic; al.pred = d_pred; al.items_per_tax = items_per_tax;
            al.out = d_out + c0; al.out_median = d_med + (size_t)c0 * R; al.out_lo = d_lo + (size_t)c0 * R;
            al.out_hi = d_hi + (size_t)c0 * R; al.leapfrog_totals = d_leap;
            assemble_kernel<<<(nc + 127) / 128, 128, 0, ls>>>(al);
            MDG_CUDA_TRY(cudaGetLastError());
            ctx->timings.n_launches++;
        }
        // ---- this chunk's results back to the caller's host buffers ----
        if ((rc = stage.copy_back((size_t)c0, (size_t)nc, ls))) return rc;
        MDG_CUDA_TRY(cudaMemcpyAsync(ln.h_leap, d_leap, MDG_NUM_RUNS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ls));
        MDG_CUDA_TRY(cudaEventRecord(ln.done, ls));
        ln.launches = ctx->timings.n_launches - launches_before;
        ln.busy = true;
        ln.owner = slot;
    }
    abandon.armed = false;
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
            MDG_CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ln.done, 0));
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
    const size_t nt = (size_t)n_tax;
    // TaxIDs per piece: bounds the per-run records (624 MB per 2^20 TaxIDs); results go straight to their rows
    const long long piece = 1ll << 20;
    const long long piece_max = std::min<long long>(n_tax, piece);
    int rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));
    FitInputs d;
    mdg_map_result* d_out;
    Stage stage(ctx->arena, mem == MDG_HOST, st);
    stage_fit_inputs(stage, d, nt, R, tax_id, k, N, mism12, noise3);
    stage.out(d_out, out, sizeof(mdg_map_result), nt);
    if ((rc = stage.commit())) return rc;
    if ((rc = ctx->map_counters.ensure(256))) return rc;
    unsigned int* d_counter = ctx->map_counters.as<unsigned int>();                           // [1] work counter
    unsigned long long* d_evals = reinterpret_cast<unsigned long long*>(d_counter + 16);      // [6] gradient evaluations
    MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, st));
    if (n_tax > 0 && (rc = ctx->map_rec.ensure((size_t)piece_max * MDG_NUM_RUNS * sizeof(mdg_map_run)))) return rc;
    const Priors pr = make_priors(*cfg);
    for (long long c0 = 0; c0 < n_tax; c0 += piece) {
        const int nc = (int)std::min<long long>(piece, n_tax - c0);
        if (c0 > 0) MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), st));
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
        MapBatchLaunch ml = {};
        ml.k = d.k + (size_t)c0 * R; ml.N = d.N + (size_t)c0 * R; ml.n_tax = nc; ml.P = P; ml.n_runs = n_runs;
        ml.pr = pr; ml.work_counter = d_counter; ml.rec = ctx->map_rec.as<mdg_map_run>();
        if ((rc = launch_map_batch(ctx, st, ml))) return rc;
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
        MapAssembleLaunch al = {};
        al.tax_id = d.tax + c0; al.k = ml.k; al.N = ml.N;
        al.mism12 = d.m12 ? d.m12 + (size_t)c0 * R * 12 : nullptr;
        al.noise3 = d.noise ? d.noise + (size_t)c0 * 3 : nullptr;
        al.n_tax = nc; al.P = P; al.n_runs = n_runs; al.rec = ml.rec; al.out = d_out + c0; al.eval_totals = d_evals;
        map_assemble_kernel<<<(nc + 127) / 128, 128, 0, st>>>(al);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches++;
        MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));  // the piece's end here; the call's at the end
        MDG_CUDA_TRY(cudaEventSynchronize(ctx->call_end));  // the events are reused by the next piece
        ctx->timings.map_ms += elapsed(ctx->work_begin, ctx->work_end);
        ctx->timings.assemble_ms += elapsed(ctx->work_end, ctx->call_end);
    }
    if ((rc = stage.copy_back(0, nt, st))) return rc;
    unsigned long long evals[MDG_NUM_RUNS];
    MDG_CUDA_TRY(cudaMemcpyAsync(evals, d_evals, sizeof evals, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));
    MDG_CUDA_TRY(cudaEventSynchronize(ctx->call_end));
    for (int r = 0; r < MDG_NUM_RUNS; ++r) ctx->timings.leapfrogs[r] = evals[r];
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->call_end);
    return MDG_OK;
}

int mdg_map_profile(mdg_ctx* ctx, int mem, int64_t n_tax, int max_position, const uint32_t* k, const uint32_t* N,
                    const mdg_fit_config* cfg, const mdg_map_result* map, double level, mdg_map_interval* out) {
    if (!ctx) { set_error("ctx is NULL"); return MDG_ERR_INVALID; }
    if (!cfg || n_tax < 0 || max_position < 1 || max_position > MDG_MAX_POSITION || (mem != MDG_HOST && mem != MDG_DEVICE) ||
        !(level > 0.0 && level < 1.0)) {
        set_error("mdg_map_profile: invalid argument (need 0 < level < 1)");
        return MDG_ERR_INVALID;
    }
    if (n_tax > 0 && (!k || !N || !map || !out)) { set_error("mdg_map_profile: NULL k/N/map/out"); return MDG_ERR_INVALID; }
    DeviceGuard guard(ctx->device);
    cudaStream_t st = ctx->stream;
    ctx->timings = mdg_timings{};
    const int P = max_position, R = 2 * P;
    const int n_prof = cfg->do_fwd_rev ? 3 : 1;
    const size_t nt = (size_t)n_tax;
    // TaxIDs per launch: keeps the item index (6 per TaxID) in 32 bits
    const long long piece = 1ll << 20;
    int rc;
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_begin, st));
    const uint32_t *d_k, *d_N;
    const mdg_map_result* d_map;
    mdg_map_interval* d_out;
    Stage stage(ctx->arena, mem == MDG_HOST, st);
    stage.in(d_k, k, nt * R * 4);
    stage.in(d_N, N, nt * R * 4);
    stage.in(d_map, map, nt * sizeof(mdg_map_result));
    stage.out(d_out, out, sizeof(mdg_map_interval), nt);
    if ((rc = stage.commit())) return rc;
    if ((rc = ctx->map_counters.ensure(256))) return rc;
    unsigned int* d_counter = ctx->map_counters.as<unsigned int>();                       // [1] work counter
    unsigned long long* d_evals = reinterpret_cast<unsigned long long*>(d_counter + 16);  // [6] gradient evaluations
    MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, st));
    const Priors pr = make_priors(*cfg);
    for (long long c0 = 0; c0 < n_tax; c0 += piece) {
        const int nc = (int)std::min<long long>(piece, n_tax - c0);
        if (c0 > 0) MDG_CUDA_TRY(cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), st));
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
        MapProfileLaunch ml = {};
        ml.k = d_k + (size_t)c0 * R; ml.N = d_N + (size_t)c0 * R; ml.map = d_map + c0;
        ml.n_tax = nc; ml.P = P; ml.n_prof = n_prof; ml.pr = pr; ml.level = level;
        ml.work_counter = d_counter; ml.eval_totals = d_evals; ml.out = d_out + c0;
        if ((rc = launch_map_profile(ctx, st, ml))) return rc;
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
        map_interval_header_kernel<<<(nc + 127) / 128, 128, 0, st>>>(ml.map, nc, n_prof, level, ml.out);
        MDG_CUDA_TRY(cudaGetLastError());
        ctx->timings.n_launches++;
        MDG_CUDA_TRY(cudaEventSynchronize(ctx->work_end));  // the events are reused by the next piece
        ctx->timings.map_ms += elapsed(ctx->work_begin, ctx->work_end);
    }
    if ((rc = stage.copy_back(0, nt, st))) return rc;
    unsigned long long evals[MDG_NUM_RUNS];
    MDG_CUDA_TRY(cudaMemcpyAsync(evals, d_evals, sizeof evals, cudaMemcpyDeviceToHost, st));
    MDG_CUDA_TRY(cudaEventRecord(ctx->call_end, st));
    MDG_CUDA_TRY(cudaEventSynchronize(ctx->call_end));
    for (int r = 0; r < MDG_NUM_RUNS; ++r) ctx->timings.leapfrogs[r] = evals[r];
    ctx->timings.total_ms = elapsed(ctx->call_begin, ctx->call_end);
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

__global__ void test_betabinom_kernel(uint64_t seed, long long n, double alpha, double beta, double trials, double* out) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    log_table_init();
    if (i < n) {
        Stream st;
        st.key = make_key(seed, 12345); st.c0 = 0u; st.c1 = (uint32_t)i; st.c2 = c2word(0, P_PPC); st.c3 = (uint32_t)(i >> 32); st.have = false; st.stash = 0.0;
        const double p = beta_variate(st, alpha, beta);
        out[i] = binomial_variate(st, trials, p);
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
    int rc = ctx->test_scratch.ensure((size_t)n * 24);
    if (rc) return rc;
    double* d = ctx->test_scratch.as<double>();
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
    int rc = ctx->test_scratch.ensure((size_t)n * 24);
    if (rc) return rc;
    double* d = ctx->test_scratch.as<double>();
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
    int rc = ctx->test_scratch.ensure((size_t)n * 40);
    if (rc) return rc;
    uint32_t* d = ctx->test_scratch.as<uint32_t>();
    MDG_CUDA_TRY(cudaMemcpyAsync(d, key2, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    MDG_CUDA_TRY(cudaMemcpyAsync(d + 2 * n, ctr4, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    test_philox_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, d, d + 2 * n, d + 6 * n);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out4, d + 6 * n, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    MDG_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return MDG_OK;
}

int mdg_test_betabinom_draws(mdg_ctx* ctx, uint64_t seed, int64_t n_draws, double alpha, double beta, double n, double* out) {
    if (!ctx || n_draws < 0 || (n_draws > 0 && !out) || !(alpha > 0.0) || !(beta > 0.0) || !(n >= 0.0)) {
        set_error("mdg_test_betabinom_draws: need n_draws >= 0, out, alpha > 0, beta > 0, n >= 0");
        return MDG_ERR_INVALID;
    }
    if (n_draws == 0) return MDG_OK;
    DeviceGuard guard(ctx->device);
    int rc = ctx->test_scratch.ensure((size_t)n_draws * 8);
    if (rc) return rc;
    double* d = ctx->test_scratch.as<double>();
    test_betabinom_kernel<<<(unsigned)((n_draws + 255) / 256), 256, 0, ctx->stream>>>(seed, n_draws, alpha, beta, n, d);
    MDG_CUDA_TRY(cudaGetLastError());
    MDG_CUDA_TRY(cudaMemcpyAsync(out, d, (size_t)n_draws * 8, cudaMemcpyDeviceToHost, ctx->stream));
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
    int rc = ctx->test_scratch.ensure((size_t)R * 8 + ne * (32 + 8 + 32 + (size_t)R * 8) + 1024);
    if (rc) return rc;
    unsigned char* base = ctx->test_scratch.as<unsigned char>();
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
    const unsigned grid = (unsigned)n_eval;
    with_npl(n_obs, [&](auto npl) {
        constexpr int NPL = decltype(npl)::value;
        auto kern = model == 0 ? test_logp_kernel<0, NPL> : test_logp_kernel<1, NPL>;
        kern<<<grid, 32, 0, st>>>(P, dk, dN, pr, lane_mask, with_jacobian, n_eval, du, dlogp, dgrad, out_ll ? dll : nullptr);
    });
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
    int rc = ctx->test_scratch.ensure(64);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    const int iters = 20000, threads = 512, blocks = ctx->num_sms * 4;
    fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->test_scratch.as<double>(), 1000);  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_begin, st));
        fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->test_scratch.as<double>(), iters);
        MDG_CUDA_TRY(cudaEventRecord(ctx->work_end, st));
        MDG_CUDA_TRY(cudaStreamSynchronize(st));
        MDG_CUDA_TRY(cudaGetLastError());
        const double ms = elapsed(ctx->work_begin, ctx->work_end);
        const double flops = 2.0 * 8.0 * iters * (double)threads * blocks;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *out_tflops = best;
    return MDG_OK;
}

}  // extern "C"
