// mdg_counts_kernel.cuh — K1 counts_reduce: the mismatch matrix -> per-row reference sums, error
// rates, signed positions, per-TaxID y_sum_total, cut flags and the dense k(z)/N(z) batch.
// Replaces counts.py:237-256 (add_reference_counts 86-89, add_error_rates 109-114, position
// handling 117-129, fillna 175-176, y_sum_total 179-204, cuts 207-209) and the dense extraction
// of fits.py:398-419; optionally the noise statistic of fits.py:359-376.
//
// This file holds what the streaming kernel (mdg_counts_stream.cuh) is built on: the launch struct,
// the bit-exact error rate, and the scans and block permute that put its per-TaxID rows into input
// order; also K1d, the row order of df_counts. counts_scan_kernel serves K0 and K8 as well.
//
// HBM-bound (111 algorithmic bytes per row, SURVEY.md 8d). A tile of rows owns every TaxID whose
// first row it holds, so no carry crosses tiles: the only traffic between tiles is ONE atomicAdd per
// tile that reserves the tile's block of dense output rows (in no particular order); a scan of the
// per-tile counts and a block permute then put the blocks into input order. A decoupled look-back
// that writes the rows straight to their final places was measured slower: every tile then waits
// for its predecessors to publish their counts (DESIGN.md §4, profiles/r01_counts_ncu.md).
#pragma once
#include "mdg_common.cuh"

namespace mdg {

enum CountsError : int { CE_NONE = 0, CE_SEGMENT_TOO_LONG = 1, CE_OVERFLOW = 2, CE_CAPACITY = 3 };

struct CountsLaunch {
    long long n_rows;
    const long long* tax_id;
    const uint32_t* n_align;
    const uint8_t* is_rev;
    const uint8_t* pos0;
    const uint32_t* counts16;
    long long stride;
    int fwd_ref, fwd_obs, rev_ref, rev_obs;
    int P;
    uint32_t min_align;
    unsigned long long min_y;
    // per-row outputs (any may be NULL)
    uint32_t* n_fwd_row;
    uint32_t* n_rev_row;
    float* f_fwd_row;
    float* f_rev_row;
    int8_t* z_row;
    unsigned long long* y_row;
    uint8_t* keep_row;
    // per-TaxID outputs
    long long* out_tax;
    uint32_t* out_nal;
    long long* out_first;
    uint32_t* out_k;
    uint32_t* out_N;
    double* out_noise;
    int vec_in;             // input column bases 16-byte aligned and stride % 4 == 0 -> 128-bit loads
    int vec_out;            // per-row output bases 16-byte aligned -> 128-bit stores
    unsigned long long* kept_counter;  // device scalar: dense rows reserved so far (unordered, one atomicAdd per tile)
    long long* tile_base;              // [n_tiles] start of the tile's block in the temporary dense arrays
    int* tile_cnt;                     // [n_tiles] kept TaxIDs of the tile
    long long capacity;                // rows available in the per-TaxID arrays
    int* error_flag;
};

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// IEEE double division, kept out of line: error_rate needs it for about one value in 2^26, but
// inlined it was if-converted and executed for every row (ncu: 14.6 % of the kernel's instructions).
__device__ __noinline__ double exact_div(double a, double b) { return a / b; }

// float32(double(k) / double(n)) with 0/0 -> 0 (counts.py:99, 254), bit-exact.
// Fast path: q = k * (1/n) refined once (Markstein): at most 1 ulp(double) from the correctly
// rounded quotient, which changes the float32 result only if q sits within a few ulps of a
// float32 rounding boundary; exactly those (about 1 in 2^26) values take the IEEE division.
__device__ __forceinline__ float error_rate(uint32_t k, uint32_t n) {
    const double a = (double)(k ? k : 1u), b = (double)(n ? n : 1u);
    const double y = rcp_pos(b);
    const double q0 = a * y;
    double q = fma(fma(-b, q0, a), y, q0);
    const unsigned low = (unsigned)__double2loint(q) & 0x1fffffffu;  // the 29 bits float32 drops
    if (low - 0x0ffffffcu <= 8u) q = exact_div(a, b);                // within 4 ulps of a tie: exact path
    return (k && n) ? (float)q : 0.0f;
}

// ---------------------------------------------------------------------------------------------
// exclusive scan of per-block counts (one CTA) -> final block starts and the total; K1d, K0 and K8
// scan with it, K1 with the two-level form below
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) counts_scan_kernel(const int* __restrict__ tile_cnt, long long n_tiles,
                                                           long long* __restrict__ final_base, long long* __restrict__ n_tax_out) {
    // warp w scans a contiguous range with coalesced 32-element steps and a running carry; the 32 warp totals are
    // scanned by warp 0; a second coalesced pass adds each warp's offset
    __shared__ long long s_tot[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long per = ((n_tiles + 31) / 32 + 31) / 32 * 32;  // elements per warp, a multiple of 32
    const long long lo = (long long)warp * per, hi = lo + per < n_tiles ? lo + per : n_tiles;
    long long running = 0;
    for (long long i = lo; i < hi; i += 32) {
        const long long t = i + lane;
        const long long v = t < hi ? (long long)tile_cnt[t] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        if (t < hi) final_base[t] = running + incl - v;
        running += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_tot[warp] = running;
    __syncthreads();
    if (warp == 0) {
        const long long v = s_tot[lane];
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        s_tot[lane] = incl - v;
        if (lane == 31) *n_tax_out = incl;
    }
    __syncthreads();
    const long long off = s_tot[warp];
    if (off != 0)
        for (long long i = lo + lane; i < hi; i += 32) final_base[i] += off;
}

// Two-level form for many tiles (the streaming kernel has one per 128 rows): every CTA scans a chunk of 1024 counts
// (one per thread, coalesced) and records the chunk total; one more tiny launch scans the chunk totals. The final
// position of tile t is chunk_off[t / 1024] + final_base[t].
constexpr int kScanChunk = 1024;

__global__ void __launch_bounds__(kScanChunk) counts_scan_local_kernel(const int* __restrict__ tile_cnt, long long n_tiles,
                                                                       long long* __restrict__ final_base, long long* __restrict__ chunk_tot) {
    __shared__ long long s_w[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long t = (long long)blockIdx.x * kScanChunk + threadIdx.x;
    const long long v = t < n_tiles ? (long long)tile_cnt[t] : 0;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const long long w = s_w[lane];
        long long wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += u; }
        s_w[lane] = wi - w;
        if (lane == 31) chunk_tot[blockIdx.x] = wi;
    }
    __syncthreads();
    if (t < n_tiles) final_base[t] = s_w[warp] + incl - v;
}

__global__ void __launch_bounds__(32) counts_scan_chunks_kernel(long long* __restrict__ chunk_tot, long long n_chunks,
                                                                long long* __restrict__ n_tax_out) {
    const int lane = threadIdx.x;
    long long running = 0;
    for (long long i = 0; i < n_chunks; i += 32) {
        const long long c = i + lane;
        const long long v = c < n_chunks ? chunk_tot[c] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        if (c < n_chunks) chunk_tot[c] = running + incl - v;  // in place: exclusive offsets
        running += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) *n_tax_out = running;
}

// K1c: move every tile's block of per-TaxID rows from its reserved (unordered) place to input order
struct CountsPermute {
    long long n_tiles;
    const long long* tile_base;
    const long long* final_base;
    const long long* chunk_off;  // two-level scan: offset of tile t's chunk (t / kScanChunk), or NULL
    const int* tile_cnt;
    int R;
    const long long* t_tax; long long* out_tax;
    const uint32_t* t_nal; uint32_t* out_nal;
    const long long* t_first; long long* out_first;
    const uint32_t* t_k; uint32_t* out_k;
    const uint32_t* t_N; uint32_t* out_N;
};

constexpr int kPermuteWarps = 4;
constexpr int kPermuteTiles = 8;  // consecutive tiles per warp (a divisor of kScanChunk): their blocks are adjacent in the output

// One warp moves the blocks of kPermuteTiles consecutive tiles. Their destinations are contiguous (the scan), so the
// warp sees one output block of `total` per-TaxID rows whose sources are up to eight pieces; the tile bookkeeping is read
// once (lanes 0-7) and handed round by shuffles, so no load depends on another load, and the k / N rows go four at a
// time — all loads of a round are issued before its stores. (Round 2's first version ran one warp per tile: 78 125 tiny
// warps = 19 532 CTAs for the 10M-row input, CTA dispatch alone took most of its 38 us.)
__global__ void __launch_bounds__(kPermuteWarps * 32, 8) counts_permute_kernel(const CountsPermute p) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const long long t0 = ((long long)blockIdx.x * kPermuteWarps + (threadIdx.x >> 5)) * kPermuteTiles;
    if (t0 >= p.n_tiles) return;
    const long long t = t0 + (lane & (kPermuteTiles - 1));
    int cnt = 0;
    long long src = 0;
    if (t < p.n_tiles) { cnt = __ldg(p.tile_cnt + t); src = __ldg(p.tile_base + t); }
    const long long dst0 = __ldg(p.final_base + t0) + (p.chunk_off ? __ldg(p.chunk_off + t0 / kScanChunk) : 0);
    int start[kPermuteTiles];
    long long srcs[kPermuteTiles];
    int total = 0;
#pragma unroll
    for (int i = 0; i < kPermuteTiles; ++i) {
        srcs[i] = __shfl_sync(FULL, src, i);
        start[i] = total;
        total += __shfl_sync(FULL, cnt, i);
    }
    if (total == 0) return;
    // source row of row j of the warp's output block (starts are non-decreasing: the last tile that starts at or
    // before j owns it; empty tiles share their start with the next one and are overridden)
    auto source_row = [&](int j) -> long long {
        long long s = srcs[0];
        int st = 0;
#pragma unroll
        for (int i = 1; i < kPermuteTiles; ++i)
            if (j >= start[i]) { s = srcs[i]; st = start[i]; }
        return s + (j - st);
    };
    for (int j = lane; j < total; j += 32) {
        const long long s = source_row(j);
        if (p.out_tax) p.out_tax[dst0 + j] = p.t_tax[s];
        if (p.out_nal) p.out_nal[dst0 + j] = p.t_nal[s];
        if (p.out_first) p.out_first[dst0 + j] = p.t_first[s];
    }
    const int R = p.R;
    for (int j0 = 0; j0 < total; j0 += 4) {
        long long s[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) s[u] = j0 + u < total ? source_row(j0 + u) : -1;
        for (int c = lane; c < R; c += 32) {
            uint32_t a[4] = {0u, 0u, 0u, 0u}, b[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (s[u] >= 0) {
                    if (p.out_k) a[u] = p.t_k[s[u] * R + c];
                    if (p.out_N) b[u] = p.t_N[s[u] * R + c];
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (s[u] >= 0) {
                    if (p.out_k) p.out_k[(dst0 + j0 + u) * R + c] = a[u];
                    if (p.out_N) p.out_N[(dst0 + j0 + u) * R + c] = b[u];
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K1d: row order of df_counts (counts.py:167-172 sort_by_alignments): TaxIDs by N_alignments descending, then
// tax_id descending (a sort of n_tax keys, done by the caller), and inside a TaxID the kept rows by
// z = +1..+P, -1..-P (sort key 1/z for z > 0 else z, descending; stable). The row-level part — one
// destination per kept row, O(rows) — is these two kernels: one warp per TaxID of the OUTPUT order.
// ---------------------------------------------------------------------------------------------
struct OrderLaunch {
    long long n_rows;
    const long long* tax_id_row;
    const int8_t* z_row;
    const uint8_t* keep_row;     // NULL: every row is kept
    long long n_tax;
    const long long* first_row;  // [n_tax] first row of every kept TaxID (input order)
    const long long* tax_order;  // [n_tax] index (into first_row) of the TaxID that comes i-th in the output
    int* len_sorted;             // [n_tax] kept rows of the i-th TaxID of the output
    const long long* out_start;  // [n_tax] exclusive scan of len_sorted
    long long* perm;             // [kept rows] source row of every output row
    int* error_flag;
};

constexpr int kOrderWarps = 4;

// rank key of a signed 1-indexed position: +1, +2, ..., then -1, -2, ...
__device__ __forceinline__ int order_zslot(int z) { return z > 0 ? z - 1 : 128 - z - 1; }

template <int PASS>
__global__ void __launch_bounds__(kOrderWarps * 32) counts_order_kernel(const OrderLaunch p) {
    __shared__ short s_key[kOrderWarps][MDG_MAX_SEGMENT_ROWS];  // zslot of the kept rows, -1 for dropped rows
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long i = (long long)blockIdx.x * kOrderWarps + warp;
    if (i >= p.n_tax) return;
    const long long r0 = p.first_row[p.tax_order[i]];
    const long long tid = p.tax_id_row[r0];
    // segment length: rows of a TaxID are contiguous
    int L = 0;
    for (int base = 0; base < MDG_MAX_SEGMENT_ROWS; base += 32) {
        const long long r = r0 + base + lane;
        const bool same = r < p.n_rows && p.tax_id_row[r] == tid;
        const unsigned m = __ballot_sync(0xffffffffu, same);
        if (m != 0xffffffffu) { L = base + __ffs(~m) - 1; break; }
        L = base + 32;
    }
    if (L >= MDG_MAX_SEGMENT_ROWS && r0 + L < p.n_rows && p.tax_id_row[r0 + L] == tid) {
        if (lane == 0) atomicMax(p.error_flag, 1);
        return;
    }
    int kept = 0;
    for (int j = lane; j < L; j += 32) {
        const bool k = p.keep_row == nullptr || p.keep_row[r0 + j] != 0;
        s_key[warp][j] = k ? (short)order_zslot((int)p.z_row[r0 + j]) : (short)-1;
        kept += k;
    }
    __syncwarp();
    if (PASS == 0) {
        kept = __reduce_add_sync(0xffffffffu, kept);
        if (lane == 0) p.len_sorted[i] = kept;
    } else {
        const long long base = p.out_start[i];
        for (int j = lane; j < L; j += 32) {
            const int kj = s_key[warp][j];
            if (kj < 0) continue;
            int rank = 0;
            for (int m = 0; m < L; ++m) {
                const int km = s_key[warp][m];
                rank += (km >= 0) && (km < kj || (km == kj && m < j));
            }
            p.perm[base + rank] = r0 + j;
        }
    }
}

}  // namespace mdg
