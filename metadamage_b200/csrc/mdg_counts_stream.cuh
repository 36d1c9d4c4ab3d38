// mdg_counts_stream.cuh — K1 counts_stream_kernel: warp-synchronous streaming counts_reduce (counts.py:237-256 +
// the dense extraction of fits.py:398-419), and the noise statistic of the kept TaxIDs (fits.py:359-376).
//
// NOTHING is shared between warps: staged through shared memory in CTA-wide tiles, the same work is bound by CTA
// barriers, not by HBM (profiles/r01_counts_ncu.md: 36 % DRAM utilisation, top stall `barrier`).
//   * one warp owns 128 consecutive rows, four per lane, loaded straight into registers with 128-bit coalesced
//     global loads (12 independent loads per lane in flight; no shared-memory staging, no TMA: the rows are used
//     once) and written back with 128-bit stores;
//   * TaxID heads, segment indices and kept ranks come from warp shuffles / ballots; per-segment sums go through a
//     129-entry shared-memory table private to the warp; the only synchronisation is __syncwarp;
//   * a warp owns every TaxID whose FIRST row is among its 128 rows; if its last TaxID runs past them it reads on,
//     32 rows at a time (those rows are L2 hits: they are some other warp's own rows), up to MDG_MAX_SEGMENT_ROWS;
//   * kept TaxIDs get their dense k/N row from the same registers; the order is restored by the
//     reserve-with-one-atomic / scan / block-permute triple of mdg_counts_kernel.cuh;
//   * the optional noise statistic has its own kernel over the kept TaxIDs (counts_noise_kernel, below).
#pragma once
#include "mdg_counts_kernel.cuh"

namespace mdg {

constexpr int kStreamRows = 128;   // rows per warp (4 per lane)
constexpr int kStreamWarps = 4;    // independent warps per CTA
#ifndef MDG_STREAM_MINBLOCKS
#define MDG_STREAM_MINBLOCKS 6
#endif

struct StreamWarpShared {
    // y_sum_total per segment of the tile, as two 32-bit sums of 16-bit halves (y = ylo + (yhi << 16); a TaxID has
    // at most 2048 rows, so neither half can wrap): native 32-bit shared-memory atomics instead of 64-bit CAS loops
    uint32_t ylo[kStreamRows + 1], yhi[kStreamRows + 1];
    uint32_t any[kStreamRows + 1];          // some row of the segment has N_alignments >= min and |z| <= P
    uint32_t dk[2 * MDG_MAX_POSITION], dN[2 * MDG_MAX_POSITION];
    uint8_t head[kStreamRows + 4];          // row (0..127) of the segment's first row
    uint8_t keep[kStreamRows + 4];
    uint8_t rank[kStreamRows + 4];          // rank among the tile's kept segments
};

__global__ void __launch_bounds__(kStreamWarps * 32, MDG_STREAM_MINBLOCKS) counts_stream_kernel(const CountsLaunch p) {
    __shared__ StreamWarpShared sh_all[kStreamWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long tile = (long long)blockIdx.x * kStreamWarps + warp;
    const long long row0 = tile * kStreamRows;
    if (row0 >= p.n_rows) return;
    StreamWarpShared& sh = sh_all[warp];
    const int n_in = (int)(p.n_rows - row0 < kStreamRows ? p.n_rows - row0 : kStreamRows);
    const int P = p.P, R = 2 * P;
    const int i0 = lane * 4;
    const long long gi = row0 + i0;
    const unsigned full = 0xffffffffu;

    // ---------------- load 4 rows per lane ----------------
    long long tax[4];
    uint32_t nal[4], a[4][4], b[4][4];  // a[o][j]: count column (fwd_ref, o) of row j; b: (rev_ref, o)
    int pos[4];
    bool rev[4], valid[4];
    const uint32_t* ca = p.counts16 + (long long)(p.fwd_ref * 4) * p.stride;
    const uint32_t* cb = p.counts16 + (long long)(p.rev_ref * 4) * p.stride;
    if (p.vec_in && n_in == kStreamRows) {
        const longlong2 t01 = *reinterpret_cast<const longlong2*>(p.tax_id + gi);
        const longlong2 t23 = *reinterpret_cast<const longlong2*>(p.tax_id + gi + 2);
        tax[0] = t01.x; tax[1] = t01.y; tax[2] = t23.x; tax[3] = t23.y;
        const uint4 n4 = *reinterpret_cast<const uint4*>(p.n_align + gi);
        nal[0] = n4.x; nal[1] = n4.y; nal[2] = n4.z; nal[3] = n4.w;
        const uchar4 pv = *reinterpret_cast<const uchar4*>(p.pos0 + gi);
        const uchar4 rv = *reinterpret_cast<const uchar4*>(p.is_rev + gi);
        pos[0] = pv.x; pos[1] = pv.y; pos[2] = pv.z; pos[3] = pv.w;
        rev[0] = rv.x != 0; rev[1] = rv.y != 0; rev[2] = rv.z != 0; rev[3] = rv.w != 0;
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            const uint4 va = *reinterpret_cast<const uint4*>(ca + (long long)o * p.stride + gi);
            const uint4 vb = *reinterpret_cast<const uint4*>(cb + (long long)o * p.stride + gi);
            a[o][0] = va.x; a[o][1] = va.y; a[o][2] = va.z; a[o][3] = va.w;
            b[o][0] = vb.x; b[o][1] = vb.y; b[o][2] = vb.z; b[o][3] = vb.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) valid[j] = true;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            valid[j] = i0 + j < n_in;
            const long long r = valid[j] ? gi + j : row0;
            tax[j] = p.tax_id[r];
            nal[j] = p.n_align[r];
            pos[j] = p.pos0[r];
            rev[j] = p.is_rev[r] != 0;
#pragma unroll
            for (int o = 0; o < 4; ++o) { a[o][j] = ca[(long long)o * p.stride + r]; b[o][j] = cb[(long long)o * p.stride + r]; }
        }
    }
    long long tax_before = 0;
    if (lane == 0 && row0 > 0) tax_before = p.tax_id[row0 - 1];

    // ---------------- row-local values (counts.py:86-129) ----------------
    uint32_t nf[4], nr[4], kf[4], kr[4], yc[4], zpack = 0;
    float ff[4], fr[4];
    bool inP[4];
    {
        uint32_t any = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            nf[j] = a[0][j] + a[1][j] + a[2][j] + a[3][j];
            nr[j] = b[0][j] + b[1][j] + b[2][j] + b[3][j];
            any |= a[0][j] | a[1][j] | a[2][j] | a[3][j] | b[0][j] | b[1][j] | b[2][j] | b[3][j];
        }
        // a uint32 sum of four terms can only wrap if some term has one of its top two bits set (utils.py:338-339)
        if (any >> 30) {
            bool ovf = false;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const unsigned long long wf = (unsigned long long)a[0][j] + a[1][j] + a[2][j] + a[3][j];
                const unsigned long long wr = (unsigned long long)b[0][j] + b[1][j] + b[2][j] + b[3][j];
                ovf |= valid[j] && (((wf | wr) >> 32) != 0);
            }
            if (ovf) atomicMax(p.error_flag, (int)CE_OVERFLOW);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            kf[j] = p.fwd_obs == 0 ? a[0][j] : (p.fwd_obs == 1 ? a[1][j] : (p.fwd_obs == 2 ? a[2][j] : a[3][j]));
            kr[j] = p.rev_obs == 0 ? b[0][j] : (p.rev_obs == 1 ? b[1][j] : (p.rev_obs == 2 ? b[2][j] : b[3][j]));
            ff[j] = error_rate(kf[j], nf[j]);
            fr[j] = error_rate(kr[j], nr[j]);
            const int zabs = pos[j] + 1;
            inP[j] = valid[j] && zabs <= P;
            yc[j] = inP[j] ? (rev[j] ? kr[j] : kf[j]) : 0u;
            zpack |= ((uint32_t)(uint8_t)(int8_t)(rev[j] ? -zabs : zabs)) << (8 * j);
        }
    }
    if (p.vec_out && n_in == kStreamRows) {
        if (p.n_fwd_row) *reinterpret_cast<uint4*>(p.n_fwd_row + gi) = make_uint4(nf[0], nf[1], nf[2], nf[3]);
        if (p.n_rev_row) *reinterpret_cast<uint4*>(p.n_rev_row + gi) = make_uint4(nr[0], nr[1], nr[2], nr[3]);
        if (p.f_fwd_row) *reinterpret_cast<float4*>(p.f_fwd_row + gi) = make_float4(ff[0], ff[1], ff[2], ff[3]);
        if (p.f_rev_row) *reinterpret_cast<float4*>(p.f_rev_row + gi) = make_float4(fr[0], fr[1], fr[2], fr[3]);
        if (p.z_row) *reinterpret_cast<uint32_t*>(p.z_row + gi) = zpack;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (!valid[j]) continue;
            if (p.n_fwd_row) p.n_fwd_row[gi + j] = nf[j];
            if (p.n_rev_row) p.n_rev_row[gi + j] = nr[j];
            if (p.f_fwd_row) p.f_fwd_row[gi + j] = ff[j];
            if (p.f_rev_row) p.f_rev_row[gi + j] = fr[j];
            if (p.z_row) p.z_row[gi + j] = (int8_t)((zpack >> (8 * j)) & 0xffu);
        }
    }

    // ---------------- TaxID heads and segment indices ----------------
    long long prev = __shfl_up_sync(full, tax[3], 1);
    if (lane == 0) prev = tax_before;
    bool head[4];
    int nheads = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        head[j] = valid[j] && ((gi + j == 0) || (tax[j] != (j == 0 ? prev : tax[j - 1])));
        nheads += head[j] ? 1 : 0;
    }
    int incl = nheads;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(full, incl, o); if (lane >= o) incl += t; }
    const int nseg = __shfl_sync(full, incl, 31);
    int seg[4];  // segment of row j; -1: a TaxID that started in an earlier tile (owned by that tile's warp)
    {
        int s = incl - nheads - 1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (head[j]) { ++s; sh.head[s] = (uint8_t)(i0 + j); }
            seg[j] = s;
        }
    }
    for (int s = lane; s <= nseg; s += 32) { sh.ylo[s] = 0u; sh.yhi[s] = 0u; sh.any[s] = 0u; }
    __syncwarp();

    // ---------------- per-TaxID y_sum_total and the cut (counts.py:179-209) ----------------
    {
        int cur = seg[0];
        uint32_t lo = 0, hi = 0, any = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (seg[j] != cur) {
                if (cur >= 0) { if (lo | hi) { atomicAdd(&sh.ylo[cur], lo); atomicAdd(&sh.yhi[cur], hi); } if (any) atomicOr(&sh.any[cur], 1u); }
                cur = seg[j]; lo = 0; hi = 0; any = 0;
            }
            lo += yc[j] & 0xffffu;
            hi += yc[j] >> 16;
            any |= (inP[j] && nal[j] >= p.min_align) ? 1u : 0u;
        }
        if (cur >= 0) { if (lo | hi) { atomicAdd(&sh.ylo[cur], lo); atomicAdd(&sh.yhi[cur], hi); } if (any) atomicOr(&sh.any[cur], 1u); }
    }
    __syncwarp();
    // the tile's last TaxID may run past the tile: read on, 32 rows at a time
    const long long last_tax = __shfl_sync(full, tax[3], 31);
    const bool has_tail = nseg > 0 && n_in == kStreamRows && row0 + kStreamRows < p.n_rows;
    const uint32_t* ckf = ca + (long long)p.fwd_obs * p.stride;
    const uint32_t* ckr = cb + (long long)p.rev_obs * p.stride;
    int tail_len = 0;
    if (has_tail) {
        uint32_t tlo = 0, thi = 0, tany = 0;  // per lane at most 64 rows: the 16-bit halves cannot wrap
        for (long long r = row0 + kStreamRows;; r += 32) {
            const long long rr = r + lane;
            const bool same = rr < p.n_rows && p.tax_id[rr] == last_tax;
            const unsigned m = __ballot_sync(full, same);
            const int n_same = (m == full) ? 32 : __ffs(~m) - 1;
            if (lane < n_same) {
                const int zabs = (int)p.pos0[rr] + 1;
                if (zabs <= P) {
                    const uint32_t v = p.is_rev[rr] ? ckr[rr] : ckf[rr];
                    tlo += v & 0xffffu;
                    thi += v >> 16;
                    tany |= p.n_align[rr] >= p.min_align ? 1u : 0u;
                }
            }
            tail_len += n_same;
            if (n_same < 32) break;
            if (tail_len > MDG_MAX_SEGMENT_ROWS) break;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            tlo += __shfl_xor_sync(full, tlo, o); thi += __shfl_xor_sync(full, thi, o); tany |= __shfl_xor_sync(full, tany, o);
        }
        if (lane == 0) { atomicAdd(&sh.ylo[nseg - 1], tlo); atomicAdd(&sh.yhi[nseg - 1], thi); atomicOr(&sh.any[nseg - 1], tany); }
        if (tail_len + (kStreamRows - (int)sh.head[nseg - 1]) > MDG_MAX_SEGMENT_ROWS && lane == 0) atomicMax(p.error_flag, (int)CE_SEGMENT_TOO_LONG);
    }
    __syncwarp();

    // ---------------- ranks of the kept TaxIDs; reserve the tile's block of dense rows ----------------
    int running = 0;
    for (int s0 = 0; s0 < nseg; s0 += 32) {
        const int s = s0 + lane;
        const bool k = s < nseg && sh.any[s] != 0u && ((unsigned long long)sh.ylo[s] + ((unsigned long long)sh.yhi[s] << 16)) >= p.min_y;
        const unsigned m = __ballot_sync(full, k);
        if (s < nseg) { sh.keep[s] = k ? 1 : 0; sh.rank[s] = (uint8_t)(running + __popc(m & ((1u << lane) - 1u))); }
        running += __popc(m);
    }
    long long base = 0;
    if (lane == 0) {
        base = running ? (long long)atomicAdd(p.kept_counter, (unsigned long long)running) : 0;
        p.tile_base[tile] = base;
        p.tile_cnt[tile] = running;
        if (base + running > p.capacity) atomicMax(p.error_flag, (int)CE_CAPACITY);
    }
    base = __shfl_sync(full, base, 0);
    __syncwarp();

    // ---------------- y_sum_total and the cut flag of the owned rows ----------------
    if (p.y_row || p.keep_row) {
        unsigned long long y[4];
        uint32_t keeppack = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            y[j] = seg[j] >= 0 ? (unsigned long long)sh.ylo[seg[j]] + ((unsigned long long)sh.yhi[seg[j]] << 16) : 0ull;
            const bool keep = seg[j] >= 0 && inP[j] && nal[j] >= p.min_align && y[j] >= p.min_y;
            keeppack |= (keep ? 1u : 0u) << (8 * j);
        }
        if (p.vec_out && n_in == kStreamRows && seg[0] >= 0) {
            if (p.y_row) {
                *reinterpret_cast<ulonglong2*>(p.y_row + gi) = make_ulonglong2(y[0], y[1]);
                *reinterpret_cast<ulonglong2*>(p.y_row + gi + 2) = make_ulonglong2(y[2], y[3]);
            }
            if (p.keep_row) *reinterpret_cast<uint32_t*>(p.keep_row + gi) = keeppack;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (!valid[j] || seg[j] < 0) continue;
                if (p.y_row) p.y_row[gi + j] = y[j];
                if (p.keep_row) p.keep_row[gi + j] = (uint8_t)((keeppack >> (8 * j)) & 1u);
            }
        }
    }

    // ---------------- dense k/N of the kept TaxIDs (fits.py:398-419); the tail rows' y / keep ----------------
    for (int s = 0; s < nseg; ++s) {
        const bool kept = sh.keep[s] != 0;
        const bool last = has_tail && s == nseg - 1 && tail_len > 0;
        if (!kept && !last) continue;
        const long long o = base + (long long)sh.rank[s];
        const bool emit = kept && o < p.capacity;
        if (emit) {
            for (int i = lane; i < R; i += 32) { sh.dk[i] = 0u; sh.dN[i] = 0u; }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (seg[j] == s && inP[j]) {
                    const int slot = rev[j] ? P + pos[j] : pos[j];
                    atomicAdd(&sh.dk[slot], rev[j] ? kr[j] : kf[j]);
                    atomicAdd(&sh.dN[slot], rev[j] ? nr[j] : nf[j]);
                }
            }
        }
        if (last) {
            const unsigned long long ys = (unsigned long long)sh.ylo[s] + ((unsigned long long)sh.yhi[s] << 16);
            for (int t0 = 0; t0 < tail_len; t0 += 32) {
                const int t = t0 + lane;
                if (t < tail_len) {
                    const long long rr = row0 + kStreamRows + t;
                    const int zabs = (int)p.pos0[rr] + 1;
                    const bool rv = p.is_rev[rr] != 0;
                    const bool in = zabs <= P;
                    if (p.y_row) p.y_row[rr] = ys;
                    if (p.keep_row) p.keep_row[rr] = (in && p.n_align[rr] >= p.min_align && ys >= p.min_y) ? 1 : 0;
                    if (emit && in) {
                        const uint32_t* cn = rv ? cb : ca;
                        const uint32_t nn = cn[rr] + cn[p.stride + rr] + cn[2 * p.stride + rr] + cn[3 * p.stride + rr];
                        const int slot = rv ? P + zabs - 1 : zabs - 1;
                        atomicAdd(&sh.dk[slot], rv ? ckr[rr] : ckf[rr]);
                        atomicAdd(&sh.dN[slot], nn);
                    }
                }
            }
        }
        if (emit) {
            __syncwarp();
            if (p.out_k) for (int i = lane; i < R; i += 32) p.out_k[o * R + i] = sh.dk[i];
            if (p.out_N) for (int i = lane; i < R; i += 32) p.out_N[o * R + i] = sh.dN[i];
            const int hr = sh.head[s];
            if (lane == (hr >> 2)) {
                const int j = hr & 3;
                const long long tx = j == 0 ? tax[0] : (j == 1 ? tax[1] : (j == 2 ? tax[2] : tax[3]));
                const uint32_t na = j == 0 ? nal[0] : (j == 1 ? nal[1] : (j == 2 ? nal[2] : nal[3]));
                if (p.out_tax) p.out_tax[o] = tx;
                if (p.out_nal) p.out_nal[o] = na;
                if (p.out_first) p.out_first[o] = row0 + hr;
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The noise statistic of the kept TaxIDs (fits.py:359-376): one warp per kept TaxID, after the permute
// (first_row in final order). Over the TaxID's rows with |z| <= P: blank CT on forward rows and GA on reverse
// rows, divide every off-diagonal column by its nan-mean, nan-std over all / forward / reverse rows.
// ---------------------------------------------------------------------------------------------
struct NoiseLaunch {
    long long n_rows;
    const long long* tax_id;
    const uint8_t* is_rev;
    const uint8_t* pos0;
    const uint32_t* counts16;
    long long stride;
    int P;
    const long long* n_tax;      // device scalar (kept TaxIDs)
    const long long* first_row;  // [n_tax]
    double* out_noise;           // [n_tax][3]
    long long capacity;
};

__global__ void __launch_bounds__(128) counts_noise_kernel(const NoiseLaunch p) {
    const int lane = threadIdx.x & 31;
    const long long n_tax = *p.n_tax < p.capacity ? *p.n_tax : p.capacity;
    const int OFF[12] = {1, 2, 3, 4, 6, 7, 8, 9, 11, 12, 13, 14};
    for (long long t = (long long)blockIdx.x * 4 + (threadIdx.x >> 5); t < n_tax; t += (long long)gridDim.x * 4) {
        const long long r0 = p.first_row[t];
        const long long tid = p.tax_id[r0];
        int L = 0;
        for (int base = 0; base < MDG_MAX_SEGMENT_ROWS; base += 32) {
            const long long r = r0 + base + lane;
            const bool same = r < p.n_rows && p.tax_id[r] == tid;
            const unsigned m = __ballot_sync(0xffffffffu, same);
            if (m != 0xffffffffu) { L = base + __ffs(~m) - 1; break; }
            L = base + 32;
        }
        const int P = p.P;
        double inv_mean[12];
#pragma unroll
        for (int c = 0; c < 12; ++c) {
            double sm = 0.0, cn = 0.0;
            const uint32_t* col = p.counts16 + (long long)OFF[c] * p.stride;
            for (int r = lane; r < L; r += 32) {
                const int zabs = (int)p.pos0[r0 + r] + 1;
                const bool rev = p.is_rev[r0 + r] != 0;
                const bool blank = (zabs > P) || (!rev && c == 5) || (rev && c == 6);
                if (!blank) { sm += (double)col[r0 + r]; cn += 1.0; }
            }
            sm = warp_sum_f64(sm); cn = warp_sum_f64(cn);
            inv_mean[c] = (cn > 0.0 && sm > 0.0) ? cn / sm : nan("");
        }
        double s1[3] = {0, 0, 0}, n1[3] = {0, 0, 0};
        for (int r = lane; r < L; r += 32) {
            const int zabs = (int)p.pos0[r0 + r] + 1;
            const bool rev = p.is_rev[r0 + r] != 0;
            if (zabs > P) continue;
#pragma unroll
            for (int c = 0; c < 12; ++c) {
                const bool blank = (!rev && c == 5) || (rev && c == 6);
                const double v = (double)p.counts16[(long long)OFF[c] * p.stride + r0 + r] * inv_mean[c];
                if (!blank && !isnan(v)) { s1[0] += v; n1[0] += 1.0; s1[rev ? 2 : 1] += v; n1[rev ? 2 : 1] += 1.0; }
            }
        }
        double mean3[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) { s1[q] = warp_sum_f64(s1[q]); n1[q] = warp_sum_f64(n1[q]); mean3[q] = s1[q] / n1[q]; }
        double s2[3] = {0, 0, 0};
        for (int r = lane; r < L; r += 32) {
            const int zabs = (int)p.pos0[r0 + r] + 1;
            const bool rev = p.is_rev[r0 + r] != 0;
            if (zabs > P) continue;
#pragma unroll
            for (int c = 0; c < 12; ++c) {
                const bool blank = (!rev && c == 5) || (rev && c == 6);
                const double v = (double)p.counts16[(long long)OFF[c] * p.stride + r0 + r] * inv_mean[c];
                if (!blank && !isnan(v)) {
                    const double d0 = v - mean3[0], d1 = v - mean3[rev ? 2 : 1];
                    s2[0] += d0 * d0; s2[rev ? 2 : 1] += d1 * d1;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 3; ++q) s2[q] = warp_sum_f64(s2[q]);
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) p.out_noise[t * 3 + q] = n1[q] > 0.0 ? sqrt(s2[q] / n1[q]) : nan("");
        }
    }
}

}  // namespace mdg
