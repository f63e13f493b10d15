// Attention pass shared by the input-space forward (gat_in_fwd.cu) and the source-major projected forward
// (gat_fwd_msg.cu): lane = edge, exact row statistics rowmax / rowsum (rowsum includes PyG's +1e-16, an empty row stores
// (0, 1e-16)) and one normalised coefficient per (edge, head) at its CSR position.  Rows of <= 32 edges (alone or in
// packs, segmented scans) are finished from registers; longer rows make a statistics sweep and a write sweep (the
// re-gathered logits are L2-warm); hub rows get the same two sweeps chunk-parallel, their chunk statistics folded in
// chunk order (alpha_hub_*).
//
// What is written per edge is the one difference between the two users (AlphaOut):
//   input space (PROJ = false): alpha before dropout with the LeakyReLU-negative region in its sign bit, and
//            jflag[e] = col[e] | (e is the last edge of its row) << 31 -- what the input-space feature passes stream;
//   projected (PROJ = true): alpha_used = edge_alpha(z, m, 1/rowsum) * keep, dropout and its survivor scale applied
//            (explicit mask or the counter RNG on perm[e], as phase A does) -- the same expression the backward
//            evaluates from the saved statistics.
#pragma once
#include "gat_phase_bwd.cuh"

namespace gnnfd {

struct AlphaOut {
    float* alpha;            // [E',H]
    int32_t* jflag;          // [E']   (input space only)
    const int32_t* perm;     // dropout: position of each edge in edge_index' (projected only)
    KeepMask keep;
    float keep_scale;
};

__device__ __forceinline__ float with_sign(float a, bool neg) { return __uint_as_float(__float_as_uint(a) | (neg ? 0x80000000u : 0u)); }

// dropout multipliers of edge e (1 without dropout)
template <int H, bool DROPOUT>
__device__ __forceinline__ void alpha_keep(const AlphaOut& o, int e, float (&kp)[H])
{
    const unsigned kb = DROPOUT ? o.keep.bits(o.perm[e], H) : 0xffu;
#pragma unroll
    for (int h = 0; h < H; ++h) kp[h] = DROPOUT ? ((kb >> h) & 1u ? o.keep_scale : 0.f) : 1.f;
}

// the write sweep of <= 32 edges of ONE row whose statistics (m, 1/s) are known
template <int H, bool PROJ, bool DROPOUT>
__device__ __forceinline__ void alpha_write_chunk(int beg, int n, bool ends_row, const float (&adst)[H], const float (&m)[H],
                                                  const float (&sinv)[H], const int32_t* __restrict__ col,
                                                  const float* __restrict__ a_src, float slope, const AlphaOut& out, int lane)
{
    if (lane < n) {
        const int e = beg + lane, j = col[e];
        float as[H], o[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
        if constexpr (PROJ) {
            float kp[H];
            alpha_keep<H, DROPOUT>(out, e, kp);
#pragma unroll
            for (int h = 0; h < H; ++h) o[h] = edge_alpha(as[h] + adst[h], slope, m[h], sinv[h]) * kp[h];
        } else {
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float z = as[h] + adst[h];
                o[h] = with_sign(expf(leaky(z, slope) - m[h]) * sinv[h], !(z > 0.f));
            }
            out.jflag[e] = j | ((ends_row && lane == n - 1) ? int(0x80000000u) : 0);
        }
        store_vecH<H>(out.alpha + int64_t(e) * H, o);
    }
}

// statistics of <= 32 edges of one row folded into the running (m, s) of the row (all lanes hold the result)
template <int H>
__device__ __forceinline__ void alpha_stat_chunk(int beg, int n, const float (&adst)[H], const int32_t* __restrict__ col,
                                                 const float* __restrict__ a_src, float slope, float (&m)[H], float (&s)[H], int lane)
{
    float e[H];
    if (lane < n) {
        const int j = col[beg + lane];
        float as[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
#pragma unroll
        for (int h = 0; h < H; ++h) e[h] = leaky(as[h] + adst[h], slope);
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) e[h] = -INFINITY;
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float cm = warp_max(e[h]);
        const float cs = warp_sum(lane < n ? expf(e[h] - cm) : 0.f);
        const float mn = fmaxf(m[h], cm);
        s[h] = s[h] * expf(m[h] - mn) + cs * expf(cm - mn);       // expf(-inf) = 0 on the first chunk
        m[h] = mn;
    }
}

// one warp per edge-balanced work item over rowptr; hub rows (above hub_threshold) are left to alpha_hub_*
template <int H, bool PROJ, bool DROPOUT>
__device__ __forceinline__ void alpha_items_body(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                 const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                 int r0, int r1, int hub_threshold, float slope, const AlphaOut& out,
                                                 float* __restrict__ rowmax, float* __restrict__ rowsum, int lane)
{
    ChunkCursor cur;
    cur.start_rows(r0, r1, hub_threshold);
    auto on_empty = [&](int r) {
        if (lane < H) {
            rowmax[int64_t(r) * H + lane] = 0.f;
            rowsum[int64_t(r) * H + lane] = 1e-16f;
        }
    };
    int row = 0, beg = 0, n = 0, k = 0, la = 0, lb = 0;
    bool first = false, last = false;
    while (true) {
        const int kind = cur.next_any(rowptr, lane, row, beg, n, first, last, k, la, lb, on_empty);
        if (!kind) break;
        if (kind == 2) {
            // pack of k whole rows: segmented scans over the lanes of each row (as fwd_phase_a_pack)
            const bool act = lane < n;
            const int e_id = beg + lane;
            int lo = 0, hi = k - 1;
#pragma unroll
            for (int it = 0; it < 5; ++it) {
                const int mid = (lo + hi) >> 1;
                const int bm = __shfl_sync(FULL, lb, mid);
                if (bm > e_id) hi = mid; else lo = min(mid + 1, k - 1);
            }
            const int sa = __shfl_sync(FULL, la, lo) - beg, sb = __shfl_sync(FULL, lb, lo) - beg - 1;
            const int r = row + lo;
            float z[H], kp[H];
            int j = 0;
            if (act) {
                j = col[e_id];
                float as[H], ad[H];
                load_vecH<H>(a_src + int64_t(j) * H, as);
                load_vecH<H>(a_dst + int64_t(r) * H, ad);
#pragma unroll
                for (int h = 0; h < H; ++h) z[h] = as[h] + ad[h];
                if (PROJ) alpha_keep<H, DROPOUT>(out, e_id, kp);
            } else {
#pragma unroll
                for (int h = 0; h < H; ++h) z[h] = -INFINITY;
            }
            float o[H], mrow[H], srow[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float e = act ? leaky(z[h], slope) : -INFINITY;
                float mx = e;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const float t = __shfl_up_sync(FULL, mx, d);
                    if (lane - d >= sa) mx = fmaxf(mx, t);
                }
                mrow[h] = __shfl_sync(FULL, mx, sb);
                const float pexp = act ? expf(e - mrow[h]) : 0.f;
                float sm = pexp;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const float t = __shfl_up_sync(FULL, sm, d);
                    if (lane - d >= sa) sm += t;
                }
                srow[h] = __shfl_sync(FULL, sm, sb) + 1e-16f;       // PyG softmax: out / (sum + 1e-16)
                if (PROJ) o[h] = act ? edge_alpha(z[h], slope, mrow[h], 1.f / srow[h]) * kp[h] : 0.f;
                else      o[h] = with_sign(pexp / srow[h], !(z[h] > 0.f));
            }
            if (act) {
                store_vecH<H>(out.alpha + int64_t(e_id) * H, o);
                if (!PROJ) out.jflag[e_id] = j | (lane == sb ? int(0x80000000u) : 0);
                if (lane == sb) {
                    store_vecH<H>(rowmax + int64_t(r) * H, mrow);
                    store_vecH<H>(rowsum + int64_t(r) * H, srow);
                }
            }
            continue;
        }
        // a single row (kind 1, first chunk of it): statistics sweep over all of its chunks, then the write sweep
        float adst[H], m[H], sv[H];
        load_vecH<H>(a_dst + int64_t(row) * H, adst);
#pragma unroll
        for (int h = 0; h < H; ++h) { m[h] = -INFINITY; sv[h] = 0.f; }
        const int row_beg = beg, r = row;
        alpha_stat_chunk<H>(beg, n, adst, col, a_src, slope, m, sv, lane);
        int row_end = beg + n;
        while (!last) {
            cur.next(rowptr, row, beg, n, first, last, on_empty);     // stays inside the row until last
            alpha_stat_chunk<H>(beg, n, adst, col, a_src, slope, m, sv, lane);
            row_end = beg + n;
        }
        float sinv[H];
#pragma unroll
        for (int h = 0; h < H; ++h) { sv[h] += 1e-16f; sinv[h] = 1.f / sv[h]; }
        if (lane == 0) {
            store_vecH<H>(rowmax + int64_t(r) * H, m);
            store_vecH<H>(rowsum + int64_t(r) * H, sv);
        }
        for (int b = row_beg; b < row_end; b += 32)
            alpha_write_chunk<H, PROJ, DROPOUT>(b, min(32, row_end - b), b + 32 >= row_end, adst, m, sinv, col, a_src, slope,
                                                out, lane);
    }
}

// hub rows: (1) statistics of every chunk, (2) one thread per (hub row, head) folds them in chunk order, (3) write sweep
template <int H>
__device__ __forceinline__ void alpha_hub_stats_body(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                     const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                     const gnnfd_hub_plan_t& plan, int c, float slope,
                                                     float* __restrict__ part_ms, int lane)
{
    const int slot = plan.chunk_hub[c], i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    float adst[H], m[H], sv[H];
    load_vecH<H>(a_dst + int64_t(i) * H, adst);
#pragma unroll
    for (int h = 0; h < H; ++h) { m[h] = -INFINITY; sv[h] = 0.f; }
    for (int b = beg; b < end; b += 32) alpha_stat_chunk<H>(b, min(32, end - b), adst, col, a_src, slope, m, sv, lane);
    if (lane == 0) {
        store_vecH<H>(part_ms + int64_t(c) * 2 * H, m);
        store_vecH<H>(part_ms + int64_t(c) * 2 * H + H, sv);
    }
}
template <int H>
__device__ __forceinline__ void alpha_hub_merge_body(const gnnfd_hub_plan_t& plan, int slot, int h,
                                                     const float* __restrict__ part_ms, float* __restrict__ rowmax,
                                                     float* __restrict__ rowsum)
{
    const int i = plan.hub_row[slot];
    float m = -INFINITY, s = 0.f;
    for (int c = plan.hub_chunk_ptr[slot]; c < plan.hub_chunk_ptr[slot + 1]; ++c) {
        const float cm = part_ms[int64_t(c) * 2 * H + h], cs = part_ms[int64_t(c) * 2 * H + H + h];
        const float mn = fmaxf(m, cm);
        s = s * expf(m - mn) + cs * expf(cm - mn);
        m = mn;
    }
    rowmax[int64_t(i) * H + h] = m;
    rowsum[int64_t(i) * H + h] = s + 1e-16f;
}
template <int H, bool PROJ, bool DROPOUT>
__device__ __forceinline__ void alpha_hub_write_body(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                     const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                     const gnnfd_hub_plan_t& plan, int c, float slope,
                                                     const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                                                     const AlphaOut& out, int lane)
{
    const int slot = plan.chunk_hub[c], i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int row_end = rowptr[i + 1], end = min(row_end, beg + plan.chunk);
    float adst[H], m[H], sinv[H];
    load_vecH<H>(a_dst + int64_t(i) * H, adst);
    load_vecH<H>(rowmax + int64_t(i) * H, m);
    load_vecH<H>(rowsum + int64_t(i) * H, sinv);
#pragma unroll
    for (int h = 0; h < H; ++h) sinv[h] = 1.f / sinv[h];
    for (int b = beg; b < end; b += 32)
        alpha_write_chunk<H, PROJ, DROPOUT>(b, min(32, end - b), b + 32 >= row_end, adst, m, sinv, col, a_src, slope, out,
                                            lane);
}

}  // namespace gnnfd
