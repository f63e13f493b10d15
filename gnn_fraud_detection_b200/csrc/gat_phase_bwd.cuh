// Shared pieces of the dst-major backward kernels: saved row statistics, phase A (lane = edge: alpha recomputed
// from the saved statistics, LeakyReLU / dropout bits), the feature-free second sweep of long rows and the hub-row
// helper kernels.  Used by gat_bwd_dst.cu (projected-feature gathers) and gat_in_bwd.cu (input-space gathers).
#pragma once
#include "gat_stream.cuh"

namespace gnnfd {

// per-warp scratch beyond the ring: dal_s [32][H] floats + bits_s [2][32] ints
template <class GE>
constexpr int bwd_extra() { return 32 * GE::H * 4 + 2 * 32 * 4; }

template <int H>
struct RowStat {            // saved forward statistics of one destination row (all lanes identical)
    float adst[H], m[H], inv[H];
};
template <int H>
__device__ __forceinline__ void load_row_stat(RowStat<H>& r, int64_t i, const float* __restrict__ a_dst,
                                              const float* __restrict__ rowmax, const float* __restrict__ rowsum)
{
    float st[H];
    load_vecH<H>(a_dst + i * H, r.adst);
    load_vecH<H>(rowmax + i * H, r.m);
    load_vecH<H>(rowsum + i * H, st);
#pragma unroll
    for (int h = 0; h < H; ++h) r.inv[h] = 1.f / st[h];
}
// alpha of one (edge, head) from its logit z and the row's saved max m and 1/sum inv.  Every backward kernel forms alpha
// through this one expression, so that their alpha_used agree bit for bit.
__device__ __forceinline__ float edge_alpha(float z, float slope, float m, float inv)
{
    return expf((z > 0.f ? z : z * slope) - m) * inv;
}
struct BwdChunk {
    int row, beg, n;
    bool first, last;
};

// phase A: alpha (into p_s[buf]), source ids (j_s[buf]), slope/keep bits (bits_s[buf])
template <class GE, bool DROPOUT>
__device__ __forceinline__ void bwd_phase_a(const BwdChunk& c, const int32_t* __restrict__ col,
                                            const int32_t* __restrict__ perm, const float* __restrict__ a_src,
                                            const float* __restrict__ a_dst, const float* __restrict__ rowmax,
                                            const float* __restrict__ rowsum, float slope,
                                            KeepMask keep, float* p_s, int* j_s, int* bits_s, int lane)
{
    constexpr int H = GE::H;
    RowStat<H> r;
    load_row_stat<H>(r, c.row, a_dst, rowmax, rowsum);
    float alpha[H];
    int j = 0, bits = 0;
    if (lane < c.n) {
        j = col[c.beg + lane];
        float as[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float z = as[h] + r.adst[h];
            bits |= int(z > 0.f) << h;
            alpha[h] = edge_alpha(z, slope, r.m[h], r.inv[h]);
        }
        if (DROPOUT) {
            bits |= int(keep.bits(perm[c.beg + lane], H)) << 8;
        } else {
            bits |= 0xff00;
        }
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) alpha[h] = 0.f;
    }
    store_vecH<H>(p_s + lane * H, alpha);
    j_s[lane] = j;
    bits_s[lane] = bits;
    __syncwarp();
}

// phase B's head reduction: d[q] is this lane's partial dot product for head q*HP + lane/G; the full sums
// d_alpha[0..H) of the edge land in dal_t[0..H).
template <class GE>
__device__ __forceinline__ void dalpha_reduce(const float (&d)[GE::NS], float* dal_t, int lane)
{
    constexpr int NS = GE::NS, HP = GE::HP, G = GE::G;
    const int sub = lane / G;
    if constexpr (NS == 4 && G == 16) {
        // reduce-scatter butterfly over the 16-lane head group: 5 shuffles instead of 4 x 4.  After the
        // xor-8 / xor-4 steps a lane keeps only slot q = 2*bit3 + bit2; xor-2 / xor-1 finish its sum.
        const bool b3 = lane & 8, b2 = lane & 4;
        const float k0 = b3 ? d[2] : d[0], k1 = b3 ? d[3] : d[1];
        const float s0 = b3 ? d[0] : d[2], s1 = b3 ? d[1] : d[3];
        const float a0 = k0 + __shfl_xor_sync(FULL, s0, 8), a1 = k1 + __shfl_xor_sync(FULL, s1, 8);
        float b = (b2 ? a1 : a0) + __shfl_xor_sync(FULL, b2 ? a0 : a1, 4);
        b += __shfl_xor_sync(FULL, b, 2);
        b += __shfl_xor_sync(FULL, b, 1);
        if ((lane & 3) == 0) dal_t[((lane >> 2) & 3) * HP + sub] = b;
    } else {
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            float dq = d[q];
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) dq += __shfl_xor_sync(FULL, dq, o);
            if ((lane & (G - 1)) == 0) dal_t[q * HP + sub] = dq;
        }
    }
}

// second sweep of a long row: dz = slope * (u - alpha * t); returns the lane-local partial of da_dst
template <class GE>
__device__ __forceinline__ void dst_sweep2(const RowStat<GE::H>& r, int beg, int end, const int32_t* __restrict__ col,
                                           const int32_t* __restrict__ csr2csc, const float* __restrict__ a_src,
                                           float slope, const float (&t)[GE::H], int lane, float* __restrict__ dz,
                                           int64_t eg_ld, float (&dad)[GE::H])
{
    constexpr int H = GE::H;
    for (int e = beg + lane; e < end; e += 32) {
        float as[H], u[H], o[H];
        const int64_t pos = csr2csc[e];          // edge gradients live in source-major order
        load_vecH<H>(a_src + int64_t(col[e]) * H, as);
        load_vecH<H>(dz + pos * eg_ld, u);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float z = as[h] + r.adst[h];
            const float sl = z > 0.f ? 1.f : slope;
            const float al = expf(z * sl - r.m[h]) * r.inv[h];
            o[h] = sl * (u[h] - al * t[h]);
            dad[h] += o[h];
        }
        store_vecH<H>(dz + pos * eg_ld, o);
    }
}
// ---- packs of whole short rows (see ChunkCursor::next_any and the forward's gat_fwd_items_pack) ------------------
// phase A needs no scans here (the row statistics are saved), but each lane works with the statistics of ITS row;
// phase B switches the dO slice at the row boundaries inside the pack (the next row's slice is loaded one row
// ahead, and the pack's dO rows -- contiguous in memory -- are pulled into L2 during phase A); phase C finishes
// every row of the pack in registers with SEGMENTED warp sums.
// bits layout per staged edge: [0,8) LeakyReLU-positive, [8,16) dropout keep, [16,21) first lane of the row,
// [21,26) last lane of the row, bit 26 = this edge is the last of its row.
//
// The row of lane `lane`'s edge inside a pack of k rows starting at edge beg: its index lo in the pack and its first /
// last lane sa / sb (lanes l < k hold row l's edge range in lane_a / lane_b).
__device__ __forceinline__ void pack_lane_segment(int beg, int k, int lane_a, int lane_b, int lane, int& lo, int& sa, int& sb)
{
    const int e_id = beg + lane;
    int hi = k - 1;
    lo = 0;
#pragma unroll
    for (int it = 0; it < 5; ++it) {
        const int mid = (lo + hi) >> 1;
        const int bm = __shfl_sync(FULL, lane_b, mid);
        if (bm > e_id) hi = mid; else lo = min(mid + 1, k - 1);
    }
    sa = __shfl_sync(FULL, lane_a, lo) - beg;
    sb = __shfl_sync(FULL, lane_b, lo) - beg - 1;
}
template <class GE, bool CONCAT, bool DROPOUT>
__device__ __forceinline__ void bwd_phase_a_pack(int row0, int beg, int n, int k, int lane_a, int lane_b,
                                                 const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                                                 const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                 const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                                                 const float* __restrict__ d_out, float slope,
                                                 KeepMask keep, float* p_s, int* j_s, int* bits_s, int lane)
{
    constexpr int H = GE::H;
    const bool act = lane < n;
    const int e_id = beg + lane;
    int lo, sa, sb;
    pack_lane_segment(beg, k, lane_a, lane_b, lane, lo, sa, sb);
    if (!CONCAT) {
        // the pack's dO rows are one contiguous block of k*C floats
        const char* pb = reinterpret_cast<const char*>(d_out + int64_t(row0) * GE::C);
        const int nbytes = k * GE::C * 4;
        for (int off = lane * 128; off < nbytes; off += 32 * 128) prefetch_l2(pb + off);
    }
    float alpha[H];
    int j = 0, bits = 0;
    if (act) {
        const int64_t row = row0 + lo;
        RowStat<H> r;
        load_row_stat<H>(r, row, a_dst, rowmax, rowsum);
        j = col[e_id];
        float as[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float z = as[h] + r.adst[h];
            bits |= int(z > 0.f) << h;
            alpha[h] = edge_alpha(z, slope, r.m[h], r.inv[h]);
        }
        if (DROPOUT) {
            bits |= int(keep.bits(perm[e_id], H)) << 8;
        } else {
            bits |= 0xff00;
        }
        bits |= (sa << 16) | (sb << 21) | (int(lane == sb) << 26);
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) alpha[h] = 0.f;
    }
    store_vecH<H>(p_s + lane * H, alpha);
    j_s[lane] = j;
    bits_s[lane] = bits;
    __syncwarp();
}

// inclusive sum over the lanes [sa, lane] of the lane's segment; the row total sits in lane sb afterwards
__device__ __forceinline__ float seg_total(float v, int sa, int sb, int lane)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(FULL, v, o);
        if (lane - o >= sa) v += t;
    }
    return __shfl_sync(FULL, v, sb);
}
// hub rows, step 2: total t of the row (chunk order), second sweep, partial da_dst
template <class GE>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_dst_hub2(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                 const int32_t* __restrict__ csr2csc, const float* __restrict__ a_src,
                 const float* __restrict__ a_dst, const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                 gnnfd_hub_plan_t plan, float slope, const float* __restrict__ t_total, float* __restrict__ dz,
                 int64_t eg_ld, float* __restrict__ part_dad)
{
    constexpr int H = GE::H;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t i = plan.hub_row[slot];
    const int c0 = plan.hub_chunk_ptr[slot], c1 = plan.hub_chunk_ptr[slot + 1];
    const int beg = rowptr[i] + (c - c0) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    RowStat<H> r;
    load_row_stat<H>(r, i, a_dst, rowmax, rowsum);
    float t[H], dad[H];
    load_vecH<H>(t_total + int64_t(slot) * H, t);      // the same total in every chunk of the row
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = 0.f;
    (void)c1;
    dst_sweep2<GE>(r, beg, end, col, csr2csc, a_src, slope, t, lane, dz, eg_ld, dad);
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
    if (lane == 0) store_vecH<H>(part_dad + int64_t(c) * H, dad);
}
// per hub row: out[dst_index] = sum over its chunks of part[c][0..H) -- one warp per hub, lanes stride over the
// chunks, fixed-shape warp reduction => deterministic.  dst_index = hub slot (BY_ROW = false) or row id.
template <int H, bool BY_ROW>
__global__ void __launch_bounds__(ROW_THREADS)
gat_hub_chunk_sum(gnnfd_hub_plan_t plan, const float* __restrict__ part, float* __restrict__ out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * ROW_WARPS + warp;
    if (slot >= plan.n_hub) return;
    float s[H];
#pragma unroll
    for (int h = 0; h < H; ++h) s[h] = 0.f;
    for (int c = plan.hub_chunk_ptr[slot] + lane; c < plan.hub_chunk_ptr[slot + 1]; c += 32) {
        float p[H];
        load_vecH<H>(part + int64_t(c) * H, p);
#pragma unroll
        for (int h = 0; h < H; ++h) s[h] += p[h];
    }
#pragma unroll
    for (int h = 0; h < H; ++h) s[h] = warp_sum(s[h]);
    const int64_t o = BY_ROW ? int64_t(plan.hub_row[slot]) : int64_t(slot);
    if (lane == 0) store_vecH<H>(out + o * H, s);
}

}  // namespace gnnfd
