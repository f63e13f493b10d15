// Phase A of the forward message-passing kernels (lane = edge): logits, LeakyReLU, chunk / segmented softmax
// statistics and the staged per-edge weights.  Shared by the projected-feature kernels (gat_fwd.cu) and the
// input-space kernels (gat_in_fwd.cu); only GE::H is used.
#pragma once
#include "gat_stream.cuh"

namespace gnnfd {

// Fused row epilogue:  v = mean/concat + bias;  v = v*scale + shift (folded eval-mode BatchNorm, optional);
// v = act(v);  v += residual[row] (optional).  Mirrors gat.py:80-91 in eval mode (BatchNorm -> ReLU -> residual).
struct EpiParams {
    const float* bias;
    const float* scale;
    const float* shift;
    const float* residual;
    int act;
};

__device__ __forceinline__ float apply_act(float v, int act)
{
    if (act == GNNFD_ACT_RELU) return fmaxf(v, 0.f);
    if (act == GNNFD_ACT_ELU) return v > 0.f ? v : expm1f(v);
    return v;
}
// the epilogue of output channel c of row i (ld = output row length), v = the head mean / concat value
__device__ __forceinline__ float epi_value(float v, int c, int64_t i, int ld, const EpiParams& ep)
{
    v = v + (ep.bias ? ep.bias[c] : 0.f);
    if (ep.scale) v = fmaf(v, ep.scale[c], ep.shift[c]);
    v = apply_act(v, ep.act);
    if (ep.residual) v += ep.residual[i * ld + c];
    return v;
}

// statistics of one chunk, relative to its own maximum (all lanes hold the same values)
template <int H>
struct ChunkStat {
    int row, n;
    bool first, last;
    float cm[H], cs[H];
};

// phase A of one chunk: writes the per-edge weights exp(e - cm) (x dropout scale) and the source ids into
// staging buffer `buf`
template <class GE, bool DROPOUT>
__device__ __forceinline__ void fwd_phase_a(ChunkStat<GE::H>& c, int beg, const int32_t* __restrict__ col,
                                            const int32_t* __restrict__ perm, const float* __restrict__ a_src,
                                            const float* __restrict__ a_dst, float slope,
                                            KeepMask keep, float keep_scale, float* p_s, int* j_s,
                                            int lane)
{
    constexpr int H = GE::H;
    float e[H], kp[H], adst[H];
    load_vecH<H>(a_dst + int64_t(c.row) * H, adst);
    int j = 0;
    if (lane < c.n) {
        j = col[beg + lane];
        float as[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
#pragma unroll
        for (int h = 0; h < H; ++h) e[h] = leaky(as[h] + adst[h], slope);
        if (DROPOUT) {
            const unsigned kbits = keep.bits(perm[beg + lane], H);
#pragma unroll
            for (int h = 0; h < H; ++h) kp[h] = (kbits >> h) & 1u ? keep_scale : 0.f;
        }
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) { e[h] = -INFINITY; kp[h] = 0.f; }
    }
    float w[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        c.cm[h] = warp_max(e[h]);
        const float p = (lane < c.n) ? expf(e[h] - c.cm[h]) : 0.f;
        c.cs[h] = warp_sum(p);
        w[h] = DROPOUT ? p * kp[h] : p;
    }
    store_vecH<H>(p_s + lane * H, w);
    j_s[lane] = j;
    __syncwarp();
}
// ---- low-degree graphs: packs of whole rows share one phase A ---------------------------------------------------
// lane = edge of the pack; the lane's row is found by a 5-step search over the rows' end offsets, softmax max / sum
// are SEGMENTED warp scans over the lanes of one row, the weights are stored already normalised (so phase B needs no
// per-row state) and the lane holding a row's last edge writes the row statistics for the backward.
template <class GE, bool DROPOUT>
__device__ __forceinline__ void fwd_phase_a_pack(int row0, int beg, int n, int k, int lane_a, int lane_b,
                                                 const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                                                 const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                 float slope, KeepMask keep, float keep_scale,
                                                 float* __restrict__ rowmax, float* __restrict__ rowsum, float* p_s,
                                                 int* j_s, int* r_s, int lane)
{
    constexpr int H = GE::H;
    const bool act = lane < n;
    const int e_id = beg + lane;
    int lo = 0, hi = k - 1;
#pragma unroll
    for (int it = 0; it < 5; ++it) {                    // smallest i with end_i > e_id
        const int mid = (lo + hi) >> 1;
        const int bm = __shfl_sync(FULL, lane_b, mid);
        if (bm > e_id) hi = mid; else lo = min(mid + 1, k - 1);
    }
    const int i = lo;
    const int sa = __shfl_sync(FULL, lane_a, i) - beg;          // first / last lane of this lane's row
    const int sb = __shfl_sync(FULL, lane_b, i) - beg - 1;
    const int row = row0 + i;
    float e[H], kp[H];
    int j = 0;
    if (act) {
        j = col[e_id];
        float as[H], adst[H];
        load_vecH<H>(a_src + int64_t(j) * H, as);
        load_vecH<H>(a_dst + int64_t(row) * H, adst);
#pragma unroll
        for (int h = 0; h < H; ++h) e[h] = leaky(as[h] + adst[h], slope);
        if (DROPOUT) {
            const unsigned kbits = keep.bits(perm[e_id], H);
#pragma unroll
            for (int h = 0; h < H; ++h) kp[h] = (kbits >> h) & 1u ? keep_scale : 0.f;
        }
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) { e[h] = -INFINITY; kp[h] = 0.f; }
    }
    float w[H], mrow[H], srow[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        float mx = e[h];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float t = __shfl_up_sync(FULL, mx, o);
            if (lane - o >= sa) mx = fmaxf(mx, t);
        }
        mrow[h] = __shfl_sync(FULL, mx, sb);
        const float p = act ? expf(e[h] - mrow[h]) : 0.f;
        float sm = p;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float t = __shfl_up_sync(FULL, sm, o);
            if (lane - o >= sa) sm += t;
        }
        srow[h] = __shfl_sync(FULL, sm, sb) + 1e-16f;           // PyG softmax: out / (sum + 1e-16)
        const float pn = p / srow[h];
        w[h] = DROPOUT ? pn * kp[h] : pn;
    }
    if (act && lane == sb) {
        store_vecH<H>(rowmax + int64_t(row) * H, mrow);
        store_vecH<H>(rowsum + int64_t(row) * H, srow);
    }
    store_vecH<H>(p_s + lane * H, w);
    j_s[lane] = j;
    r_s[lane] = act ? (row | (lane == sb ? int(0x80000000u) : 0)) : 0;
    __syncwarp();
}

}  // namespace gnnfd
