// (3) fused LeakyReLU + online segment softmax + alpha-weighted neighbour gather-sum (forward).
//
// Replaces edge_update + message + aggregate + head mean/concat + bias of PyG's GATConv.forward at the
// reference call sites src/models/gat.py:80 / src/models/tgn.py:94 (SURVEY.md 8(a2) steps E, A, O).
//
// One warp streams one edge-balanced work item (gat_stream.cuh).  Per chunk of <= 32 edges of a row:
//   phase A  lane = edge: gather the source logits (32 B), LeakyReLU, chunk max / sum by warp shuffles;
//            exp() is evaluated once per (edge, head), relative to the CHUNK max, and staged in shared
//            memory, so phase A needs no row state and can run one chunk ahead of the feature traffic;
//   phase B  the chunk's source rows arrive through the bulk-copy ring; per row one online-softmax
//            rescale (m, s, acc) by the chunk statistics, then per edge 4 conflict-free 128-bit shared
//            loads and 16 FMAs per lane.
// Rows longer than the hub threshold are split edge-balanced into chunks (one warp each) whose partial
// (m, s, acc) are merged in chunk order by the online-softmax combine rule -- deterministic.
#include "gat_stream.cuh"
#include "gat_phase_fwd.cuh"

#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;
// the source-major head-mean forward (gat_fwd_msg.cu)
bool gat_fwd_srcmajor_applies(const gnnfd_graph_t* g, int concat);
size_t gat_fwd_srcmajor_ws_bytes(const gnnfd_graph_t* g, int H, int C);
int gat_fwd_srcmajor(const gnnfd_graph_t* g, const void* xw, int xw_dtype, int H, int C, const float* a_src,
                     const float* a_dst, const EpiParams& ep, float negative_slope, const uint8_t* keep_mask, float p_drop,
                     uint64_t seed, float* out, float* rowmax, float* rowsum, void* ws, size_t ws_bytes, cudaStream_t st);

// normalise by the softmax denominator, save the row statistics, head mean/concat + bias + activation
template <class GE, bool CONCAT>
__device__ __forceinline__ void fwd_epilogue(int64_t i, const float (&m)[GE::H], const float (&s)[GE::H],
                                             float (&acc)[GE::NS][GE::VW], const EpiParams& ep,
                                             float* __restrict__ out, float* __restrict__ rowmax,
                                             float* __restrict__ rowsum, int lane, bool write_stats = true)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, HP = GE::HP, D = GE::D, C = GE::C, G = GE::G;
    const int sub = lane / G;
    float st[H], inv[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        st[h] = s[h] + 1e-16f;   // PyG softmax: out / (sum + 1e-16)
        inv[h] = 1.f / st[h];
    }
    if (lane == 0 && write_stats) {
        store_vecH<H>(rowmax + i * H, m);
        store_vecH<H>(rowsum + i * H, st);
    }
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const float f = pick<HP>(inv, q, sub);
#pragma unroll
        for (int k = 0; k < VW; ++k) acc[q][k] *= f;
    }
    if (CONCAT) {
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const int c0 = VW * (lane + 32 * q);
            float r[VW];
#pragma unroll
            for (int k = 0; k < VW; ++k) r[k] = epi_value(acc[q][k], c0 + k, i, D, ep);
#pragma unroll
            for (int k = 0; k < VW; k += 4)
                stg_stream(reinterpret_cast<float4*>(out + i * D + c0 + k), make_float4(r[k], r[k + 1], r[k + 2], r[k + 3]));
        }
    } else {
        float r[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            r[k] = 0.f;
#pragma unroll
            for (int q = 0; q < NS; ++q) r[k] += acc[q][k];
#pragma unroll
            for (int o = G; o < 32; o <<= 1) r[k] += __shfl_xor_sync(FULL, r[k], o);
        }
        if (sub == 0) {
            const int c0 = VW * lane;  // lane < G here
#pragma unroll
            for (int k = 0; k < VW; ++k) r[k] = epi_value(r[k] * (1.f / H), c0 + k, i, C, ep);   // 1/H: exact
#pragma unroll
            for (int k = 0; k < VW; k += 4)
                stg_stream(reinterpret_cast<float4*>(out + i * C + c0 + k), make_float4(r[k], r[k + 1], r[k + 2], r[k + 3]));
        }
    }
}


// What happens when a row (or a hub chunk) is complete.
template <class GE, bool CONCAT>
struct RowEpilogue {
    EpiParams ep; float* out; float* rowmax; float* rowsum;
    __device__ __forceinline__ void finish(int row, const float (&m)[GE::H], const float (&s)[GE::H],
                                           float (&acc)[GE::NS][GE::VW], int lane) const
    {
        fwd_epilogue<GE, CONCAT>(row, m, s, acc, ep, out, rowmax, rowsum, lane);
    }
    // rows of a pack: the weights were normalised in phase A (which also saved the row statistics)
    __device__ __forceinline__ void finish_norm(int row, float (&acc)[GE::NS][GE::VW], int lane) const
    {
        float m[GE::H], s[GE::H];
#pragma unroll
        for (int h = 0; h < GE::H; ++h) { m[h] = 0.f; s[h] = 1.f; }     // 1 + 1e-16 == 1 in fp32: no rescale
        fwd_epilogue<GE, CONCAT>(row, m, s, acc, ep, out, rowmax, rowsum, lane, /*write_stats=*/false);
    }
    __device__ __forceinline__ void empty(int row, int lane) const
    {
        float m[GE::H], s[GE::H], acc[GE::NS][GE::VW];
#pragma unroll
        for (int h = 0; h < GE::H; ++h) { m[h] = 0.f; s[h] = 0.f; }
#pragma unroll
        for (int q = 0; q < GE::NS; ++q)
#pragma unroll
            for (int k = 0; k < GE::VW; ++k) acc[q][k] = 0.f;
        fwd_epilogue<GE, CONCAT>(row, m, s, acc, ep, out, rowmax, rowsum, lane);
    }
};
template <class GE>
struct PartialSink {   // hub chunk: unnormalised partial (m, s, acc) of chunk c
    float* part_ms; float* part_acc; int c;
    __device__ __forceinline__ void finish(int, const float (&m)[GE::H], const float (&s)[GE::H],
                                           float (&acc)[GE::NS][GE::VW], int lane) const
    {
        if (lane == 0) {
            store_vecH<GE::H>(part_ms + int64_t(c) * 2 * GE::H, m);
            store_vecH<GE::H>(part_ms + int64_t(c) * 2 * GE::H + GE::H, s);
        }
#pragma unroll
        for (int q = 0; q < GE::NS; ++q)
#pragma unroll
            for (int k = 0; k < GE::VW; k += 4)
                *reinterpret_cast<float4*>(part_acc + int64_t(c) * GE::D + GE::VW * (lane + 32 * q) + k) =
                    make_float4(acc[q][k], acc[q][k + 1], acc[q][k + 2], acc[q][k + 3]);
    }
    __device__ __forceinline__ void empty(int, int) const {}
};

// The stream loop: phase A runs one chunk ahead of the ring consumption.
template <class GE, bool DROPOUT, class Sink>
__device__ __forceinline__ void fwd_stream(ChunkCursor& cur, WarpRing<GE>& ring, const Sink& sink,
                                           const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                           const int32_t* __restrict__ perm,
                                           const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                                           const float* __restrict__ a_dst, float slope,
                                           KeepMask keep, float keep_scale, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, HP = GE::HP;
    const int sub = lane / GE::G;
    auto on_empty = [&](int r) { sink.empty(r, lane); };
    ChunkStat<H> c0, c1;
    int b0 = 0;                         // staging buffer of the current chunk
    int beg;
    if (!cur.next(rowptr, c0.row, beg, c0.n, c0.first, c0.last, on_empty)) return;
    fwd_phase_a<GE, DROPOUT>(c0, beg, col, perm, a_src, a_dst, slope, keep, keep_scale, ring.p_s + b0 * 32 * H,
                             ring.j_s + b0 * 32, lane);
    int issued0 = 0, issued1 = 0;       // edges of the current / next chunk already handed to the copy engine
    float m[H], s[H], acc[NS][VW];
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        while (ring.has_room() && issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
        // phase A of the next chunk while the current chunk's rows are in flight
        const bool have1 = cur.next(rowptr, c1.row, beg, c1.n, c1.first, c1.last, on_empty);
        issued1 = 0;
        if (have1)
            fwd_phase_a<GE, DROPOUT>(c1, beg, col, perm, a_src, a_dst, slope, keep, keep_scale,
                                     ring.p_s + (b0 ^ 1) * 32 * H, ring.j_s + (b0 ^ 1) * 32, lane);
        // online-softmax combine of the running row state with this chunk
        if (c0.first) {
#pragma unroll
            for (int h = 0; h < H; ++h) { m[h] = -INFINITY; s[h] = 0.f; }
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int k = 0; k < VW; ++k) acc[q][k] = 0.f;
        }
        float fch[H];
        {
            float fold[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float mn = fmaxf(m[h], c0.cm[h]);
                fold[h] = expf(m[h] - mn);          // 0 on the first chunk (m = -inf)
                fch[h] = expf(c0.cm[h] - mn);
                s[h] = s[h] * fold[h] + c0.cs[h] * fch[h];
                m[h] = mn;
            }
            if (!c0.first) {
#pragma unroll
                for (int q = 0; q < NS; ++q) {
                    const float f = pick<HP>(fold, q, sub);
#pragma unroll
                    for (int k = 0; k < VW; ++k) acc[q][k] *= f;
                }
            }
        }
        float fq[NS];
#pragma unroll
        for (int q = 0; q < NS; ++q) fq[q] = pick<HP>(fch, q, sub);
        const float* p0 = ring.p_s + b0 * 32 * H;
        for (int t = 0; t < c0.n; ++t) {
            const uint8_t* row = ring.front();
            float v[NS][VW], wq[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                lds_slot(row, q, lane, v[q]);
                wq[q] = p0[t * H + q * HP + sub] * fq[q];
            }
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int k = 0; k < VW; ++k) acc[q][k] = fmaf(wq[q], v[q][k], acc[q][k]);
            ring.pop();
            // refill the freed slot: rest of this chunk first, then run ahead into the next one
            if (issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
            else if (have1 && issued1 < c1.n) ring.issue(xw, j1[issued1++], lane);
        }
        if (c0.last) sink.finish(c0.row, m, s, acc, lane);
        if (!have1) break;
        c0 = c1;
        issued0 = issued1;
        b0 ^= 1;
    }
}

template <class GE, bool CONCAT, bool DROPOUT>
__device__ __forceinline__ void fwd_stream_pack(ChunkCursor& cur, WarpRing<GE, 256>& ring, const RowEpilogue<GE, CONCAT>& sink,
                                                const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                const int32_t* __restrict__ perm,
                                                const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                                                const float* __restrict__ a_dst, float slope,
                                                KeepMask keep, float keep_scale, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, HP = GE::HP;
    const int sub = lane / GE::G;
    auto on_empty = [&](int r) { sink.empty(r, lane); };
    int* r_all = reinterpret_cast<int*>(ring.extra);            // [2][32] row id | last-edge flag per staged edge
    ChunkStat<H> c0, c1;
    int kind0 = 0, kind1 = 0;
    int b0 = 0, beg, k, la, lb;
    auto phase_a = [&](ChunkStat<H>& c, int kind, int buf) {
        if (kind == 2)
            fwd_phase_a_pack<GE, DROPOUT>(c.row, beg, c.n, k, la, lb, col, perm, a_src, a_dst, slope, keep, keep_scale,
                                          sink.rowmax, sink.rowsum, ring.p_s + buf * 32 * H, ring.j_s + buf * 32,
                                          r_all + buf * 32, lane);
        else
            fwd_phase_a<GE, DROPOUT>(c, beg, col, perm, a_src, a_dst, slope, keep, keep_scale, ring.p_s + buf * 32 * H,
                                     ring.j_s + buf * 32, lane);
    };
    kind0 = cur.next_any(rowptr, lane, c0.row, beg, c0.n, c0.first, c0.last, k, la, lb, on_empty);
    if (!kind0) return;
    phase_a(c0, kind0, b0);
    int issued0 = 0, issued1 = 0;
    float m[H], s[H], acc[NS][VW];
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        while (ring.has_room() && issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
        kind1 = cur.next_any(rowptr, lane, c1.row, beg, c1.n, c1.first, c1.last, k, la, lb, on_empty);
        issued1 = 0;
        if (kind1) phase_a(c1, kind1, b0 ^ 1);
        if (c0.first) {
#pragma unroll
            for (int h = 0; h < H; ++h) { m[h] = -INFINITY; s[h] = 0.f; }
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int kk = 0; kk < VW; ++kk) acc[q][kk] = 0.f;
        }
        float fq[NS];
        if (kind0 == 2) {
#pragma unroll
            for (int q = 0; q < NS; ++q) fq[q] = 1.f;
        } else {
            float fch[H], fold[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float mn = fmaxf(m[h], c0.cm[h]);
                fold[h] = expf(m[h] - mn);
                fch[h] = expf(c0.cm[h] - mn);
                s[h] = s[h] * fold[h] + c0.cs[h] * fch[h];
                m[h] = mn;
            }
            if (!c0.first) {
#pragma unroll
                for (int q = 0; q < NS; ++q) {
                    const float f = pick<HP>(fold, q, sub);
#pragma unroll
                    for (int kk = 0; kk < VW; ++kk) acc[q][kk] *= f;
                }
            }
#pragma unroll
            for (int q = 0; q < NS; ++q) fq[q] = pick<HP>(fch, q, sub);
        }
        const float* p0 = ring.p_s + b0 * 32 * H;
        const int* r0 = r_all + b0 * 32;
        for (int t = 0; t < c0.n; ++t) {
            const uint8_t* rowp = ring.front();
            float v[NS][VW], wq[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                lds_slot(rowp, q, lane, v[q]);
                wq[q] = p0[t * H + q * HP + sub] * fq[q];
            }
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int kk = 0; kk < VW; ++kk) acc[q][kk] = fmaf(wq[q], v[q][kk], acc[q][kk]);
            ring.pop();
            if (issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
            else if (kind1 && issued1 < c1.n) ring.issue(xw, j1[issued1++], lane);
            if (kind0 == 2) {
                const int rs = r0[t];
                if (rs < 0) {                                   // last edge of a packed row
                    sink.finish_norm(rs & 0x7fffffff, acc, lane);
#pragma unroll
                    for (int q = 0; q < NS; ++q)
#pragma unroll
                        for (int kk = 0; kk < VW; ++kk) acc[q][kk] = 0.f;
                }
            }
        }
        if (kind0 == 1 && c0.last) sink.finish(c0.row, m, s, acc, lane);
        if (!kind1) break;
        c0 = c1;
        kind0 = kind1;
        issued0 = issued1;
        b0 ^= 1;
    }
}

template <class GE, bool CONCAT, bool DROPOUT>
__global__ void __launch_bounds__(ST_THREADS, st_min_ctas<GE>())
gat_fwd_items_pack(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                   const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                   const float* __restrict__ a_dst, EpiParams ep, gnnfd_item_plan_t items,
                   int hub_threshold, float slope, KeepMask keep, float keep_scale,
                   float* __restrict__ out, float* __restrict__ rowmax, float* __restrict__ rowsum)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * ST_WARPS + warp;
    if (item >= items.n_items) return;
    WarpRing<GE, 256> ring;
    ring.init(smem + warp * StreamGeo<GE, 256>::WARP_BYTES, lane);
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    RowEpilogue<GE, CONCAT> sink{ep, out, rowmax, rowsum};
    fwd_stream_pack<GE, CONCAT, DROPOUT>(cur, ring, sink, rowptr, col, perm, xw, a_src, a_dst, slope, keep, keep_scale, lane);
}

// one warp per (hub row, chunk): partial (m, s, unnormalised acc)
template <class GE, bool DROPOUT>
__global__ void __launch_bounds__(ST_THREADS, st_min_ctas<GE>())
gat_fwd_hub_chunks(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                   const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                   const float* __restrict__ a_dst, gnnfd_hub_plan_t plan, float slope,
                   KeepMask keep, float keep_scale, float* __restrict__ part_ms,
                   float* __restrict__ part_acc)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ST_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    WarpRing<GE> ring;
    ring.init(smem + warp * StreamGeo<GE>::WARP_BYTES, lane);
    ChunkCursor cur;
    cur.start_segment(i, beg, end);
    PartialSink<GE> sink{part_ms, part_acc, c};
    fwd_stream<GE, DROPOUT>(cur, ring, sink, rowptr, col, perm, xw, a_src, a_dst, slope, keep, keep_scale, lane);
}

// one CTA per hub row: warp w folds chunks w, w+8, ... with the online-softmax combine rule, then the eight
// warp states are folded in warp order -- a fixed order, so the result is deterministic
template <class GE, bool CONCAT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_fwd_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part_ms, const float* __restrict__ part_acc,
                  EpiParams ep, float* __restrict__ out, float* __restrict__ rowmax, float* __restrict__ rowsum)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, HP = GE::HP, D = GE::D;
    __shared__ __align__(16) float st_ms[ROW_WARPS][2 * H];
    __shared__ __align__(16) float st_acc[ROW_WARPS][D];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int sub = lane / GE::G;
    const int64_t i = plan.hub_row[slot];
    const int c0 = plan.hub_chunk_ptr[slot], c1 = plan.hub_chunk_ptr[slot + 1];
    float M[H], s[H], acc[NS][VW];
#pragma unroll
    for (int h = 0; h < H; ++h) { M[h] = -INFINITY; s[h] = 0.f; }
#pragma unroll
    for (int q = 0; q < NS; ++q)
#pragma unroll
        for (int k = 0; k < VW; ++k) acc[q][k] = 0.f;
    auto fold = [&](const float (&mc)[H], const float (&sc)[H], const float* __restrict__ pacc) {
        float fo[H], fn[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float mn = fmaxf(M[h], mc[h]);
            fo[h] = (M[h] == -INFINITY) ? 0.f : expf(M[h] - mn);
            fn[h] = (mc[h] == -INFINITY) ? 0.f : expf(mc[h] - mn);
            s[h] = s[h] * fo[h] + sc[h] * fn[h];
            M[h] = mn;
        }
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const float a = pick<HP>(fo, q, sub), bq = pick<HP>(fn, q, sub);
#pragma unroll
            for (int k = 0; k < VW; k += 4) {
                const float4 v = *reinterpret_cast<const float4*>(pacc + VW * (lane + 32 * q) + k);
                acc[q][k] = fmaf(v.x, bq, acc[q][k] * a);
                acc[q][k + 1] = fmaf(v.y, bq, acc[q][k + 1] * a);
                acc[q][k + 2] = fmaf(v.z, bq, acc[q][k + 2] * a);
                acc[q][k + 3] = fmaf(v.w, bq, acc[q][k + 3] * a);
            }
        }
    };
    for (int c = c0 + warp; c < c1; c += ROW_WARPS) {
        float mc[H], sc[H];
        load_vecH<H>(part_ms + int64_t(c) * 2 * H, mc);
        load_vecH<H>(part_ms + int64_t(c) * 2 * H + H, sc);
        fold(mc, sc, part_acc + int64_t(c) * D);
    }
    if (lane == 0) {
        store_vecH<H>(&st_ms[warp][0], M);
        store_vecH<H>(&st_ms[warp][H], s);
    }
#pragma unroll
    for (int q = 0; q < NS; ++q)
#pragma unroll
        for (int k = 0; k < VW; k += 4)
            *reinterpret_cast<float4*>(&st_acc[warp][VW * (lane + 32 * q) + k]) =
                make_float4(acc[q][k], acc[q][k + 1], acc[q][k + 2], acc[q][k + 3]);
    __syncthreads();
    if (warp != 0) return;
    for (int w = 1; w < ROW_WARPS; ++w) {
        float mc[H], sc[H];
#pragma unroll
        for (int h = 0; h < H; ++h) { mc[h] = st_ms[w][h]; sc[h] = st_ms[w][H + h]; }
        fold(mc, sc, &st_acc[w][0]);
    }
    fwd_epilogue<GE, CONCAT>(i, M, s, acc, ep, out, rowmax, rowsum, lane);
}

// alpha[e,h] in CSR order from the saved row statistics; warp per row, lane = edge
template <int H>
__global__ void __launch_bounds__(ROW_THREADS)
gat_alpha_rows(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
               const float* __restrict__ a_dst, const float* __restrict__ rowmax, const float* __restrict__ rowsum,
               int64_t n_dst, float slope, float* __restrict__ alpha)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = int64_t(blockIdx.x) * ROW_WARPS + warp;
    if (i >= n_dst) return;
    const int beg = rowptr[i], end = rowptr[i + 1];
    float adst[H], m[H], st[H];
    load_vecH<H>(a_dst + i * H, adst);
    load_vecH<H>(rowmax + i * H, m);
    load_vecH<H>(rowsum + i * H, st);
    for (int e = beg + lane; e < end; e += 32) {
        float as[H], al[H];
        load_vecH<H>(a_src + int64_t(col[e]) * H, as);
#pragma unroll
        for (int h = 0; h < H; ++h) al[h] = expf(leaky(as[h] + adst[h], slope) - m[h]) / st[h];
        store_vecH<H>(alpha + int64_t(e) * H, al);
    }
}

template <class K>
static int set_smem(K kernel, int bytes)
{
    GNNFD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return GNNFD_OK;
}

template <class GE>
static int launch_fwd(const gnnfd_graph_t* g, const void* xw_, const float* a_src, const float* a_dst,
                      EpiParams ep, float slope, int concat, const uint8_t* keep_mask, float p_drop, uint64_t seed,
                      float* out, float* rowmax, float* rowsum, void* ws, size_t ws_bytes, cudaStream_t st)
{
    using XT = typename GE::XT;
    constexpr int SMEM = StreamGeo<GE>::CTA_BYTES;
    const XT* xw = reinterpret_cast<const XT*>(xw_);
    const int64_t n = g->n_dst;
    if (n == 0) return GNNFD_OK;
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG,
                  "gat_fwd: the graph has no work-item plan over rowptr (gnnfd_item_plan)");
    const bool drop = p_drop > 0.f;              // explicit mask, or (mask == NULL) the counter-based RNG keyed on seed
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + ST_WARPS - 1) / ST_WARPS);
    int rc = GNNFD_OK;
    // packs of whole short rows share one phase A: 2.2x on the Elliptic-size graph (2 edges per row), and still 11 %
    // on the 200M-edge power-law graph, whose rows are mostly short, against a kernel that streams row by row
    constexpr int SMEM_P = StreamGeo<GE, 256>::CTA_BYTES;
#define GNNFD_FWD_ITEMS_PACK(CC, DD)                                                                                  \
    rc = set_smem(gat_fwd_items_pack<GE, CC, DD>, SMEM_P);                                                            \
    if (rc) return rc;                                                                                                \
    gat_fwd_items_pack<GE, CC, DD><<<grid, ST_THREADS, SMEM_P, st>>>(g->rowptr, g->col, g->perm, xw, a_src, a_dst, ep, \
                                                                     g->items_dst, thr, slope, keep, ks, out, rowmax, rowsum)
    if (concat) { if (drop) { GNNFD_FWD_ITEMS_PACK(true, true); } else { GNNFD_FWD_ITEMS_PACK(true, false); } }
    else        { if (drop) { GNNFD_FWD_ITEMS_PACK(false, true); } else { GNNFD_FWD_ITEMS_PACK(false, false); } }
#undef GNNFD_FWD_ITEMS_PACK
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const size_t need = carve_bytes(size_t(pl.n_chunk) * 2 * GE::H, 4) + carve_bytes(size_t(pl.n_chunk) * GE::D, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_fwd: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        float* part_ms = carve<float>(p, size_t(pl.n_chunk) * 2 * GE::H);
        float* part_acc = carve<float>(p, size_t(pl.n_chunk) * GE::D);
        const unsigned gc = (unsigned)((pl.n_chunk + ST_WARPS - 1) / ST_WARPS);
        const unsigned gh = (unsigned)pl.n_hub;   // one CTA per hub row
        if (drop) {
            rc = set_smem(gat_fwd_hub_chunks<GE, true>, SMEM);
            if (rc) return rc;
            gat_fwd_hub_chunks<GE, true><<<gc, ST_THREADS, SMEM, st>>>(g->rowptr, g->col, g->perm, xw, a_src, a_dst, pl,
                                                                       slope, keep, ks, part_ms, part_acc);
        } else {
            rc = set_smem(gat_fwd_hub_chunks<GE, false>, SMEM);
            if (rc) return rc;
            gat_fwd_hub_chunks<GE, false><<<gc, ST_THREADS, SMEM, st>>>(g->rowptr, g->col, g->perm, xw, a_src, a_dst, pl,
                                                                        slope, keep, ks, part_ms, part_acc);
        }
        if (concat)
            gat_fwd_hub_merge<GE, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_ms, part_acc, ep, out, rowmax, rowsum);
        else
            gat_fwd_hub_merge<GE, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_ms, part_acc, ep, out, rowmax, rowsum);
        g_launches += 2;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who)
{
    GNNFD_REQUIRE(g != nullptr, GNNFD_ERR_ARG, "%s: graph is NULL", who);
    GNNFD_REQUIRE(g->n_dst >= 0 && g->n_src >= 0 && g->n_edges >= 0, GNNFD_ERR_ARG, "%s: negative graph size", who);
    GNNFD_REQUIRE(g->n_dst == 0 || g->rowptr, GNNFD_ERR_ARG, "%s: rowptr is NULL", who);
    GNNFD_REQUIRE(g->n_edges == 0 || (g->col && g->perm), GNNFD_ERR_ARG, "%s: col/perm is NULL", who);
    if (need_csc)
        GNNFD_REQUIRE(g->n_src == 0 || (g->colptr && (g->n_edges == 0 || (g->csc_row && g->csc_eid))), GNNFD_ERR_ARG,
                      "%s: the CSC twin (colptr/csc_row/csc_eid) is required", who);
    return GNNFD_OK;
}


// the keep bits of the counter-based attention-dropout RNG, written out as a [E',H] uint8 mask in edge_index' order
// (test / debugging hook: the kernels themselves never materialise it)
__global__ void dropout_mask_kernel(KeepMask km, int64_t n_edges, int H, uint8_t* __restrict__ out)
{
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < n_edges; e += int64_t(gridDim.x) * blockDim.x) {
        const unsigned b = km.bits(e, H);
        for (int h = 0; h < H; ++h) out[e * H + h] = uint8_t((b >> h) & 1u);
    }
}

}  // namespace gnnfd

using namespace gnnfd;

extern "C" {

int gnnfd_dropout_mask(uint64_t dropout_seed, float p_drop, int64_t n_edges, int H, uint8_t* keep_mask, float* scale_host,
                       gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(p_drop > 0.f && p_drop < 1.f && H >= 1 && H <= 8 && n_edges >= 0, GNNFD_ERR_ARG, "dropout_mask: bad argument");
    float ks = 1.f;
    const KeepMask km = make_keep(nullptr, p_drop, dropout_seed, &ks);
    if (scale_host) *scale_host = ks;
    if (n_edges == 0) return GNNFD_OK;
    GNNFD_REQUIRE(keep_mask, GNNFD_ERR_ARG, "dropout_mask: keep_mask is NULL");
    int64_t blocks = (n_edges + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    dropout_mask_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(km, n_edges, H, keep_mask);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int gnnfd_gat_fwd_workspace_bytes(const gnnfd_graph_t* g, int H, int C, size_t* bytes)
{
    GNNFD_REQUIRE(g && bytes, GNNFD_ERR_ARG, "gat_fwd_workspace_bytes: NULL argument");
    const size_t nc = (size_t)g->hub_dst.n_chunk;
    *bytes = carve_bytes(nc * 2 * H, 4) + carve_bytes(nc * size_t(H) * C, 4) + 256;
    // the source-major head-mean form also keeps alpha_used [E',H] and the messages [E',C] here; concat is not known
    if (gat_fwd_srcmajor_applies(g, 0)) *bytes += gat_fwd_srcmajor_ws_bytes(g, H, C);
    return GNNFD_OK;
}

int gnnfd_gat_fwd_fused(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src, const float* a_dst,
                        const float* bias, int H, int C, float negative_slope, int concat, int act,
                        const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, const float* post_scale, const float* post_shift,
                        const float* residual, float* out, float* rowmax, float* rowsum, void* ws, size_t ws_bytes,
                        gnnfd_stream_t stream)
{
    int rc = check_graph(g, false, "gat_fwd");
    if (rc) return rc;
    GNNFD_REQUIRE(g->n_dst == 0 || (xw && a_src && a_dst && out && rowmax && rowsum), GNNFD_ERR_ARG,
                  "gat_fwd: NULL tensor");
    GNNFD_REQUIRE(p_drop >= 0.f && p_drop < 1.f, GNNFD_ERR_ARG, "gat_fwd: dropout p must be in [0,1)");
    GNNFD_REQUIRE(p_drop == 0.f || g->n_edges == 0 || g->perm, GNNFD_ERR_ARG, "gat_fwd: attention dropout needs perm");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(xw) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                  GNNFD_ERR_ARG, "gat_fwd: xw/out must be 16-byte aligned");
    GNNFD_REQUIRE((post_scale == nullptr) == (post_shift == nullptr), GNNFD_ERR_ARG,
                  "gat_fwd: post_scale and post_shift must be given together");
    cudaStream_t st = (cudaStream_t)stream;
    const EpiParams ep{bias, post_scale, post_shift, residual, act};
    if (gat_fwd_srcmajor_applies(g, concat))
        return gat_fwd_srcmajor(g, xw, xw_dtype, H, C, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, dropout_seed, out,
                                rowmax, rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_F32)
        return launch_fwd<Geo<8, 64, float>>(g, xw, a_src, a_dst, ep, negative_slope, concat, keep_mask, p_drop, dropout_seed, out, rowmax,
                                             rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_BF16)
        return launch_fwd<Geo<8, 64, __nv_bfloat16>>(g, xw, a_src, a_dst, ep, negative_slope, concat, keep_mask, p_drop, dropout_seed, out,
                                                     rowmax, rowsum, ws, ws_bytes, st);
    if (H == 4 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_fwd<Geo<4, 32, float>>(g, xw, a_src, a_dst, ep, negative_slope, concat, keep_mask, p_drop, dropout_seed, out, rowmax,
                                             rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_fwd<Geo<8, 32, float>>(g, xw, a_src, a_dst, ep, negative_slope, concat, keep_mask, p_drop, dropout_seed, out, rowmax,
                                             rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 128 && xw_dtype == GNNFD_F32)
        return launch_fwd<Geo<8, 128, float>>(g, xw, a_src, a_dst, ep, negative_slope, concat, keep_mask, p_drop, dropout_seed, out,
                                              rowmax, rowsum, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_fwd: (heads=%d, out_channels=%d, dtype=%d) is not built; "
                  "available: (8,64,f32), (8,64,bf16), (8,32,f32), (8,128,f32), (4,32,f32)", H, C, xw_dtype);
    return GNNFD_ERR_UNSUPPORTED;
}

int gnnfd_gat_fwd(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src, const float* a_dst,
                  const float* bias, int H, int C, float negative_slope, int concat, int act,
                  const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, float* out, float* rowmax, float* rowsum, void* ws,
                  size_t ws_bytes, gnnfd_stream_t stream)
{
    return gnnfd_gat_fwd_fused(g, xw, xw_dtype, a_src, a_dst, bias, H, C, negative_slope, concat, act, keep_mask, p_drop, dropout_seed,
                               nullptr, nullptr, nullptr, out, rowmax, rowsum, ws, ws_bytes, stream);
}

int gnnfd_gat_alpha(const gnnfd_graph_t* g, const float* a_src, const float* a_dst, const float* rowmax,
                    const float* rowsum, int H, float negative_slope, float* alpha, gnnfd_stream_t stream)
{
    int rc = check_graph(g, false, "gat_alpha");
    if (rc) return rc;
    if (g->n_dst == 0 || g->n_edges == 0) return GNNFD_OK;
    GNNFD_REQUIRE(a_src && a_dst && rowmax && rowsum && alpha, GNNFD_ERR_ARG, "gat_alpha: NULL tensor");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((g->n_dst + ROW_WARPS - 1) / ROW_WARPS);
    if (H == 8)
        gat_alpha_rows<8><<<grid, ROW_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, rowmax, rowsum, g->n_dst,
                                                        negative_slope, alpha);
    else if (H == 4)
        gat_alpha_rows<4><<<grid, ROW_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, rowmax, rowsum, g->n_dst,
                                                        negative_slope, alpha);
    else
        GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_alpha: heads=%d is not built", H);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // extern "C"
