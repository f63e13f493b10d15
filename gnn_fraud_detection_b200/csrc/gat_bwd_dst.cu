// (4a) backward, dst-major pass (autograd mirror of GATConv.forward's edge_update/aggregate, triggered by
// loss.backward() at src/train.py:142; closed forms in SURVEY.md 8(a3)).
//
// For the head mean on a graph with direct edge-gradient slots, gnnfd_gat_bwd_dst runs the two-pass form of
// gat_bwd_dalpha.cu (d_alpha source-major, then a dst pass that reads no features).  The kernels below are the
// single-pass gather form, used for concat, for the multi-GPU receive layout and for the destination-range row view.
//
// Same warp-stream structure as the forward (gat_stream.cuh): one warp per edge-balanced work item, the
// 2 KB source rows arrive through the bulk-copy ring.  Per chunk of <= 32 edges:
//   phase A  lane = edge: recompute alpha from the saved row statistics, remember the LeakyReLU slope and
//            dropout bits; runs one chunk ahead of the feature traffic;
//   phase B  per staged source row: d_alpha[e,h] = <dO_h[i], xw[j]> -- 16 FMAs per lane then a 16-lane
//            butterfly per head slot;
//   phase C  lane = edge: u = alpha * d_alpha; rows that fit one chunk finish in registers
//            (t = sum u, dz = slope * (u - alpha t)); longer rows park u in the dz buffer and make a
//            second, feature-free sweep once t is known; hub rows are split into chunks whose partial t /
//            da_dst are merged in chunk order -- deterministic.
// Writes alpha_used [E',H] and dz [E',H] in SOURCE-MAJOR order (slot csr2csc[e] for dst-sorted edge e), so the
// src-major pass -- and across GPUs the exchange to the source owners -- reads them contiguously; and
// da_dst [n_dst,H].
#include "gat_stream.cuh"
#include "gat_phase_bwd.cuh"

#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;
int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who);
bool gat_bwd_dst_srcmajor_applies(const gnnfd_graph_t* g, int concat);       // gat_bwd_dalpha.cu
int gat_bwd_dst_srcmajor(const gnnfd_graph_t* g, const void* xw, int xw_dtype, int H, int C, const float* a_src,
                         const float* a_dst, const float* rowmax, const float* rowsum, const float* d_out,
                         float negative_slope, const uint8_t* keep_mask, float p_drop, uint64_t seed, float* alpha_used,
                         float* dz, float* da_dst, void* ws, size_t ws_bytes, cudaStream_t st);


// dO_h slice owned by this lane (already divided by H for the head mean)
template <class GE, bool CONCAT>
__device__ __forceinline__ void load_g(float (&g)[GE::NS][GE::VW], int64_t i, const float* __restrict__ d_out, int lane)
{
    constexpr int NS = GE::NS, VW = GE::VW, C = GE::C, D = GE::D, H = GE::H;
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const int e0 = VW * (lane + 32 * q);
        const float* p = CONCAT ? d_out + i * D + e0 : d_out + i * C + (e0 % C);
#pragma unroll
        for (int k = 0; k < VW; k += 4) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(p + k));
            const float sc = CONCAT ? 1.f : 1.f / H;
            g[q][k] = t.x * sc; g[q][k + 1] = t.y * sc; g[q][k + 2] = t.z * sc; g[q][k + 3] = t.w * sc;
        }
    }
}


// One (hub row, range) segment: the partial t of the segment goes to part_t[chunk_id]; the second sweep is a
// separate kernel once every chunk's t is known.
template <class GE, bool CONCAT, bool DROPOUT>
__device__ __forceinline__ void bwd_dst_stream(ChunkCursor& cur, WarpRing<GE, bwd_extra<GE>()>& ring,
                                               const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                               const int32_t* __restrict__ perm, const int32_t* __restrict__ csr2csc,
                                               const typename GE::XT* __restrict__ xw,
                                               const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                               const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                                               const float* __restrict__ d_out, float slope,
                                               KeepMask keep, float keep_scale,
                                               float* __restrict__ alpha_used, float* __restrict__ dz, int64_t eg_ld,
                                               float* __restrict__ part_t, int chunk_id, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW;
    float* dal_s = reinterpret_cast<float*>(ring.extra);
    int* bits_s = reinterpret_cast<int*>(ring.extra + 32 * H * 4);
    auto on_empty = [](int) {};
    BwdChunk c0, c1;
    int b0 = 0;
    if (!cur.next(rowptr, c0.row, c0.beg, c0.n, c0.first, c0.last, on_empty)) return;
    bwd_phase_a<GE, DROPOUT>(c0, col, perm, a_src, a_dst, rowmax, rowsum, slope, keep, ring.p_s + b0 * 32 * H,
                             ring.j_s + b0 * 32, bits_s + b0 * 32, lane);
    float g0[NS][VW], g1[NS][VW];
    load_g<GE, CONCAT>(g0, c0.row, d_out, lane);
    int issued0 = 0, issued1 = 0;
    float trow[H];               // running t = sum alpha*d_alpha of the segment
#pragma unroll
    for (int h = 0; h < H; ++h) trow[h] = 0.f;
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        while (ring.has_room() && issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
        const bool have1 = cur.next(rowptr, c1.row, c1.beg, c1.n, c1.first, c1.last, on_empty);
        issued1 = 0;
        if (have1) {
            bwd_phase_a<GE, DROPOUT>(c1, col, perm, a_src, a_dst, rowmax, rowsum, slope, keep,
                                     ring.p_s + (b0 ^ 1) * 32 * H, ring.j_s + (b0 ^ 1) * 32, bits_s + (b0 ^ 1) * 32, lane);
            if (c1.first) load_g<GE, CONCAT>(g1, c1.row, d_out, lane);
        }
        if (c0.first) {
#pragma unroll
            for (int h = 0; h < H; ++h) trow[h] = 0.f;
        }
        // phase B: dot products of the staged rows with this row's dO slice
        for (int t = 0; t < c0.n; ++t) {
            const uint8_t* row = ring.front();
            float v[NS][VW];
#pragma unroll
            for (int q = 0; q < NS; ++q) lds_slot(row, q, lane, v[q]);
            float d[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                d[q] = 0.f;
#pragma unroll
                for (int k = 0; k < VW; ++k) d[q] = fmaf(g0[q][k], v[q][k], d[q]);
            }
            dalpha_reduce<GE>(d, dal_s + t * H, lane);
            ring.pop();
            if (issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
            else if (have1 && issued1 < c1.n) ring.issue(xw, j1[issued1++], lane);
        }
        __syncwarp();
        // phase C: lane = edge
        {
            float alpha[H], dal[H], u[H], au[H];
            const float* p0 = ring.p_s + b0 * 32 * H;
            const int bits = bits_s[b0 * 32 + lane];
#pragma unroll
            for (int k = 0; k < H / 4; ++k) {
                const float4 a4 = *reinterpret_cast<const float4*>(p0 + lane * H + 4 * k);
                const float4 d4 = *reinterpret_cast<const float4*>(dal_s + lane * H + 4 * k);
                alpha[4 * k] = a4.x; alpha[4 * k + 1] = a4.y; alpha[4 * k + 2] = a4.z; alpha[4 * k + 3] = a4.w;
                dal[4 * k] = d4.x; dal[4 * k + 1] = d4.y; dal[4 * k + 2] = d4.z; dal[4 * k + 3] = d4.w;
            }
            const bool live = lane < c0.n;
            const int64_t pos = live ? csr2csc[c0.beg + lane] : 0;    // source-major slot of this edge
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float ks = (bits >> (8 + h)) & 1 ? keep_scale : 0.f;
                u[h] = live ? alpha[h] * dal[h] * ks : 0.f;
                au[h] = alpha[h] * ks;
            }
            if (live) {
                store_vecH<H>(alpha_used + pos * eg_ld, au);
                store_vecH<H>(dz + pos * eg_ld, u);       // parked until t is known
            }
#pragma unroll
            for (int h = 0; h < H; ++h) trow[h] += warp_sum(u[h]);
            if (c0.last && lane == 0) store_vecH<H>(part_t + int64_t(chunk_id) * H, trow);
        }
        __syncwarp();
        if (!have1) break;
        if (c1.first) {
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int k = 0; k < VW; ++k) g0[q][k] = g1[q][k];
        }
        c0 = c1;
        issued0 = issued1;
        b0 ^= 1;
    }
}

template <class GE, bool CONCAT, bool DROPOUT>
__device__ __forceinline__ void bwd_dst_stream_pack(ChunkCursor& cur, WarpRing<GE, bwd_extra<GE>()>& ring,
                                                    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                    const int32_t* __restrict__ perm, const int32_t* __restrict__ csr2csc,
                                                    const typename GE::XT* __restrict__ xw,
                                                    const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                    const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                                                    const float* __restrict__ d_out, float slope,
                                                    KeepMask keep, float keep_scale,
                                                    float* __restrict__ alpha_used, float* __restrict__ dz, int64_t eg_ld,
                                                    float* __restrict__ da_dst, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW;
    float* dal_s = reinterpret_cast<float*>(ring.extra);
    int* bits_s = reinterpret_cast<int*>(ring.extra + 32 * H * 4);
    auto on_empty = [&](int r) {
        if (lane < H) da_dst[int64_t(r) * H + lane] = 0.f;
    };
    BwdChunk c0, c1;
    int kind0 = 0, kind1 = 0, k0 = 0, k1 = 0, la = 0, lb = 0;
    int b0 = 0;
    auto phase_a = [&](const BwdChunk& c, int kind, int kk, int buf) {
        if (kind == 2)
            bwd_phase_a_pack<GE, CONCAT, DROPOUT>(c.row, c.beg, c.n, kk, la, lb, col, perm, a_src, a_dst, rowmax, rowsum, d_out,
                                                  slope, keep, ring.p_s + buf * 32 * H, ring.j_s + buf * 32, bits_s + buf * 32, lane);
        else
            bwd_phase_a<GE, DROPOUT>(c, col, perm, a_src, a_dst, rowmax, rowsum, slope, keep, ring.p_s + buf * 32 * H,
                                     ring.j_s + buf * 32, bits_s + buf * 32, lane);
    };
    kind0 = cur.next_any(rowptr, lane, c0.row, c0.beg, c0.n, c0.first, c0.last, k0, la, lb, on_empty);
    if (!kind0) return;
    phase_a(c0, kind0, k0, b0);
    float g0[NS][VW], g1[NS][VW];
    load_g<GE, CONCAT>(g0, c0.row, d_out, lane);
    int issued0 = 0, issued1 = 0;
    float trow[H];
    int row_beg = c0.beg;
#pragma unroll
    for (int h = 0; h < H; ++h) trow[h] = 0.f;
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        while (ring.has_room() && issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
        kind1 = cur.next_any(rowptr, lane, c1.row, c1.beg, c1.n, c1.first, c1.last, k1, la, lb, on_empty);
        issued1 = 0;
        if (kind1) phase_a(c1, kind1, k1, b0 ^ 1);
        // g1 = dO slice of the NEXT row in stream order: the second row of this pack, else the next chunk's row
        if (kind0 == 2) load_g<GE, CONCAT>(g1, c0.row + 1, d_out, lane);
        else if (kind1 && c1.first) load_g<GE, CONCAT>(g1, c1.row, d_out, lane);
        if (c0.first) {
            row_beg = c0.beg;
#pragma unroll
            for (int h = 0; h < H; ++h) trow[h] = 0.f;
        }
        int rows_done = 0;
        const int* bits0 = bits_s + b0 * 32;
        for (int t = 0; t < c0.n; ++t) {
            const uint8_t* row = ring.front();
            float v[NS][VW];
#pragma unroll
            for (int q = 0; q < NS; ++q) lds_slot(row, q, lane, v[q]);
            float d[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                d[q] = 0.f;
#pragma unroll
                for (int kk = 0; kk < VW; ++kk) d[q] = fmaf(g0[q][kk], v[q][kk], d[q]);
            }
            dalpha_reduce<GE>(d, dal_s + t * H, lane);
            ring.pop();
            if (issued0 < c0.n) ring.issue(xw, j0[issued0++], lane);
            else if (kind1 && issued1 < c1.n) ring.issue(xw, j1[issued1++], lane);
            if (kind0 == 2 && t + 1 < c0.n && ((bits0[t] >> 26) & 1)) {
                // row boundary inside the pack: switch to the next row's dO slice, fetch the one after it
#pragma unroll
                for (int q = 0; q < NS; ++q)
#pragma unroll
                    for (int kk = 0; kk < VW; ++kk) g0[q][kk] = g1[q][kk];
                ++rows_done;
                if (rows_done + 1 < k0) load_g<GE, CONCAT>(g1, c0.row + rows_done + 1, d_out, lane);
                else if (kind1 && c1.first) load_g<GE, CONCAT>(g1, c1.row, d_out, lane);
            }
        }
        __syncwarp();
        {
            float alpha[H], dal[H], u[H], au[H];
            const float* p0 = ring.p_s + b0 * 32 * H;
            const int bits = bits0[lane];
#pragma unroll
            for (int kk = 0; kk < H / 4; ++kk) {
                const float4 a4 = *reinterpret_cast<const float4*>(p0 + lane * H + 4 * kk);
                const float4 d4 = *reinterpret_cast<const float4*>(dal_s + lane * H + 4 * kk);
                alpha[4 * kk] = a4.x; alpha[4 * kk + 1] = a4.y; alpha[4 * kk + 2] = a4.z; alpha[4 * kk + 3] = a4.w;
                dal[4 * kk] = d4.x; dal[4 * kk + 1] = d4.y; dal[4 * kk + 2] = d4.z; dal[4 * kk + 3] = d4.w;
            }
            const bool live = lane < c0.n;
            const int64_t pos = live ? csr2csc[c0.beg + lane] : 0;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float ks = (bits >> (8 + h)) & 1 ? keep_scale : 0.f;
                u[h] = live ? alpha[h] * dal[h] * ks : 0.f;
                au[h] = alpha[h] * ks;
            }
            if (kind0 == 2) {
                const int sa = (bits >> 16) & 31, sb = live ? (bits >> 21) & 31 : lane;
                const bool lastf = live && ((bits >> 26) & 1);
                float o[H], dad[H];
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float tt = seg_total(u[h], sa, sb, lane);
                    const float sl = (bits >> h) & 1 ? 1.f : slope;
                    o[h] = live ? sl * (u[h] - alpha[h] * tt) : 0.f;
                    dad[h] = seg_total(o[h], sa, sb, lane);
                }
                if (live) {
                    store_vecH<H>(alpha_used + pos * eg_ld, au);
                    store_vecH<H>(dz + pos * eg_ld, o);
                }
                const unsigned lastm = __ballot_sync(FULL, lastf);
                if (lastf) {
                    const int64_t r = c0.row + __popc(lastm & ((1u << lane) - 1u));
                    store_vecH<H>(da_dst + r * H, dad);
                }
            } else if (c0.first && c0.last) {
                float o[H], dad[H];
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float tt = warp_sum(u[h]);
                    const float sl = (bits >> h) & 1 ? 1.f : slope;
                    o[h] = live ? sl * (u[h] - alpha[h] * tt) : 0.f;
                    dad[h] = warp_sum(o[h]);
                }
                if (live) {
                    store_vecH<H>(alpha_used + pos * eg_ld, au);
                    store_vecH<H>(dz + pos * eg_ld, o);
                }
                if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
            } else {
                if (live) {
                    store_vecH<H>(alpha_used + pos * eg_ld, au);
                    store_vecH<H>(dz + pos * eg_ld, u);
                }
#pragma unroll
                for (int h = 0; h < H; ++h) trow[h] += warp_sum(u[h]);
                if (c0.last) {
                    __syncwarp();
                    RowStat<H> r;
                    load_row_stat<H>(r, c0.row, a_dst, rowmax, rowsum);
                    float dad[H];
#pragma unroll
                    for (int h = 0; h < H; ++h) dad[h] = 0.f;
                    dst_sweep2<GE>(r, row_beg, c0.beg + c0.n, col, csr2csc, a_src, slope, trow, lane, dz, eg_ld, dad);
#pragma unroll
                    for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
                    if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
                }
            }
        }
        __syncwarp();
        if (!kind1) break;
        if (c1.first) {
#pragma unroll
            for (int q = 0; q < NS; ++q)
#pragma unroll
                for (int kk = 0; kk < VW; ++kk) g0[q][kk] = g1[q][kk];
        }
        c0 = c1;
        kind0 = kind1;
        k0 = k1;
        issued0 = issued1;
        b0 ^= 1;
    }
}

template <class GE, bool CONCAT, bool DROPOUT>
__global__ void __launch_bounds__(ST_THREADS, st_min_ctas<GE>())
gat_bwd_dst_items_pack(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                       const int32_t* __restrict__ csr2csc, const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                       const float* __restrict__ a_dst, const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                       const float* __restrict__ d_out, gnnfd_item_plan_t items, int hub_threshold, float slope,
                       KeepMask keep, float keep_scale, float* __restrict__ alpha_used,
                       float* __restrict__ dz, int64_t eg_ld, float* __restrict__ da_dst)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * ST_WARPS + warp;
    if (item >= items.n_items) return;
    WarpRing<GE, bwd_extra<GE>()> ring;
    ring.init(smem + warp * StreamGeo<GE, bwd_extra<GE>()>::WARP_BYTES, lane);
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    bwd_dst_stream_pack<GE, CONCAT, DROPOUT>(cur, ring, rowptr, col, perm, csr2csc, xw, a_src, a_dst, rowmax, rowsum, d_out, slope,
                                             keep, keep_scale, alpha_used, dz, eg_ld, da_dst, lane);
}

// hub rows, step 1: one warp per chunk -- first sweep, partial t
template <class GE, bool CONCAT, bool DROPOUT>
__global__ void __launch_bounds__(ST_THREADS, st_min_ctas<GE>())
gat_bwd_dst_hub1(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ perm,
                 const int32_t* __restrict__ csr2csc, const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                 const float* __restrict__ a_dst, const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                 const float* __restrict__ d_out, gnnfd_hub_plan_t plan, float slope,
                 KeepMask keep, float keep_scale, float* __restrict__ alpha_used,
                 float* __restrict__ dz, int64_t eg_ld, float* __restrict__ part_t)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ST_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    WarpRing<GE, bwd_extra<GE>()> ring;
    ring.init(smem + warp * StreamGeo<GE, bwd_extra<GE>()>::WARP_BYTES, lane);
    ChunkCursor cur;
    cur.start_segment(i, beg, end);
    bwd_dst_stream<GE, CONCAT, DROPOUT>(cur, ring, rowptr, col, perm, csr2csc, xw, a_src, a_dst, rowmax, rowsum, d_out, slope,
                                        keep, keep_scale, alpha_used, dz, eg_ld, part_t, c, lane);
}

template <class K>
static int set_smem_bwd(K kernel, int bytes)
{
    GNNFD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return GNNFD_OK;
}

template <class GE>
static int launch_bwd_dst(const gnnfd_graph_t* g, const void* xw_, const float* a_src, const float* a_dst,
                          const float* rowmax, const float* rowsum, const float* d_out, float slope, int concat,
                          const uint8_t* keep_mask, float p_drop, uint64_t seed, float* alpha_used, float* dz, float* da_dst, void* ws,
                          size_t ws_bytes, cudaStream_t st)
{
    using XT = typename GE::XT;
    constexpr int SMEM = StreamGeo<GE, bwd_extra<GE>()>::CTA_BYTES;
    const XT* xw = reinterpret_cast<const XT*>(xw_);
    const int64_t n = g->n_dst;
    if (n == 0) return GNNFD_OK;
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG,
                  "gat_bwd_dst: the graph has no work-item plan over rowptr (gnnfd_item_plan)");
    const bool drop = p_drop > 0.f;              // explicit mask, or (mask == NULL) the counter-based RNG keyed on seed
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + ST_WARPS - 1) / ST_WARPS);
    // two dense [E',H] arrays, or the halves of one interleaved [E',2H] buffer (dz == alpha_used + H)
    const int64_t eg_ld = (dz == alpha_used + GE::H) ? 2 * GE::H : GE::H;
    int rc = GNNFD_OK;
    // packs of whole short rows share one phase A
#define GNNFD_BWD_ITEMS_PACK(CC, DD)                                                                                   \
    rc = set_smem_bwd(gat_bwd_dst_items_pack<GE, CC, DD>, SMEM);                                                       \
    if (rc) return rc;                                                                                                 \
    gat_bwd_dst_items_pack<GE, CC, DD><<<grid, ST_THREADS, SMEM, st>>>(g->rowptr, g->col, g->perm, g->csr2csc, xw, a_src, a_dst,    \
                                                                       rowmax, rowsum, d_out, g->items_dst, thr, slope, keep, \
                                                                       ks, alpha_used, dz, eg_ld, da_dst)
    if (concat) { if (drop) { GNNFD_BWD_ITEMS_PACK(true, true); } else { GNNFD_BWD_ITEMS_PACK(true, false); } }
    else        { if (drop) { GNNFD_BWD_ITEMS_PACK(false, true); } else { GNNFD_BWD_ITEMS_PACK(false, false); } }
#undef GNNFD_BWD_ITEMS_PACK
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const size_t need = 2 * carve_bytes(size_t(pl.n_chunk) * GE::H, 4) + carve_bytes(size_t(pl.n_hub) * GE::H, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_bwd_dst: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        float* part_t = carve<float>(p, size_t(pl.n_chunk) * GE::H);
        float* part_dad = carve<float>(p, size_t(pl.n_chunk) * GE::H);
        float* t_total = carve<float>(p, size_t(pl.n_hub) * GE::H);
        const unsigned gh = (unsigned)((pl.n_hub + ROW_WARPS - 1) / ROW_WARPS);
        const unsigned gc = (unsigned)((pl.n_chunk + ST_WARPS - 1) / ST_WARPS);
        const unsigned gc2 = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
#define GNNFD_BWD_HUB1(CC, DD)                                                                                         \
    rc = set_smem_bwd(gat_bwd_dst_hub1<GE, CC, DD>, SMEM);                                                             \
    if (rc) return rc;                                                                                                 \
    gat_bwd_dst_hub1<GE, CC, DD><<<gc, ST_THREADS, SMEM, st>>>(g->rowptr, g->col, g->perm, g->csr2csc, xw, a_src, a_dst, rowmax,     \
                                                               rowsum, d_out, pl, slope, keep, ks, alpha_used, dz, eg_ld, part_t)
        if (concat) { if (drop) { GNNFD_BWD_HUB1(true, true); } else { GNNFD_BWD_HUB1(true, false); } }
        else        { if (drop) { GNNFD_BWD_HUB1(false, true); } else { GNNFD_BWD_HUB1(false, false); } }
#undef GNNFD_BWD_HUB1
        gat_hub_chunk_sum<GE::H, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_t, t_total);
        gat_bwd_dst_hub2<GE><<<gc2, ROW_THREADS, 0, st>>>(g->rowptr, g->col, g->csr2csc, a_src, a_dst, rowmax, rowsum, pl, slope,
                                                          t_total, dz, eg_ld, part_dad);
        gat_hub_chunk_sum<GE::H, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_dad, da_dst);
        g_launches += 4;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace gnnfd

using namespace gnnfd;

extern "C" {

int gnnfd_gat_bwd_dst(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src, const float* a_dst,
                      const float* rowmax, const float* rowsum, const float* d_out, int H, int C,
                      float negative_slope, int concat, const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, float* alpha_used,
                      float* dz, float* da_dst, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    int rc = check_graph(g, false, "gat_bwd_dst");
    if (rc) return rc;
    GNNFD_REQUIRE(g->n_dst == 0 || (xw && a_src && a_dst && rowmax && rowsum && d_out && da_dst), GNNFD_ERR_ARG,
                  "gat_bwd_dst: NULL tensor");
    GNNFD_REQUIRE(g->n_edges == 0 || (alpha_used && dz), GNNFD_ERR_ARG, "gat_bwd_dst: alpha_used/dz is NULL");
    GNNFD_REQUIRE(g->n_edges == 0 || g->csr2csc, GNNFD_ERR_ARG,
                  "gat_bwd_dst: csr2csc is NULL (edge gradients are emitted in source-major order)");
    GNNFD_REQUIRE(p_drop >= 0.f && p_drop < 1.f, GNNFD_ERR_ARG, "gat_bwd_dst: dropout p must be in [0,1)");
    cudaStream_t st = (cudaStream_t)stream;
    if (gat_bwd_dst_srcmajor_applies(g, concat))
        return gat_bwd_dst_srcmajor(g, xw, xw_dtype, H, C, a_src, a_dst, rowmax, rowsum, d_out, negative_slope, keep_mask,
                                    p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst<Geo<8, 64, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope, concat,
                                                 keep_mask, p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_BF16)
        return launch_bwd_dst<Geo<8, 64, __nv_bfloat16>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope,
                                                         concat, keep_mask, p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 4 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst<Geo<4, 32, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope, concat,
                                                 keep_mask, p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst<Geo<8, 32, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope, concat,
                                                 keep_mask, p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 128 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst<Geo<8, 128, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope, concat,
                                                  keep_mask, p_drop, dropout_seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_bwd_dst: (heads=%d, out_channels=%d, dtype=%d) is not built; "
                  "available: (8,64,f32), (8,64,bf16), (8,32,f32), (8,128,f32), (4,32,f32)", H, C, xw_dtype);
    return GNNFD_ERR_UNSUPPORTED;
}

}  // extern "C"
