// (4b) backward, src-major pass (autograd mirror of GATConv.forward, triggered by loss.backward() at
// src/train.py:142; closed forms in SURVEY.md 8(a3)).
//
// CSC, warp per source row: dxw[j] = sum_e alpha_used[e] * dO_h[dst(e)] -- with the head mean every head
// shares dOut[i]/H, so the per-edge gather is only C*4 = 256 B -- plus the logit terms
// da_src[j]*att_src + da_dst[j]*att_dst fused into the row epilogue; da_src[j] = sum_e dz[e].
// Source rows with more than the hub threshold of out-edges are split into chunks (one warp each) whose
// partial sums are merged in chunk order -- deterministic.
#include "gat_common.cuh"

#include <atomic>
#include <climits>
#include <cstdlib>

namespace gnnfd {
extern std::atomic<long long> g_launches;
int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who);
bool gat_bwd_dst_srcmajor_applies(const gnnfd_graph_t* g, int concat);       // gat_bwd_dalpha.cu
size_t gat_bwd_dst_srcmajor_ws_bytes(const gnnfd_graph_t* g, int H);

constexpr int SRC_MINB = 4;
constexpr int BWD_U = 4;
// The rows kernel at 8 x 128 channels (32 accumulators per lane): two CTAs per SM instead of SRC_MINB, and
// with concat one dO row in flight per lane instead of BWD_U (each is 32 more registers), so that nothing spills.
template <class GE>
constexpr int src_minb()
{
    return GE::D > 512 ? 2 : SRC_MINB;
}
template <class GE, bool CONCAT>
constexpr int src_unroll()
{
    return (GE::D > 512 && CONCAT) ? 1 : BWD_U;
}

// ---------------------------------------------------------------------------------------------------------
// src-major pass
// ---------------------------------------------------------------------------------------------------------
template <class GE, bool CONCAT>
__device__ __forceinline__ void src_range(int beg, int end, const int32_t* __restrict__ csc_row,
                                          const int32_t* __restrict__ csc_eid, const float* __restrict__ alpha_used,
                                          const float* __restrict__ dz, int64_t eg_ld, const float* __restrict__ d_out,
                                          float (&acc)[GE::NS][4], float (&das)[GE::H], float* p_s, int* i_s, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, HP = GE::HP, D = GE::D, C = GE::C, U = src_unroll<GE, CONCAT>();
    const int sub = lane / GE::G;
    const int cm = (4 * lane) % C;   // C divides 128, so every slot of this lane has the same channel offset
    for (int base = beg; base < end; base += 32) {
        const int n = min(32, end - base);
        int i = 0;
        if (lane < n) {
            // edge gradients are normally stored in source-major order; csc_eid != NULL = indirect (multi-GPU receive buffer)
            const int64_t eid = csc_eid ? int64_t(csc_eid[base + lane]) : int64_t(base + lane);
            i = csc_row[base + lane];
            float al[H], dzv[H];
            load_vecH<H>(alpha_used + eid * eg_ld, al);
            load_vecH<H>(dz + eid * eg_ld, dzv);
#pragma unroll
            for (int h = 0; h < H; ++h) das[h] += dzv[h];
            store_vecH<H>(p_s + lane * H, al);
        }
        i_s[lane] = i;
        __syncwarp();
        for (int t = 0; t < n; t += U) {
            float g[U][CONCAT ? NS : 1][4], wq[U][NS];
#pragma unroll
            for (int uu = 0; uu < U; ++uu) {
                const bool ok = t + uu < n;
                const int tt = ok ? t + uu : t;
                const int64_t ii = i_s[tt];
#pragma unroll
                for (int q = 0; q < (CONCAT ? NS : 1); ++q) {
                    const float* p = CONCAT ? d_out + ii * D + 4 * (lane + 32 * q) : d_out + ii * C + cm;
                    float4 tv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ok) tv = CONCAT ? ldg_stream(reinterpret_cast<const float4*>(p)) : __ldg(reinterpret_cast<const float4*>(p));
                    g[uu][q][0] = tv.x; g[uu][q][1] = tv.y; g[uu][q][2] = tv.z; g[uu][q][3] = tv.w;
                }
#pragma unroll
                for (int q = 0; q < NS; ++q) wq[uu][q] = ok ? p_s[tt * H + q * HP + sub] : 0.f;
            }
#pragma unroll
            for (int uu = 0; uu < U; ++uu)
#pragma unroll
                for (int q = 0; q < NS; ++q)
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc[q][k] = fmaf(wq[uu][q], g[uu][CONCAT ? q : 0][k], acc[q][k]);
        }
        __syncwarp();
    }
}

template <class GE, bool CONCAT>
__device__ __forceinline__ void src_epilogue(int64_t j, float (&acc)[GE::NS][4], const float (&das)[GE::H],
                                             const float* __restrict__ att_src, const float* __restrict__ att_dst,
                                             const float* __restrict__ da_dst_full, float* __restrict__ dxw,
                                             float* __restrict__ da_src, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, HP = GE::HP, D = GE::D;
    const int sub = lane / GE::G;
    float dad[H];
    if (da_dst_full) load_vecH<H>(da_dst_full + j * H, dad);
    else {
#pragma unroll
        for (int h = 0; h < H; ++h) dad[h] = 0.f;
    }
    if (lane == 0) store_vecH<H>(da_src + j * H, das);
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const int e0 = 4 * (lane + 32 * q);
        const float fs = pick<HP>(das, q, sub), fd = pick<HP>(dad, q, sub);
        const float4 as4 = __ldg(reinterpret_cast<const float4*>(att_src + e0));
        const float4 ad4 = __ldg(reinterpret_cast<const float4*>(att_dst + e0));
        const float sc = CONCAT ? 1.f : 1.f / H;
        float4 o;
        o.x = fmaf(acc[q][0], sc, fmaf(fs, as4.x, fd * ad4.x));
        o.y = fmaf(acc[q][1], sc, fmaf(fs, as4.y, fd * ad4.y));
        o.z = fmaf(acc[q][2], sc, fmaf(fs, as4.z, fd * ad4.z));
        o.w = fmaf(acc[q][3], sc, fmaf(fs, as4.w, fd * ad4.w));
        stg_stream(reinterpret_cast<float4*>(dxw + j * D + e0), o);
    }
}

template <class GE, bool CONCAT>
__global__ void __launch_bounds__(ROW_THREADS, src_minb<GE>())
gat_bwd_src_rows(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                 const int32_t* __restrict__ csc_eid, const float* __restrict__ alpha_used,
                 const float* __restrict__ dz, int64_t eg_ld, const float* __restrict__ d_out, const float* __restrict__ att_src,
                 const float* __restrict__ att_dst, const float* __restrict__ da_dst_full, gnnfd_item_plan_t items,
                 int hub_threshold, int look, float* __restrict__ dxw, float* __restrict__ da_src)
{
    constexpr int H = GE::H, NS = GE::NS;
    __shared__ __align__(16) float p_sh[ROW_WARPS][32 * H];
    __shared__ int i_sh[ROW_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // one warp per edge-balanced work item (a run of whole source rows, ~target out-edges in total)
    const int item = blockIdx.x * ROW_WARPS + warp;
    if (item >= items.n_items) return;
    const int j_end = items.item_start[item + 1];
    // L2 look-ahead: the item's edges are one contiguous CSC range, so the warp prefetches the dOut rows (and the
    // alpha/dz lines) of the edges up to `look` positions ahead of the row it is working on (in batches of 32).
    // The gathers below then hit L2 instead of paying a DRAM round trip per dependent step, without holding any
    // registers for the data.  look = 0 disables it.
    const int e_item_end = colptr[j_end];
    int pf = colptr[items.item_start[item]];
    int pf_i = (pf + lane < e_item_end) ? csc_row[pf + lane] : -1;
    for (int64_t j = items.item_start[item]; j < j_end; ++j) {
        const int beg = colptr[j], end = colptr[j + 1];
        if (end - beg > hub_threshold) {                // split rows are produced by the hub kernels
            if (pf < end) {
                pf = end;
                pf_i = (pf + lane < e_item_end) ? csc_row[pf + lane] : -1;
            }
            continue;
        }
        while (pf < e_item_end && pf < beg + look) {
            if (pf_i >= 0) {
                const float* pr = d_out + int64_t(pf_i) * (CONCAT ? GE::D : GE::C);
#pragma unroll
                for (int b = 0; b < (CONCAT ? GE::D : GE::C) * 4; b += 128) prefetch_l2(reinterpret_cast<const char*>(pr) + b);
                if (!csc_eid) prefetch_l2(alpha_used + int64_t(pf + lane) * eg_ld);
            }
            pf += 32;
            pf_i = (pf + lane < e_item_end) ? csc_row[pf + lane] : -1;
        }
        float acc[NS][4], das[H];
#pragma unroll
        for (int q = 0; q < NS; ++q)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[q][k] = 0.f;
#pragma unroll
        for (int h = 0; h < H; ++h) das[h] = 0.f;
        src_range<GE, CONCAT>(beg, end, csc_row, csc_eid, alpha_used, dz, eg_ld, d_out, acc, das, p_sh[warp], i_sh[warp], lane);
#pragma unroll
        for (int h = 0; h < H; ++h) das[h] = warp_sum(das[h]);
        src_epilogue<GE, CONCAT>(j, acc, das, att_src, att_dst, da_dst_full, dxw, da_src, lane);
    }
}

template <class GE, bool CONCAT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_src_hub_chunks(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                       const int32_t* __restrict__ csc_eid, const float* __restrict__ alpha_used,
                       const float* __restrict__ dz, int64_t eg_ld, const float* __restrict__ d_out, gnnfd_hub_plan_t plan,
                       float* __restrict__ part_acc, float* __restrict__ part_das)
{
    constexpr int H = GE::H, NS = GE::NS, D = GE::D;
    __shared__ __align__(16) float p_sh[ROW_WARPS][32 * H];
    __shared__ int i_sh[ROW_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t j = plan.hub_row[slot];
    const int beg = colptr[j] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(colptr[j + 1], beg + plan.chunk);
    float acc[NS][4], das[H];
#pragma unroll
    for (int q = 0; q < NS; ++q)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[q][k] = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) das[h] = 0.f;
    src_range<GE, CONCAT>(beg, end, csc_row, csc_eid, alpha_used, dz, eg_ld, d_out, acc, das, p_sh[warp], i_sh[warp], lane);
#pragma unroll
    for (int h = 0; h < H; ++h) das[h] = warp_sum(das[h]);
    if (lane == 0) store_vecH<H>(part_das + int64_t(c) * H, das);
#pragma unroll
    for (int q = 0; q < NS; ++q)
        *reinterpret_cast<float4*>(part_acc + int64_t(c) * D + 4 * (lane + 32 * q)) =
            make_float4(acc[q][0], acc[q][1], acc[q][2], acc[q][3]);
}

template <class GE, bool CONCAT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_src_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part_acc, const float* __restrict__ part_das,
                      const float* __restrict__ att_src, const float* __restrict__ att_dst,
                      const float* __restrict__ da_dst_full, float* __restrict__ dxw, float* __restrict__ da_src)
{
    constexpr int H = GE::H, NS = GE::NS, D = GE::D;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * ROW_WARPS + warp;
    if (slot >= plan.n_hub) return;
    const int64_t j = plan.hub_row[slot];
    float acc[NS][4], das[H];
#pragma unroll
    for (int q = 0; q < NS; ++q)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[q][k] = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) das[h] = 0.f;
    for (int c = plan.hub_chunk_ptr[slot]; c < plan.hub_chunk_ptr[slot + 1]; ++c) {
        float pd[H];
        load_vecH<H>(part_das + int64_t(c) * H, pd);
#pragma unroll
        for (int h = 0; h < H; ++h) das[h] += pd[h];
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const float4 v = *reinterpret_cast<const float4*>(part_acc + int64_t(c) * D + 4 * (lane + 32 * q));
            acc[q][0] += v.x; acc[q][1] += v.y; acc[q][2] += v.z; acc[q][3] += v.w;
        }
    }
    src_epilogue<GE, CONCAT>(j, acc, das, att_src, att_dst, da_dst_full, dxw, da_src, lane);
}

template <class GE>
static int launch_bwd_src(const gnnfd_graph_t* g, const float* alpha_used, const float* dz, const float* d_out,
                          const float* att_src, const float* att_dst, const float* da_dst_full, int concat, float* dxw,
                          float* da_src, void* ws, size_t ws_bytes, cudaStream_t st)
{
    const int64_t n = g->n_src;
    if (n == 0) return GNNFD_OK;
    const int32_t* eid_ptr = g->edge_grads_indirect ? g->csc_eid : nullptr;
    // two dense [E',H] arrays, or the halves of one interleaved [E',2H] buffer (dz == alpha_used + H)
    const int64_t eg_ld = (dz == alpha_used + GE::H) ? 2 * GE::H : GE::H;
    const int thr = g->hub_src.n_hub > 0 ? g->hub_src.threshold : INT_MAX;
    GNNFD_REQUIRE(g->items_src.n_items > 0 && g->items_src.item_start, GNNFD_ERR_ARG,
                  "gat_bwd_src: the graph has no work-item plan over colptr (gnnfd_item_plan)");
    const unsigned grid = (unsigned)((g->items_src.n_items + ROW_WARPS - 1) / ROW_WARPS);
    static const int look = [] {
        const char* e = getenv("GNNFD_SRC_LOOKAHEAD");     // edges of L2 look-ahead per warp (tuning knob)
        return e ? atoi(e) : 0;      // measured on the 200M-edge graph: every distance > 0 is slower (L2 thrash)
    }();
    if (concat)
        gat_bwd_src_rows<GE, true><<<grid, ROW_THREADS, 0, st>>>(g->colptr, g->csc_row, eid_ptr, alpha_used, dz, eg_ld, d_out,
                                                                 att_src, att_dst, da_dst_full, g->items_src, thr, look, dxw, da_src);
    else
        gat_bwd_src_rows<GE, false><<<grid, ROW_THREADS, 0, st>>>(g->colptr, g->csc_row, eid_ptr, alpha_used, dz, eg_ld, d_out,
                                                                  att_src, att_dst, da_dst_full, g->items_src, thr, look, dxw, da_src);
    g_launches += 1;
    if (g->hub_src.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_src;
        const size_t need = carve_bytes(size_t(pl.n_chunk) * GE::D, 4) + carve_bytes(size_t(pl.n_chunk) * GE::H, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_bwd_src: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        float* part_acc = carve<float>(p, size_t(pl.n_chunk) * GE::D);
        float* part_das = carve<float>(p, size_t(pl.n_chunk) * GE::H);
        const unsigned gc = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
        const unsigned gh = (unsigned)((pl.n_hub + ROW_WARPS - 1) / ROW_WARPS);
        if (concat) {
            gat_bwd_src_hub_chunks<GE, true><<<gc, ROW_THREADS, 0, st>>>(g->colptr, g->csc_row, eid_ptr, alpha_used, dz, eg_ld,
                                                                         d_out, pl, part_acc, part_das);
            gat_bwd_src_hub_merge<GE, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_acc, part_das, att_src, att_dst,
                                                                        da_dst_full, dxw, da_src);
        } else {
            gat_bwd_src_hub_chunks<GE, false><<<gc, ROW_THREADS, 0, st>>>(g->colptr, g->csc_row, eid_ptr, alpha_used, dz, eg_ld,
                                                                          d_out, pl, part_acc, part_das);
            gat_bwd_src_hub_merge<GE, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_acc, part_das, att_src, att_dst,
                                                                         da_dst_full, dxw, da_src);
        }
        g_launches += 2;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace gnnfd

using namespace gnnfd;

extern "C" {

int gnnfd_gat_bwd_workspace_bytes(const gnnfd_graph_t* g, int H, int C, size_t* bytes)
{
    GNNFD_REQUIRE(g && bytes, GNNFD_ERR_ARG, "gat_bwd_workspace_bytes: NULL argument");
    const size_t nd = (size_t)g->hub_dst.n_chunk, ns = (size_t)g->hub_src.n_chunk;
    // the dst pass: its two-pass form (head mean) also keeps the [E',2H] records here; concat is not known at this point
    const size_t a = gat_bwd_dst_srcmajor_applies(g, 0) ? gat_bwd_dst_srcmajor_ws_bytes(g, H)
                                                        : 2 * carve_bytes(nd * H, 4) + carve_bytes(size_t(g->hub_dst.n_hub) * H, 4);
    const size_t b = carve_bytes(ns * size_t(H) * C, 4) + carve_bytes(ns * H, 4);
    *bytes = (a > b ? a : b) + 256;
    return GNNFD_OK;
}

int gnnfd_gat_bwd_src(const gnnfd_graph_t* g, const float* alpha_used, const float* dz, const float* d_out,
                      const float* att_src, const float* att_dst, const float* da_dst_full, int H, int C, int concat,
                      float* dxw, float* da_src, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    int rc = check_graph(g, true, "gat_bwd_src");
    if (rc) return rc;
    GNNFD_REQUIRE(g->n_src == 0 || (att_src && att_dst && dxw && da_src), GNNFD_ERR_ARG, "gat_bwd_src: NULL tensor");
    GNNFD_REQUIRE(g->n_edges == 0 || (alpha_used && dz && d_out), GNNFD_ERR_ARG, "gat_bwd_src: NULL edge tensor");
    cudaStream_t st = (cudaStream_t)stream;
    if (H == 8 && C == 64)
        return launch_bwd_src<Geo<8, 64, float>>(g, alpha_used, dz, d_out, att_src, att_dst, da_dst_full, concat, dxw,
                                                 da_src, ws, ws_bytes, st);
    if (H == 4 && C == 32)
        return launch_bwd_src<Geo<4, 32, float>>(g, alpha_used, dz, d_out, att_src, att_dst, da_dst_full, concat, dxw,
                                                 da_src, ws, ws_bytes, st);
    if (H == 8 && C == 32)
        return launch_bwd_src<Geo<8, 32, float>>(g, alpha_used, dz, d_out, att_src, att_dst, da_dst_full, concat, dxw,
                                                 da_src, ws, ws_bytes, st);
    if (H == 8 && C == 128)
        return launch_bwd_src<Geo<8, 128, float>>(g, alpha_used, dz, d_out, att_src, att_dst, da_dst_full, concat, dxw,
                                                  da_src, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_bwd_src: (heads=%d, out_channels=%d) is not built; "
                  "available: (8,64), (8,32), (8,128), (4,32)", H, C);
    return GNNFD_ERR_UNSUPPORTED;
}

}  // extern "C"
