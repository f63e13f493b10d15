// (4a) backward, dst-major pass for the head mean (concat = False): two passes, no per-edge feature-row gather.
//
// d_alpha[e,h] = <dO[i]/H, xw[j,h,:]> needs no row reduction, and with the head mean dO[i] is one C-float row
// shared by all heads.  So d_alpha is computed SOURCE-major, where xw[j] is read once, and only the 256 B dO[i] row
// is gathered per edge; the row reductions follow in a second pass that reads no features.
//   pass 1 (CSC, one warp per source row j; gat_bwd_dalpha_src_rows / _hub): xw[j] is held in registers in the
//            slot layout of gat_common.cuh.  Per chunk of <= 32 out-edges the warp copies the chunk's dO rows into
//            shared memory (cp.async, all in flight at once) while each lane (= edge) computes alpha from the
//            destination's saved statistics exactly as phase A does.  Then per edge 16 FMAs and phase B's butterfly
//            give d_alpha with phase B's arithmetic.  The edge's 64 B slot of the edge-gradient buffer (its CSC
//            position) receives the pre-dropout alpha, with the sign bit set where the logit is on the LeakyReLU's
//            negative side, and d_alpha.  Sources above the hub threshold are split by the hub_src plan; every output
//            is per edge, so the chunks need no merge.
//   pass 2 (CSR; gat_bwd_dst_eg_items / _hub1 / _hub2): the chunk, pack and hub_dst schedule of the gather kernels,
//            lane = edge, reading the slot at csr2csc[e] instead of the row xw[col[e]].  Keep bits, u = alpha *
//            d_alpha * keep, t, dz and da_dst use the same warp sums in the same order as the gather kernels, and
//            the slot is overwritten with (alpha_used, dz) by the thread that read it.
// Per edge this moves ~4 + 256 + 96 + 64 B (pass 1) and ~4 + 64 + 64 B (pass 2) instead of a 2 KB row.  alpha_used
// equals the gather kernels' bit for bit; dz and da_dst differ in the last bits on rows longer than one chunk, where
// the gather kernels recompute alpha for the second sweep with a contracted multiply-add.
#include "gat_stream.cuh"
#include "gat_phase_bwd.cuh"

#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;

constexpr int DA_WARPS = 4;                  // warps per CTA in pass 1 (the dO staging fits static shared memory)
constexpr int DA_THREADS = DA_WARPS * 32;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(st_smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
constexpr uint32_t NEG_FLAG = 0x80000000u;   // sign bit of the stored alpha: LeakyReLU-negative logit

// ---------------------------------------------------------------------------------------------------------
// pass 1: source-major d_alpha
// ---------------------------------------------------------------------------------------------------------
// out-edges [beg, end) of source row j (a whole row, or one hub chunk of it).  Per chunk the warp copies the chunk's
// dO rows into do_s [32][C] (cp.async, all in flight at once) while the lanes compute alpha.
template <class GE>
__device__ __forceinline__ void dalpha_range(int64_t j, int beg, int end, const int32_t* __restrict__ csc_row,
                                             const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                                             const float* __restrict__ a_dst, const float* __restrict__ rowmax,
                                             const float* __restrict__ rowsum, const float* __restrict__ d_out,
                                             float slope, float* __restrict__ alpha_used, float* __restrict__ dz,
                                             int64_t eg_ld, float* do_s, float* dal_s, int* i_s, int lane)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, C = GE::C;
    static_assert((32 * VW) % C == 0, "every slot of a lane must see the same dO channels");
    float v[NS][VW];
#pragma unroll
    for (int q = 0; q < NS; ++q) load_slot(xw + j * GE::D, q, lane, v[q]);
    const int cm = (VW * lane) % C;          // dO channels of this lane's slots
    const float sc = 1.f / H;
    for (int base = beg; base < end; base += 32) {
        const int n = min(32, end - base);
        const int64_t i = lane < n ? csc_row[base + lane] : 0;
        i_s[lane] = int(i);
        __syncwarp();
        // C/4 lanes copy one dO row (16 B each): every instruction moves 32/(C/4) whole rows
        {
            constexpr int LPR = C / 4, RPI = 32 / LPR;
            const int sub = lane / LPR, c4 = 4 * (lane % LPR);
#pragma unroll
            for (int r = 0; r < 32; r += RPI)
                if (r + sub < n) cp_async16(do_s + (r + sub) * C + c4, d_out + int64_t(i_s[r + sub]) * C + c4);
        }
        if (lane < n) {
            // alpha as phase A computes it (load_row_stat), four heads at a time
#pragma unroll
            for (int k = 0; k < H / 4; ++k) {
                const float4 as = __ldg(reinterpret_cast<const float4*>(a_src + j * H) + k);
                const float4 ad = __ldg(reinterpret_cast<const float4*>(a_dst + i * H) + k);
                const float4 mx = __ldg(reinterpret_cast<const float4*>(rowmax + i * H) + k);
                const float4 sm = __ldg(reinterpret_cast<const float4*>(rowsum + i * H) + k);
                const float zs[4] = {as.x + ad.x, as.y + ad.y, as.z + ad.z, as.w + ad.w};
                const float ms[4] = {mx.x, mx.y, mx.z, mx.w}, ss[4] = {sm.x, sm.y, sm.z, sm.w};
                float al[4];
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const float z = zs[h], inv = 1.f / ss[h];
                    const bool pos = z > 0.f;
                    const float a = expf((pos ? z : z * slope) - ms[h]) * inv;
                    al[h] = __uint_as_float(__float_as_uint(a) | (pos ? 0u : NEG_FLAG));
                }
                reinterpret_cast<float4*>(alpha_used + int64_t(base + lane) * eg_ld)[k] = make_float4(al[0], al[1], al[2], al[3]);
            }
        }
        cp_async_wait_all();
        __syncwarp();
        for (int t = 0; t < n; ++t) {
            float g[VW];
#pragma unroll
            for (int k = 0; k < VW; k += 4) {
                const float4 tv = *reinterpret_cast<const float4*>(do_s + t * C + cm + k);
                g[k] = tv.x * sc; g[k + 1] = tv.y * sc; g[k + 2] = tv.z * sc; g[k + 3] = tv.w * sc;
            }
            float d[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                d[q] = 0.f;
#pragma unroll
                for (int k = 0; k < VW; ++k) d[q] = fmaf(g[k], v[q][k], d[q]);
            }
            dalpha_reduce<GE>(d, dal_s + t * H, lane);
        }
        __syncwarp();
        if (lane < n) {
            float dal[H];
#pragma unroll
            for (int k = 0; k < H / 4; ++k) {
                const float4 d4 = *reinterpret_cast<const float4*>(dal_s + lane * H + 4 * k);
                dal[4 * k] = d4.x; dal[4 * k + 1] = d4.y; dal[4 * k + 2] = d4.z; dal[4 * k + 3] = d4.w;
            }
            store_vecH<H>(dz + int64_t(base + lane) * eg_ld, dal);
        }
        __syncwarp();
    }
}

// one warp per edge-balanced work item over colptr (a run of whole source rows); hub rows are left to _hub
template <class GE>
__global__ void __launch_bounds__(DA_THREADS, 6)
gat_bwd_dalpha_src_rows(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                        const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                        const float* __restrict__ a_dst, const float* __restrict__ rowmax,
                        const float* __restrict__ rowsum, const float* __restrict__ d_out, gnnfd_item_plan_t items,
                        int hub_threshold, float slope, float* __restrict__ alpha_used, float* __restrict__ dz,
                        int64_t eg_ld)
{
    __shared__ __align__(16) float do_sh[DA_WARPS][32 * GE::C];
    __shared__ __align__(16) float dal_sh[DA_WARPS][32 * GE::H];
    __shared__ int i_sh[DA_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * DA_WARPS + warp;
    if (item >= items.n_items) return;
    const int j_end = items.item_start[item + 1];
    for (int64_t j = items.item_start[item]; j < j_end; ++j) {
        const int beg = colptr[j], end = colptr[j + 1];
        if (end == beg || end - beg > hub_threshold) continue;
        dalpha_range<GE>(j, beg, end, csc_row, xw, a_src, a_dst, rowmax, rowsum, d_out, slope, alpha_used, dz, eg_ld,
                         do_sh[warp], dal_sh[warp], i_sh[warp], lane);
    }
}

// one warp per chunk of a hub source row
template <class GE>
__global__ void __launch_bounds__(DA_THREADS, 6)
gat_bwd_dalpha_src_hub(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                       const typename GE::XT* __restrict__ xw, const float* __restrict__ a_src,
                       const float* __restrict__ a_dst, const float* __restrict__ rowmax,
                       const float* __restrict__ rowsum, const float* __restrict__ d_out, gnnfd_hub_plan_t plan,
                       float slope, float* __restrict__ alpha_used, float* __restrict__ dz, int64_t eg_ld)
{
    __shared__ __align__(16) float do_sh[DA_WARPS][32 * GE::C];
    __shared__ __align__(16) float dal_sh[DA_WARPS][32 * GE::H];
    __shared__ int i_sh[DA_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * DA_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t j = plan.hub_row[slot];
    const int beg = colptr[j] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(colptr[j + 1], beg + plan.chunk);
    dalpha_range<GE>(j, beg, end, csc_row, xw, a_src, a_dst, rowmax, rowsum, d_out, slope, alpha_used, dz, eg_ld,
                     do_sh[warp], dal_sh[warp], i_sh[warp], lane);
}

// ---------------------------------------------------------------------------------------------------------
// pass 2: feature-free dst-major reductions
// ---------------------------------------------------------------------------------------------------------
// pass 1's slot of one edge, lane = edge.  The slot is read here and overwritten later by the same thread, so
// plain (coherent) loads are used.
template <int H>
struct EgEdge {
    float a[H], d[H];      // alpha with the LeakyReLU-negative flag, d_alpha
    int pos;               // source-major slot
    unsigned keep;         // dropout keep bits
};
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_load(EgEdge<H>& x, int e, bool live, const int32_t* __restrict__ perm,
                                        const int32_t* __restrict__ csr2csc, KeepMask keep,
                                        const float* alpha_used, const float* dz, int64_t eg_ld)
{
    x.pos = 0;
    x.keep = 0xffu;
#pragma unroll
    for (int h = 0; h < H; ++h) x.a[h] = x.d[h] = 0.f;
    if (!live) return;
    x.pos = csr2csc[e];
#pragma unroll
    for (int k = 0; k < H / 4; ++k) {
        const float4 a4 = reinterpret_cast<const float4*>(alpha_used + int64_t(x.pos) * eg_ld)[k];
        const float4 d4 = reinterpret_cast<const float4*>(dz + int64_t(x.pos) * eg_ld)[k];
        x.a[4 * k] = a4.x; x.a[4 * k + 1] = a4.y; x.a[4 * k + 2] = a4.z; x.a[4 * k + 3] = a4.w;
        x.d[4 * k] = d4.x; x.d[4 * k + 1] = d4.y; x.d[4 * k + 2] = d4.z; x.d[4 * k + 3] = d4.w;
    }
    if (DROPOUT) x.keep = keep.bits(perm[e], H);
}
// head h of an edge, phase C's arithmetic: pre-dropout alpha, LeakyReLU slope, keep scale, u = alpha * d_alpha * keep
struct EgHead {
    float alpha, sl, ks, u;
};
template <int H>
__device__ __forceinline__ EgHead eg_head(const EgEdge<H>& x, int h, bool live, float slope, float keep_scale)
{
    EgHead r;
    const uint32_t w = __float_as_uint(x.a[h]);
    r.alpha = __uint_as_float(w & ~NEG_FLAG);
    r.sl = (w & NEG_FLAG) ? slope : 1.f;
    r.ks = (x.keep >> h) & 1 ? keep_scale : 0.f;
    r.u = live ? r.alpha * x.d[h] * r.ks : 0.f;
    return r;
}
// the final slot: alpha_used = alpha * keep, dz
template <int H>
__device__ __forceinline__ void eg_store(const EgEdge<H>& x, const float (&o)[H], float keep_scale, float* alpha_used,
                                         float* dz, int64_t eg_ld)
{
    float au[H];
#pragma unroll
    for (int h = 0; h < H; ++h)
        au[h] = __uint_as_float(__float_as_uint(x.a[h]) & ~NEG_FLAG) * ((x.keep >> h) & 1 ? keep_scale : 0.f);
    store_vecH<H>(alpha_used + int64_t(x.pos) * eg_ld, au);
    store_vecH<H>(dz + int64_t(x.pos) * eg_ld, o);
}
// second sweep of a row (or hub chunk) whose t is known: final alpha_used and dz into the slots, lane-local da_dst
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_sweep2(int beg, int end, const int32_t* __restrict__ perm,
                                          const int32_t* __restrict__ csr2csc, KeepMask keep, float keep_scale,
                                          float slope, const float (&t)[H], float* alpha_used, float* dz,
                                          int64_t eg_ld, float (&dad)[H], int lane)
{
    for (int e = beg + lane; e < end; e += 32) {
        EgEdge<H> x;
        eg_load<H, DROPOUT>(x, e, true, perm, csr2csc, keep, alpha_used, dz, eg_ld);
        float o[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const EgHead v = eg_head<H>(x, h, true, slope, keep_scale);
            o[h] = v.sl * (v.u - v.alpha * t[h]);
            dad[h] += o[h];
        }
        eg_store<H>(x, o, keep_scale, alpha_used, dz, eg_ld);
    }
}

// one warp per edge-balanced work item over rowptr; the chunk and pack sequence of gat_bwd_dst_items_pack, with the
// next chunk's slots loaded while the current one is reduced
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS, 2)
gat_bwd_dst_eg_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                     const int32_t* __restrict__ csr2csc, gnnfd_item_plan_t items, int hub_threshold, float slope,
                     KeepMask keep, float keep_scale, float* alpha_used, float* dz, int64_t eg_ld,
                     float* __restrict__ da_dst)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * ROW_WARPS + warp;
    if (item >= items.n_items) return;
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    auto on_empty = [&](int r) {
        if (lane < H) da_dst[int64_t(r) * H + lane] = 0.f;
    };
    BwdChunk c0, c1;
    int k0 = 0, k1 = 0, la = 0, lb = 0, lo = 0;
    int sa0 = 0, sb0 = 0, sa1 = 0, sb1 = 0;
    int kind0 = cur.next_any(rowptr, lane, c0.row, c0.beg, c0.n, c0.first, c0.last, k0, la, lb, on_empty);
    if (!kind0) return;
    if (kind0 == 2) pack_lane_segment(c0.beg, k0, la, lb, lane, lo, sa0, sb0);
    EgEdge<H> x0, x1;
    eg_load<H, DROPOUT>(x0, c0.beg + lane, lane < c0.n, perm, csr2csc, keep, alpha_used, dz, eg_ld);
    float trow[H];               // running t = sum alpha*d_alpha of the current (multi-chunk) row
    int row_beg = c0.beg;        // first edge of the current row
#pragma unroll
    for (int h = 0; h < H; ++h) trow[h] = 0.f;
    while (true) {
        const int kind1 = cur.next_any(rowptr, lane, c1.row, c1.beg, c1.n, c1.first, c1.last, k1, la, lb, on_empty);
        if (kind1 == 2) pack_lane_segment(c1.beg, k1, la, lb, lane, lo, sa1, sb1);
        if (kind1) eg_load<H, DROPOUT>(x1, c1.beg + lane, lane < c1.n, perm, csr2csc, keep, alpha_used, dz, eg_ld);
        if (c0.first) {
            row_beg = c0.beg;
#pragma unroll
            for (int h = 0; h < H; ++h) trow[h] = 0.f;
        }
        const bool live = lane < c0.n;
        if (kind0 == 2) {
            // a pack of whole rows: segmented warp sums
            const int sa = live ? sa0 : 0, sb = live ? sb0 : lane;
            const bool lastf = live && lane == sb0;
            float o[H], dad[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const EgHead v = eg_head<H>(x0, h, live, slope, keep_scale);
                const float tt = seg_total(v.u, sa, sb, lane);
                o[h] = live ? v.sl * (v.u - v.alpha * tt) : 0.f;
                dad[h] = seg_total(o[h], sa, sb, lane);
            }
            if (live) eg_store<H>(x0, o, keep_scale, alpha_used, dz, eg_ld);
            const unsigned lastm = __ballot_sync(FULL, lastf);
            if (lastf) store_vecH<H>(da_dst + (c0.row + __popc(lastm & ((1u << lane) - 1u))) * int64_t(H), dad);
        } else if (c0.first && c0.last) {
            // the whole row is in registers
            float o[H], dad[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const EgHead v = eg_head<H>(x0, h, live, slope, keep_scale);
                const float tt = warp_sum(v.u);
                o[h] = live ? v.sl * (v.u - v.alpha * tt) : 0.f;
                dad[h] = warp_sum(o[h]);
            }
            if (live) eg_store<H>(x0, o, keep_scale, alpha_used, dz, eg_ld);
            if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
        } else {
            // a row of several chunks: accumulate t, then a second sweep over the row's slots
#pragma unroll
            for (int h = 0; h < H; ++h) trow[h] += warp_sum(eg_head<H>(x0, h, live, slope, keep_scale).u);
            if (c0.last) {
                float dad[H];
#pragma unroll
                for (int h = 0; h < H; ++h) dad[h] = 0.f;
                eg_sweep2<H, DROPOUT>(row_beg, c0.beg + c0.n, perm, csr2csc, keep, keep_scale, slope, trow, alpha_used, dz,
                                      eg_ld, dad, lane);
#pragma unroll
                for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
                if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
            }
        }
        if (!kind1) break;
        c0 = c1;
        kind0 = kind1;
        k0 = k1;
        sa0 = sa1;
        sb0 = sb1;
        x0 = x1;
    }
}

// hub rows, step 1: one warp per chunk -- partial t of the chunk
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_dst_eg_hub1(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                    const int32_t* __restrict__ csr2csc, gnnfd_hub_plan_t plan, float slope, KeepMask keep,
                    float keep_scale, const float* alpha_used, const float* dz, int64_t eg_ld,
                    float* __restrict__ part_t)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    float trow[H];
#pragma unroll
    for (int h = 0; h < H; ++h) trow[h] = 0.f;
    for (int base = beg; base < end; base += 32) {
        const bool live = base + lane < end;
        EgEdge<H> x;
        eg_load<H, DROPOUT>(x, base + lane, live, perm, csr2csc, keep, alpha_used, dz, eg_ld);
#pragma unroll
        for (int h = 0; h < H; ++h) trow[h] += warp_sum(eg_head<H>(x, h, live, slope, keep_scale).u);
    }
    if (lane == 0) store_vecH<H>(part_t + int64_t(c) * H, trow);
}

// hub rows, step 2: the row's total t (chunk order), second sweep, partial da_dst
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_dst_eg_hub2(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                    const int32_t* __restrict__ csr2csc, gnnfd_hub_plan_t plan, float slope, KeepMask keep,
                    float keep_scale, const float* __restrict__ t_total, float* alpha_used, float* dz, int64_t eg_ld,
                    float* __restrict__ part_dad)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    float t[H], dad[H];
    load_vecH<H>(t_total + int64_t(slot) * H, t);
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = 0.f;
    eg_sweep2<H, DROPOUT>(beg, end, perm, csr2csc, keep, keep_scale, slope, t, alpha_used, dz, eg_ld, dad, lane);
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
    if (lane == 0) store_vecH<H>(part_dad + int64_t(c) * H, dad);
}

template <class GE, bool DROPOUT>
static void launch_dst_eg(const gnnfd_graph_t* g, float slope, KeepMask keep, float ks, float* alpha_used, float* dz,
                          int64_t eg_ld, float* da_dst, float* part_t, float* part_dad, float* t_total, cudaStream_t st)
{
    constexpr int H = GE::H;
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + ROW_WARPS - 1) / ROW_WARPS);
    gat_bwd_dst_eg_items<H, DROPOUT><<<grid, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, g->items_dst, thr,
                                                                    slope, keep, ks, alpha_used, dz, eg_ld, da_dst);
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const unsigned gh = (unsigned)((pl.n_hub + ROW_WARPS - 1) / ROW_WARPS);
        const unsigned gc = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
        gat_bwd_dst_eg_hub1<H, DROPOUT><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, pl, slope, keep, ks,
                                                                     alpha_used, dz, eg_ld, part_t);
        gat_hub_chunk_sum<H, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_t, t_total);
        gat_bwd_dst_eg_hub2<H, DROPOUT><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, pl, slope, keep, ks,
                                                                     t_total, alpha_used, dz, eg_ld, part_dad);
        gat_hub_chunk_sum<H, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_dad, da_dst);
        g_launches += 4;
    }
}

template <class GE>
static int launch_bwd_dst_srcmajor(const gnnfd_graph_t* g, const void* xw_, const float* a_src, const float* a_dst,
                                   const float* rowmax, const float* rowsum, const float* d_out, float slope,
                                   const uint8_t* keep_mask, float p_drop, uint64_t seed, float* alpha_used, float* dz,
                                   float* da_dst, void* ws, size_t ws_bytes, cudaStream_t st)
{
    using XT = typename GE::XT;
    constexpr int H = GE::H;
    const XT* xw = reinterpret_cast<const XT*>(xw_);
    if (g->n_dst == 0) return GNNFD_OK;
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG,
                  "gat_bwd_dst: the graph has no work-item plan over rowptr (gnnfd_item_plan)");
    // two dense [E',H] arrays, or the halves of one interleaved [E',2H] buffer (dz == alpha_used + H)
    const int64_t eg_ld = (dz == alpha_used + H) ? 2 * H : H;
    float *part_t = nullptr, *part_dad = nullptr, *t_total = nullptr;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const size_t need = 2 * carve_bytes(size_t(pl.n_chunk) * H, 4) + carve_bytes(size_t(pl.n_hub) * H, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_bwd_dst: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        part_t = carve<float>(p, size_t(pl.n_chunk) * H);
        part_dad = carve<float>(p, size_t(pl.n_chunk) * H);
        t_total = carve<float>(p, size_t(pl.n_hub) * H);
    }
    if (g->n_edges > 0) {
        const int thr = g->hub_src.n_hub > 0 ? g->hub_src.threshold : INT_MAX;
        const unsigned grid = (unsigned)((g->items_src.n_items + DA_WARPS - 1) / DA_WARPS);
        gat_bwd_dalpha_src_rows<GE><<<grid, DA_THREADS, 0, st>>>(g->colptr, g->csc_row, xw, a_src, a_dst, rowmax, rowsum,
                                                                  d_out, g->items_src, thr, slope, alpha_used, dz, eg_ld);
        g_launches += 1;
        if (g->hub_src.n_hub > 0) {
            const unsigned gc = (unsigned)((g->hub_src.n_chunk + DA_WARPS - 1) / DA_WARPS);
            gat_bwd_dalpha_src_hub<GE><<<gc, DA_THREADS, 0, st>>>(g->colptr, g->csc_row, xw, a_src, a_dst, rowmax,
                                                                   rowsum, d_out, g->hub_src, slope, alpha_used, dz, eg_ld);
            g_launches += 1;
        }
    }
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    if (p_drop > 0.f)
        launch_dst_eg<GE, true>(g, slope, keep, ks, alpha_used, dz, eg_ld, da_dst, part_t, part_dad, t_total, st);
    else
        launch_dst_eg<GE, false>(g, slope, keep, ks, alpha_used, dz, eg_ld, da_dst, part_t, part_dad, t_total, st);
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

// The two-pass backward applies to the head mean on a graph whose CSC positions are the edge-gradient slots
// (not the indirect multi-GPU receive layout) and whose sources and destinations are one node set.
bool gat_bwd_dst_srcmajor_applies(const gnnfd_graph_t* g, int concat)
{
    return !concat && !g->edge_grads_indirect && g->n_src == g->n_dst && g->colptr && g->csc_row &&
           g->items_src.n_items > 0 && g->items_src.item_start;
}

int gat_bwd_dst_srcmajor(const gnnfd_graph_t* g, const void* xw, int xw_dtype, int H, int C, const float* a_src,
                         const float* a_dst, const float* rowmax, const float* rowsum, const float* d_out,
                         float negative_slope, const uint8_t* keep_mask, float p_drop, uint64_t seed, float* alpha_used,
                         float* dz, float* da_dst, void* ws, size_t ws_bytes, cudaStream_t st)
{
    if (H == 8 && C == 64 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst_srcmajor<Geo<8, 64, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope,
                                                          keep_mask, p_drop, seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_BF16)
        return launch_bwd_dst_srcmajor<Geo<8, 64, __nv_bfloat16>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out,
                                                                  negative_slope, keep_mask, p_drop, seed, alpha_used, dz,
                                                                  da_dst, ws, ws_bytes, st);
    if (H == 4 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst_srcmajor<Geo<4, 32, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope,
                                                          keep_mask, p_drop, seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_bwd_dst: (heads=%d, out_channels=%d, dtype=%d) is not built", H, C,
                  xw_dtype);
    return GNNFD_ERR_UNSUPPORTED;
}

}  // namespace gnnfd
