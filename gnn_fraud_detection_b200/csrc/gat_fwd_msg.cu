// (3b) forward, source-major form for the head mean (concat = False): three passes, no per-edge feature-row gather.
//
// With the head mean and known row statistics, alpha[e,h] is a per-edge scalar and
//     out[i] = epilogue( sum_{e -> i} v_e ),   v_e = (1/H) sum_h alpha_used[e,h] * xw[j,h,:]   (one C-float row)
// so the 2 KB row xw[j] is needed once per SOURCE, not once per edge:
//   pass A (CSR; gat_fwd_alpha_items / _hub_stats / _hub_merge / _hub_write): the attention pass of gat_alpha.cuh --
//            exact rowmax / rowsum and alpha_used [E',H] at the CSR position, dropout applied, formed with edge_alpha
//            from the final statistics (the expression the backward evaluates).  Gathers only a_src[col[e]].
//   pass B (CSC; gat_fwd_msg_src_stream / _hub): one warp streams the out-edges of one work item in CSC order, across
//            source-row boundaries, as tasks of <= 32 edges of one source row (the structure of the backward's
//            gat_bwd_dalpha_src_stream).  xw[j] goes into one of MS_XROWS row slots when a task starts a new source
//            row, each task's alpha_used[csc_eid[p]] vectors into a per-warp ring (16-byte cp.async, one commit group
//            per task), so later tasks' loads are in flight while the current one is reduced.  Per edge every lane does
//            the FMAs of its heads, a shfl_xor butterfly folds the head groups, and v_e goes to CSR position csc_eid[p]
//            of an [E',C] fp32 buffer as full-line stores.  Hub sources are split by the hub_src plan (_hub); every
//            output is per edge, so no merge.
//   pass C (CSR; gat_fwd_sum_items / _hub / _hub_merge): out[i] = sum of the row's v_e in CSR edge order, one
//            coalesced C-float load per edge, then the row epilogue (bias, folded BatchNorm, activation, residual).
//            Hub rows are summed in hub_dst chunks whose partials are added in chunk order: deterministic, no atomics.
// Per edge this moves ~4 + 32 + 32 B (A), ~4 + 32 + 4*C B plus D*sizeof(xw) per source (B) and 4*C B (C), against
// D*sizeof(xw) + ~36 B per edge for the gather kernels.  The concat forward keeps the gather kernels: its message would
// be the whole D-element row.
#include "gat_alpha.cuh"
#include "gat_phase_fwd.cuh"

#include <atomic>
#include <climits>
#include <cstdlib>

namespace gnnfd {
extern std::atomic<long long> g_launches;
bool gat_srcmajor_applies(const gnnfd_graph_t* g, int concat);   // gat_bwd_dalpha.cu

constexpr int MS_WARPS = 4;                  // warps per CTA in pass B
constexpr int MS_THREADS = MS_WARPS * 32;
constexpr int MS_RING = 64;                  // alpha vectors per warp (pass B stream): two whole 32-edge tasks
constexpr int MS_XROWS = 4;                  // xw row slots per warp (pass B stream)
constexpr int MS_TASKS = 8;                  // tasks in flight per warp at most (cp.async groups)
constexpr int SUM_WARPS = 8;                 // warps per CTA in pass C
constexpr int SUM_THREADS = SUM_WARPS * 32;

__device__ __forceinline__ void ms_cp_async16(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(st_smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void ms_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most n of this thread's commit groups are pending (n < MS_TASKS)
__device__ __forceinline__ void ms_cp_async_wait_pending(int n)
{
    switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
    }
}
static_assert(MS_TASKS <= 8 && MS_TASKS <= 32, "ms_cp_async_wait_pending covers 8 groups; one lane holds each task");
static_assert(MS_RING >= 32, "a task of 32 edges must fit the alpha ring, or the stream could never issue it");

// ---------------------------------------------------------------------------------------------------------
// pass A: the attention pass (gat_alpha.cuh, PROJ = true)
// ---------------------------------------------------------------------------------------------------------
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_fwd_alpha_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
                    const float* __restrict__ a_dst, gnnfd_item_plan_t items, int hub_threshold, float slope, AlphaOut out,
                    float* __restrict__ rowmax, float* __restrict__ rowsum)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * ROW_WARPS + warp;
    if (item >= items.n_items) return;
    alpha_items_body<H, true, DROPOUT>(rowptr, col, a_src, a_dst, items.item_start[item], items.item_start[item + 1],
                                             hub_threshold, slope, out, rowmax, rowsum, lane);
}
template <int H>
__global__ void __launch_bounds__(ROW_THREADS)
gat_fwd_alpha_hub_stats(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
                        const float* __restrict__ a_dst, gnnfd_hub_plan_t plan, float slope, float* __restrict__ part_ms)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    alpha_hub_stats_body<H>(rowptr, col, a_src, a_dst, plan, c, slope, part_ms, lane);
}
template <int H>
__global__ void gat_fwd_alpha_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part_ms, float* __restrict__ rowmax,
                                        float* __restrict__ rowsum)
{
    if (threadIdx.x >= H) return;
    alpha_hub_merge_body<H>(plan, blockIdx.x, threadIdx.x, part_ms, rowmax, rowsum);
}
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_fwd_alpha_hub_write(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
                        const float* __restrict__ a_dst, gnnfd_hub_plan_t plan, float slope, const float* __restrict__ rowmax,
                        const float* __restrict__ rowsum, AlphaOut out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * ROW_WARPS + warp;
    if (c >= plan.n_chunk) return;
    alpha_hub_write_body<H, true, DROPOUT>(rowptr, col, a_src, a_dst, plan, c, slope, rowmax, rowsum, out, lane);
}

// ---------------------------------------------------------------------------------------------------------
// pass B: source-major messages
// ---------------------------------------------------------------------------------------------------------
// copies the alpha_used vectors of edges [eid_0 .. eid_{n-1}] (lane l holds eid_l) into the ring slots
// (first + r) % MS_RING: H/4 lanes per vector, 16 B each
template <int H>
__device__ __forceinline__ void copy_alpha(float* al_s, int first, int n, int eid, const float* __restrict__ alpha,
                                           int lane)
{
    constexpr int LPV = H / 4, VPI = 32 / LPV;
    const int sub = lane / LPV, c4 = 4 * (lane % LPV);
    for (int r = 0; r < n; r += VPI) {
        const int er = __shfl_sync(FULL, eid, (r + sub) & 31);
        if (r + sub < n) ms_cp_async16(al_s + ((first + r + sub) % MS_RING) * H + c4, alpha + int64_t(er) * H + c4);
    }
}
// v_e of one edge against the xw row v (slot layout) and its alpha vector al (shared memory), stored at row eid of vout
template <class GE>
__device__ __forceinline__ void msg_edge(const float (&v)[GE::NS][GE::VW], const float* al, int64_t eid,
                                         float* __restrict__ vout, int lane)
{
    constexpr int NS = GE::NS, VW = GE::VW, HP = GE::HP, G = GE::G, C = GE::C, H = GE::H;
    const int sub = lane / G;
    float r[VW];
#pragma unroll
    for (int k = 0; k < VW; ++k) r[k] = 0.f;
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const float a = al[q * HP + sub];
#pragma unroll
        for (int k = 0; k < VW; ++k) r[k] = fmaf(a, v[q][k], r[k]);
    }
#pragma unroll
    for (int k = 0; k < VW; ++k)
#pragma unroll
        for (int o = G; o < 32; o <<= 1) r[k] += __shfl_xor_sync(FULL, r[k], o);
    if (lane < G) {                           // lane l < G holds channels [VW*l, VW*l + VW)
#pragma unroll
        for (int k = 0; k < VW; k += 4)
            stg_stream(reinterpret_cast<float4*>(vout + eid * C + VW * lane + k),
                       make_float4(r[k] * (1.f / H), r[k + 1] * (1.f / H), r[k + 2] * (1.f / H), r[k + 3] * (1.f / H)));
    }
}

// per-warp shared memory of the pass-B stream
template <class GE>
struct MsGeo {
    static constexpr int AL_BYTES = MS_RING * GE::H * 4;
    static constexpr int XROW_BYTES = GE::D * int(sizeof(typename GE::XT));
    static constexpr int X_BYTES = MS_XROWS * XROW_BYTES;
    static constexpr int EID_BYTES = MS_RING * 4;
    static constexpr int WARP_BYTES = ((X_BYTES + AL_BYTES + EID_BYTES + 127) / 128) * 128;
    static constexpr int CTA_BYTES = MS_WARPS * WARP_BYTES;
};

// one warp per edge-balanced work item over colptr (a run of whole source rows); hub rows are left to _hub.
// A task is a chunk of <= 32 out-edges of one source row (ChunkCursor over colptr); it is issued once its edges fit
// the alpha ring, a task slot is free and, if it starts a new source row, an xw slot is free.  Lane k % MS_TASKS holds
// task k as (n | new-row flag | xw slot).
template <class GE>
__global__ void __launch_bounds__(MS_THREADS, 4)
gat_fwd_msg_src_stream(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_eid,
                       const typename GE::XT* __restrict__ xw, const float* __restrict__ alpha, gnnfd_item_plan_t items,
                       int hub_threshold, float* __restrict__ vout)
{
    using SG = MsGeo<GE>;
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW;
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * MS_WARPS + warp;
    if (item >= items.n_items) return;
    uint8_t* base = smem + warp * SG::WARP_BYTES;
    uint8_t* x_s = base;
    float* al_s = reinterpret_cast<float*>(base + SG::X_BYTES);
    int* eid_s = reinterpret_cast<int*>(base + SG::X_BYTES + SG::AL_BYTES);

    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    auto no_empty = [](int) {};
    int nj = 0, nbeg = 0, nn = 0;              // the next task not yet issued
    bool nfirst = false, nlast = false;
    bool have = cur.next(colptr, nj, nbeg, nn, nfirst, nlast, no_empty);
    int e_issued = 0, e_done = 0;              // edges through the alpha ring
    int t_issued = 0, t_done = 0;              // tasks
    int x_issued = 0, x_done = 0;              // xw rows
    int task = 0;                              // this lane's entry of the task queue
    auto issue = [&]() {
        while (have && e_issued - e_done + nn <= MS_RING && t_issued - t_done < MS_TASKS &&
               (!nfirst || x_issued - x_done < MS_XROWS)) {
            const int eid = lane < nn ? csc_eid[nbeg + lane] : 0;
            if (lane < nn) eid_s[(e_issued + lane) % MS_RING] = eid;
            copy_alpha<H>(al_s, e_issued, nn, eid, alpha, lane);
            const int xs = x_issued % MS_XROWS;
            if (nfirst) {
                const uint8_t* src = reinterpret_cast<const uint8_t*>(xw + int64_t(nj) * GE::D);
#pragma unroll
                for (int q = 0; q < NS; ++q)
                    ms_cp_async16(x_s + xs * SG::XROW_BYTES + (lane + 32 * q) * 16, src + (lane + 32 * q) * 16);
                ++x_issued;
            }
            ms_cp_async_commit();
            if (lane == t_issued % MS_TASKS) task = nn | (int(nfirst) << 6) | (xs << 7);
            e_issued += nn;
            ++t_issued;
            have = cur.next(colptr, nj, nbeg, nn, nfirst, nlast, no_empty);
        }
    };
    issue();
    float v[NS][VW];                           // xw row of the current source, slot layout
    while (t_done < t_issued) {
        ms_cp_async_wait_pending(t_issued - t_done - 1);
        __syncwarp();
        const int tk = __shfl_sync(FULL, task, t_done % MS_TASKS);
        const int n = tk & 63;
        if (tk & 64) {
#pragma unroll
            for (int q = 0; q < NS; ++q) lds_slot(x_s + (tk >> 7) * SG::XROW_BYTES, q, lane, v[q]);
            ++x_done;
        }
        for (int t = 0; t < n; ++t) {
            const int slot = (e_done + t) % MS_RING;
            msg_edge<GE>(v, al_s + slot * H, eid_s[slot], vout, lane);
        }
        __syncwarp();                          // the task's slots are read before they are refilled
        e_done += n;
        ++t_done;
        issue();
    }
}

// one warp per chunk of a hub source row: xw[j] in registers, per 32 edges the alpha vectors through shared memory
template <class GE>
__global__ void __launch_bounds__(MS_THREADS, 6)
gat_fwd_msg_src_hub(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_eid,
                    const typename GE::XT* __restrict__ xw, const float* __restrict__ alpha, gnnfd_hub_plan_t plan,
                    float* __restrict__ vout)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW;
    __shared__ __align__(16) float al_sh[MS_WARPS][32 * H];
    __shared__ int eid_sh[MS_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * MS_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t j = plan.hub_row[slot];
    const int beg = colptr[j] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(colptr[j + 1], beg + plan.chunk);
    float v[NS][VW];
#pragma unroll
    for (int q = 0; q < NS; ++q) load_slot(xw + j * GE::D, q, lane, v[q]);
    for (int b = beg; b < end; b += 32) {
        const int n = min(32, end - b);
        if (lane < n) {
            const int eid = csc_eid[b + lane];
            float a[H];
            load_vecH<H>(alpha + int64_t(eid) * H, a);
            store_vecH<H>(&al_sh[warp][lane * H], a);
            eid_sh[warp][lane] = eid;
        }
        __syncwarp();
        for (int t = 0; t < n; ++t) msg_edge<GE>(v, &al_sh[warp][t * H], eid_sh[warp][t], vout, lane);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// pass C: row sums of the messages, then the row epilogue
// ---------------------------------------------------------------------------------------------------------
// sum of the C-float rows [beg, end) of v, in edge order within each of the RPW lane groups (edge e goes to group
// (e - beg) % RPW, the groups are added in a fixed order); lanes l < C/4 return channels [4l, 4l+4)
template <int C>
__device__ __forceinline__ float4 sum_rows(const float* __restrict__ v, int beg, int end, int lane)
{
    constexpr int LPR = C / 4, RPW = 32 / LPR, U = 4;
    const int sub = lane / LPR, c4 = 4 * (lane % LPR);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e0 = beg; e0 < end; e0 += RPW * U) {
        float4 t[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * RPW + sub;
            t[u] = e < end ? ldg_stream(reinterpret_cast<const float4*>(v + int64_t(e) * C + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            acc.x += t[u].x; acc.y += t[u].y; acc.z += t[u].z; acc.w += t[u].w;
        }
    }
#pragma unroll
    for (int o = LPR; o < 32; o <<= 1) {
        acc.x += __shfl_xor_sync(FULL, acc.x, o);
        acc.y += __shfl_xor_sync(FULL, acc.y, o);
        acc.z += __shfl_xor_sync(FULL, acc.z, o);
        acc.w += __shfl_xor_sync(FULL, acc.w, o);
    }
    return acc;
}
template <int C>
__device__ __forceinline__ void sum_epilogue(int64_t i, float4 s, const EpiParams& ep, float* __restrict__ out, int lane)
{
    if (lane < C / 4) {
        const int c0 = 4 * lane;
        stg_stream(reinterpret_cast<float4*>(out + i * C + c0),
                   make_float4(epi_value(s.x, c0, i, C, ep), epi_value(s.y, c0 + 1, i, C, ep),
                               epi_value(s.z, c0 + 2, i, C, ep), epi_value(s.w, c0 + 3, i, C, ep)));
    }
}

// one warp per edge-balanced work item over rowptr; hub rows are left to _hub / _hub_merge
template <int C>
__global__ void __launch_bounds__(SUM_THREADS)
gat_fwd_sum_items(const int32_t* __restrict__ rowptr, const float* __restrict__ v, gnnfd_item_plan_t items,
                  int hub_threshold, EpiParams ep, float* __restrict__ out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * SUM_WARPS + warp;
    if (item >= items.n_items) return;
    const int r1 = items.item_start[item + 1];
    for (int i = items.item_start[item]; i < r1; ++i) {
        const int beg = rowptr[i], end = rowptr[i + 1];
        if (end - beg > hub_threshold) continue;
        sum_epilogue<C>(i, sum_rows<C>(v, beg, end, lane), ep, out, lane);
    }
}
// one warp per hub_dst chunk: its partial sum
template <int C>
__global__ void __launch_bounds__(SUM_THREADS)
gat_fwd_sum_hub(const int32_t* __restrict__ rowptr, const float* __restrict__ v, gnnfd_hub_plan_t plan,
                float* __restrict__ part)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * SUM_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c], i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    const float4 s = sum_rows<C>(v, beg, end, lane);
    if (lane < C / 4) *reinterpret_cast<float4*>(part + int64_t(c) * C + 4 * lane) = s;
}
// one warp per hub row: the chunk partials added in chunk order, then the row epilogue
template <int C>
__global__ void __launch_bounds__(SUM_THREADS)
gat_fwd_sum_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part, EpiParams ep, float* __restrict__ out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * SUM_WARPS + warp;
    if (slot >= plan.n_hub) return;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < C / 4)
        for (int c = plan.hub_chunk_ptr[slot]; c < plan.hub_chunk_ptr[slot + 1]; ++c) {
            const float4 p = *reinterpret_cast<const float4*>(part + int64_t(c) * C + 4 * lane);
            s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
        }
    sum_epilogue<C>(plan.hub_row[slot], s, ep, out, lane);
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
// GNNFD_FWD_SRCMAJOR=0 keeps the head-mean forward on the gather kernels (A/B runs)
static bool srcmajor_enabled()
{
    static const bool on = [] {
        const char* e = getenv("GNNFD_FWD_SRCMAJOR");
        return e ? atoi(e) != 0 : true;
    }();
    return on;
}
bool gat_fwd_srcmajor_applies(const gnnfd_graph_t* g, int concat) { return srcmajor_enabled() && gat_srcmajor_applies(g, concat); }

// workspace of the source-major form beyond the gather kernels' hub partials: alpha_used [E',H], v [E',C]
size_t gat_fwd_srcmajor_ws_bytes(const gnnfd_graph_t* g, int H, int C)
{
    return carve_bytes(size_t(g->n_edges) * H, 4) + carve_bytes(size_t(g->n_edges) * C, 4);
}

template <class GE, bool DROPOUT>
static void launch_alpha(const gnnfd_graph_t* g, const float* a_src, const float* a_dst, float slope, const AlphaOut& ao,
                         float* rowmax, float* rowsum, float* part_ms, cudaStream_t st)
{
    constexpr int H = GE::H;
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + ROW_WARPS - 1) / ROW_WARPS);
    gat_fwd_alpha_items<H, DROPOUT><<<grid, ROW_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, g->items_dst, thr, slope,
                                                                   ao, rowmax, rowsum);
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const unsigned gc = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
        gat_fwd_alpha_hub_stats<H><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, pl, slope, part_ms);
        gat_fwd_alpha_hub_merge<H><<<(unsigned)pl.n_hub, 32, 0, st>>>(pl, part_ms, rowmax, rowsum);
        gat_fwd_alpha_hub_write<H, DROPOUT><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, pl, slope, rowmax,
                                                                         rowsum, ao);
        g_launches += 3;
    }
}

template <class GE>
static int launch_fwd_srcmajor(const gnnfd_graph_t* g, const void* xw_, const float* a_src, const float* a_dst,
                               const EpiParams& ep, float slope, const uint8_t* keep_mask, float p_drop, uint64_t seed,
                               float* out, float* rowmax, float* rowsum, void* ws, size_t ws_bytes, cudaStream_t st)
{
    using XT = typename GE::XT;
    constexpr int H = GE::H, C = GE::C;
    const XT* xw = reinterpret_cast<const XT*>(xw_);
    if (g->n_dst == 0) return GNNFD_OK;
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG,
                  "gat_fwd: the graph has no work-item plan over rowptr (gnnfd_item_plan)");
    // the gather kernels' hub partials (reused here: chunk statistics of pass A, chunk sums of pass C), then the two
    // per-edge buffers
    const size_t nc = size_t(g->hub_dst.n_chunk);
    const size_t need = carve_bytes(nc * 2 * H, 4) + carve_bytes(nc * size_t(GE::D), 4) + gat_fwd_srcmajor_ws_bytes(g, H, C);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_fwd: workspace %zu < %zu", ws_bytes, need);
    char* p = reinterpret_cast<char*>(ws);
    float* part_ms = carve<float>(p, nc * 2 * H);
    float* part_sum = carve<float>(p, nc * size_t(GE::D));
    float* alpha = carve<float>(p, size_t(g->n_edges) * H);
    float* v = carve<float>(p, size_t(g->n_edges) * C);

    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    const AlphaOut ao{alpha, nullptr, g->perm, keep, ks};
    if (p_drop > 0.f) launch_alpha<GE, true>(g, a_src, a_dst, slope, ao, rowmax, rowsum, part_ms, st);
    else              launch_alpha<GE, false>(g, a_src, a_dst, slope, ao, rowmax, rowsum, part_ms, st);

    if (g->n_edges > 0) {
        constexpr int SMEM = MsGeo<GE>::CTA_BYTES;
        GNNFD_CUDA(cudaFuncSetAttribute(gat_fwd_msg_src_stream<GE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        const int thr = g->hub_src.n_hub > 0 ? g->hub_src.threshold : INT_MAX;
        const unsigned grid = (unsigned)((g->items_src.n_items + MS_WARPS - 1) / MS_WARPS);
        gat_fwd_msg_src_stream<GE><<<grid, MS_THREADS, SMEM, st>>>(g->colptr, g->csc_eid, xw, alpha, g->items_src, thr, v);
        g_launches += 1;
        if (g->hub_src.n_hub > 0) {
            const unsigned gc = (unsigned)((g->hub_src.n_chunk + MS_WARPS - 1) / MS_WARPS);
            gat_fwd_msg_src_hub<GE><<<gc, MS_THREADS, 0, st>>>(g->colptr, g->csc_eid, xw, alpha, g->hub_src, v);
            g_launches += 1;
        }
    }

    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + SUM_WARPS - 1) / SUM_WARPS);
    gat_fwd_sum_items<C><<<grid, SUM_THREADS, 0, st>>>(g->rowptr, v, g->items_dst, thr, ep, out);
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const unsigned gc = (unsigned)((pl.n_chunk + SUM_WARPS - 1) / SUM_WARPS);
        const unsigned gh = (unsigned)((pl.n_hub + SUM_WARPS - 1) / SUM_WARPS);
        gat_fwd_sum_hub<C><<<gc, SUM_THREADS, 0, st>>>(g->rowptr, v, pl, part_sum);
        gat_fwd_sum_hub_merge<C><<<gh, SUM_THREADS, 0, st>>>(pl, part_sum, ep, out);
        g_launches += 2;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int gat_fwd_srcmajor(const gnnfd_graph_t* g, const void* xw, int xw_dtype, int H, int C, const float* a_src,
                     const float* a_dst, const EpiParams& ep, float negative_slope, const uint8_t* keep_mask, float p_drop,
                     uint64_t seed, float* out, float* rowmax, float* rowsum, void* ws, size_t ws_bytes, cudaStream_t st)
{
    if (H == 8 && C == 64 && xw_dtype == GNNFD_F32)
        return launch_fwd_srcmajor<Geo<8, 64, float>>(g, xw, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, seed, out,
                                                      rowmax, rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 64 && xw_dtype == GNNFD_BF16)
        return launch_fwd_srcmajor<Geo<8, 64, __nv_bfloat16>>(g, xw, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, seed,
                                                              out, rowmax, rowsum, ws, ws_bytes, st);
    if (H == 4 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_fwd_srcmajor<Geo<4, 32, float>>(g, xw, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, seed, out,
                                                      rowmax, rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_fwd_srcmajor<Geo<8, 32, float>>(g, xw, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, seed, out,
                                                      rowmax, rowsum, ws, ws_bytes, st);
    if (H == 8 && C == 128 && xw_dtype == GNNFD_F32)
        return launch_fwd_srcmajor<Geo<8, 128, float>>(g, xw, a_src, a_dst, ep, negative_slope, keep_mask, p_drop, seed, out,
                                                       rowmax, rowsum, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_fwd: (heads=%d, out_channels=%d, dtype=%d) is not built; "
                  "available: (8,64,f32), (8,64,bf16), (8,32,f32), (8,128,f32), (4,32,f32)", H, C, xw_dtype);
    return GNNFD_ERR_UNSUPPORTED;
}

}  // namespace gnnfd
