// (4a) backward, dst-major pass for the head mean (concat = False): two passes, no per-edge feature-row gather.
//
// d_alpha[e,h] = <dO[i]/H, xw[j,h,:]> needs no row reduction, and with the head mean dO[i] is one C-float row
// shared by all heads.  So d_alpha is computed SOURCE-major, where xw[j] is read once, and only the 256 B dO[i] row
// is gathered per edge; the row reductions follow in a second pass that reads no features.
//   pass 1 (CSC; gat_bwd_dalpha_src_stream / _hub): one warp streams the out-edges of one work item in CSC order,
//            across source-row boundaries, as tasks of <= 32 edges of one source row.  Each task's dO rows go into a
//            per-warp ring of DA_RING row slots and, when the task starts a new source row, xw[j] into one of
//            DA_XROWS row slots (16-byte cp.async, 16 lanes per dO row, one commit group per task), so the next
//            tasks' rows are in flight while the current one is reduced; a_src[j] rides in the xw row slot.  Per
//            edge 16 FMAs and phase B's butterfly give d_alpha with phase B's arithmetic; the record
//            {d_alpha, a_src[j]} is stored at the edge's CSR position csc_eid[p] of an [E',2H] workspace buffer.
//            Sources above the hub threshold are split by the hub_src plan (_hub, one warp per chunk); every output
//            is per edge, so the chunks need no merge.
//   pass 2 (CSR; gat_bwd_dst_eg_items / _hub1 / _hub2): the chunk, pack and hub_dst schedule of the gather kernels,
//            lane = edge.  It reads only contiguous streams -- the record, csr2csc (and perm) over the edge range, the
//            row statistics over the row range -- with the next chunk in flight, recomputes alpha with edge_alpha from
//            the record's a_src, and forms u = alpha * d_alpha * keep, t, dz and da_dst with the same warp sums in the
//            same order as the gather kernels.  (alpha_used, dz) go to the edge's source-major slot csr2csc[e], each
//            32-B vector (H = 8) as one 256-bit store, so that a lane writes whole sectors at its random address.
// Per edge this moves ~4 + 4 + 256 + 64 B (pass 1) and ~64 + 4 + 64 B (pass 2).  The record is 4H B wider than a bare
// d_alpha so that pass 2 has no dependent gather (col[e] -> a_src[col[e]]).  alpha_used equals the gather kernels' bit
// for bit; dz and da_dst differ in the last bits on rows longer than one chunk, where the gather kernels recompute
// alpha for the second sweep with a contracted multiply-add.
#include "gat_stream.cuh"
#include "gat_phase_bwd.cuh"

#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;

constexpr int DA_WARPS = 4;                  // warps per CTA in pass 1
constexpr int DA_THREADS = DA_WARPS * 32;
constexpr int DA_RING = 32;                  // dO row slots per warp (pass 1 stream): a whole 32-edge task fits
constexpr int DA_XROWS = 2;                  // xw row slots per warp (pass 1 stream)
constexpr int DA_TASKS = 8;                  // tasks in flight per warp at most (cp.async groups)
// warps per CTA of the hub kernel, which stages 32 dO rows per warp in static shared memory: 8 KB per warp at C = 64;
// at C = 128 two warps keep the 16 KB per warp under the 48 KB static limit
template <class GE>
constexpr int da_hub_warps()
{
    return GE::C > 64 ? 2 : DA_WARPS;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(st_smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most n of this thread's commit groups are pending (n < DA_TASKS)
__device__ __forceinline__ void cp_async_wait_pending(int n)
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
static_assert(DA_TASKS <= 8 && DA_TASKS <= 32, "cp_async_wait_pending covers 8 groups; one lane holds each task");
static_assert(DA_RING >= 32, "a task of 32 edges must fit the dO ring, or the stream could never issue it");
constexpr uint32_t NEG_FLAG = 0x80000000u;   // sign bit of alpha held in registers: LeakyReLU-negative logit

// ---------------------------------------------------------------------------------------------------------
// pass 1: source-major d_alpha
// ---------------------------------------------------------------------------------------------------------
// copies dO rows [i_0 .. i_{n-1}] (lane l holds i_l) into the slots (first + r) % SLOTS: C/4 lanes per row, 16 B
// each, so every instruction moves 32/(C/4) whole rows
template <class GE, int SLOTS>
__device__ __forceinline__ void copy_do_rows(float* do_s, int first, int n, int i, const float* __restrict__ d_out,
                                             int lane)
{
    constexpr int C = GE::C, LPR = C / 4, RPI = 32 / LPR;
    const int sub = lane / LPR, c4 = 4 * (lane % LPR);
    for (int r = 0; r < n; r += RPI) {
        const int ir = __shfl_sync(FULL, i, (r + sub) & 31);
        if (r + sub < n) cp_async16(do_s + ((first + r + sub) % SLOTS) * C + c4, d_out + int64_t(ir) * C + c4);
    }
}
// d_alpha of one edge against the dO row staged at g_row: phase B's FMAs and butterfly, result in dal_t[0..H)
template <class GE>
__device__ __forceinline__ void dalpha_edge(const float (&v)[GE::NS][GE::VW], const float* g_row, float* dal_t, int lane)
{
    constexpr int NS = GE::NS, VW = GE::VW, C = GE::C, H = GE::H;
    static_assert((32 * VW) % C == 0, "every slot of a lane must see the same dO channels");
    const int cm = (VW * lane) % C;          // dO channels of this lane's slots
    const float sc = 1.f / H;
    float g[VW];
#pragma unroll
    for (int k = 0; k < VW; k += 4) {
        const float4 tv = *reinterpret_cast<const float4*>(g_row + cm + k);
        g[k] = tv.x * sc; g[k + 1] = tv.y * sc; g[k + 2] = tv.z * sc; g[k + 3] = tv.w * sc;
    }
    float d[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        d[q] = 0.f;
#pragma unroll
        for (int k = 0; k < VW; ++k) d[q] = fmaf(g[k], v[q][k], d[q]);
    }
    dalpha_reduce<GE>(d, dal_t, lane);
}

// one edge's record {d_alpha[0..H) from shared memory, a_src[j][0..H) of its source} to its CSR position
template <int H>
__device__ __forceinline__ void store_record(float* __restrict__ dst, const float* dal_t, const float (&as)[H])
{
    float dal[H];
#pragma unroll
    for (int k = 0; k < H / 4; ++k) {
        const float4 d4 = *reinterpret_cast<const float4*>(dal_t + 4 * k);
        dal[4 * k] = d4.x; dal[4 * k + 1] = d4.y; dal[4 * k + 2] = d4.z; dal[4 * k + 3] = d4.w;
    }
    store_vecH_wide<H>(dst, dal);
    store_vecH_wide<H>(dst + H, as);
}

// per-warp shared memory of the pass-1 stream
template <class GE>
struct DaGeo {
    static constexpr int DO_BYTES = DA_RING * GE::C * 4;
    static constexpr int XROW_BYTES = GE::D * int(sizeof(typename GE::XT));
    static constexpr int XSLOT_BYTES = XROW_BYTES + GE::H * 4;    // xw[j], then a_src[j]
    static constexpr int X_BYTES = DA_XROWS * XSLOT_BYTES;
    static constexpr int DAL_BYTES = 32 * GE::H * 4;
    static constexpr int EID_BYTES = DA_RING * 4;
    static constexpr int WARP_BYTES = ((DO_BYTES + X_BYTES + DAL_BYTES + EID_BYTES + 127) / 128) * 128;
    static constexpr int CTA_BYTES = DA_WARPS * WARP_BYTES;
};

// one warp per edge-balanced work item over colptr (a run of whole source rows); hub rows are left to _hub.
// A task is a chunk of <= 32 out-edges of one source row (ChunkCursor over colptr); it is issued once its edges fit
// the dO ring, a task slot is free and, if it starts a new source row, an xw slot is free.  Lane k % DA_TASKS holds
// task k as (n | new-row flag | xw slot).
template <class GE>
__global__ void __launch_bounds__(DA_THREADS, 4)
gat_bwd_dalpha_src_stream(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                          const int32_t* __restrict__ csc_eid, const typename GE::XT* __restrict__ xw,
                          const float* __restrict__ a_src, const float* __restrict__ d_out, gnnfd_item_plan_t items,
                          int hub_threshold, float* __restrict__ rec)
{
    using SG = DaGeo<GE>;
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, C = GE::C;
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * DA_WARPS + warp;
    if (item >= items.n_items) return;
    uint8_t* base = smem + warp * SG::WARP_BYTES;
    float* do_s = reinterpret_cast<float*>(base);
    uint8_t* x_s = base + SG::DO_BYTES;
    float* dal_s = reinterpret_cast<float*>(base + SG::DO_BYTES + SG::X_BYTES);
    int* eid_s = reinterpret_cast<int*>(base + SG::DO_BYTES + SG::X_BYTES + SG::DAL_BYTES);

    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    auto no_empty = [](int) {};
    int nj = 0, nbeg = 0, nn = 0;              // the next task not yet issued
    bool nfirst = false, nlast = false;
    bool have = cur.next(colptr, nj, nbeg, nn, nfirst, nlast, no_empty);
    int e_issued = 0, e_done = 0;              // edges through the dO ring
    int t_issued = 0, t_done = 0;              // tasks
    int x_issued = 0, x_done = 0;              // xw rows
    int task = 0;                              // this lane's entry of the task queue
    auto issue = [&]() {
        while (have && e_issued - e_done + nn <= DA_RING && t_issued - t_done < DA_TASKS &&
               (!nfirst || x_issued - x_done < DA_XROWS)) {
            const bool live = lane < nn;
            const int i = live ? csc_row[nbeg + lane] : 0;
            if (live) eid_s[(e_issued + lane) % DA_RING] = csc_eid[nbeg + lane];
            copy_do_rows<GE, DA_RING>(do_s, e_issued, nn, i, d_out, lane);
            const int xs = x_issued % DA_XROWS;
            if (nfirst) {
                const uint8_t* src = reinterpret_cast<const uint8_t*>(xw + int64_t(nj) * GE::D);
#pragma unroll
                for (int q = 0; q < NS; ++q)
                    cp_async16(x_s + xs * SG::XSLOT_BYTES + (lane + 32 * q) * 16, src + (lane + 32 * q) * 16);
                if (lane < H / 4)
                    cp_async16(x_s + xs * SG::XSLOT_BYTES + SG::XROW_BYTES + lane * 16,
                               a_src + int64_t(nj) * H + 4 * lane);
                ++x_issued;
            }
            cp_async_commit();
            if (lane == t_issued % DA_TASKS) task = nn | (int(nfirst) << 6) | (xs << 7);
            e_issued += nn;
            ++t_issued;
            have = cur.next(colptr, nj, nbeg, nn, nfirst, nlast, no_empty);
        }
    };
    issue();
    float v[NS][VW];                           // xw row of the current source, slot layout
    float as[H];                               // a_src of the current source
    while (t_done < t_issued) {
        cp_async_wait_pending(t_issued - t_done - 1);
        __syncwarp();
        const int tk = __shfl_sync(FULL, task, t_done % DA_TASKS);
        const int n = tk & 63;
        if (tk & 64) {
#pragma unroll
            for (int q = 0; q < NS; ++q) lds_slot(x_s + (tk >> 7) * SG::XSLOT_BYTES, q, lane, v[q]);
            const float* as_s = reinterpret_cast<const float*>(x_s + (tk >> 7) * SG::XSLOT_BYTES + SG::XROW_BYTES);
#pragma unroll
            for (int h = 0; h < H; ++h) as[h] = as_s[h];
            ++x_done;
        }
        for (int t = 0; t < n; ++t) dalpha_edge<GE>(v, do_s + ((e_done + t) % DA_RING) * C, dal_s + t * H, lane);
        __syncwarp();
        if (lane < n) store_record<H>(rec + int64_t(eid_s[(e_done + lane) % DA_RING]) * 2 * H, dal_s + lane * H, as);
        __syncwarp();                          // the task's slots are read before they are refilled
        e_done += n;
        ++t_done;
        issue();
    }
}

// one warp per chunk of a hub source row: xw[j] in registers, per 32 edges the dO rows staged with cp.async
template <class GE>
__global__ void __launch_bounds__(32 * da_hub_warps<GE>(), 6)
gat_bwd_dalpha_src_hub(const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_row,
                       const int32_t* __restrict__ csc_eid, const typename GE::XT* __restrict__ xw,
                       const float* __restrict__ a_src, const float* __restrict__ d_out, gnnfd_hub_plan_t plan,
                       float* __restrict__ rec)
{
    constexpr int H = GE::H, NS = GE::NS, VW = GE::VW, C = GE::C;
    constexpr int W = da_hub_warps<GE>();
    __shared__ __align__(16) float do_sh[W][32 * C];
    __shared__ __align__(16) float dal_sh[W][32 * H];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * W + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int64_t j = plan.hub_row[slot];
    const int beg = colptr[j] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(colptr[j + 1], beg + plan.chunk);
    float* do_s = do_sh[warp];
    float* dal_s = dal_sh[warp];
    float v[NS][VW], as[H];
#pragma unroll
    for (int q = 0; q < NS; ++q) load_slot(xw + j * GE::D, q, lane, v[q]);
    load_vecH<H>(a_src + j * H, as);
    for (int base = beg; base < end; base += 32) {
        const int n = min(32, end - base);
        const bool live = lane < n;
        const int i = live ? csc_row[base + lane] : 0;
        const int eid = live ? csc_eid[base + lane] : 0;
        copy_do_rows<GE, 32>(do_s, 0, n, i, d_out, lane);
        cp_async_commit();
        cp_async_wait_pending(0);
        __syncwarp();
        for (int t = 0; t < n; ++t) dalpha_edge<GE>(v, do_s + t * C, dal_s + t * H, lane);
        __syncwarp();
        if (live) store_record<H>(rec + int64_t(eid) * 2 * H, dal_s + lane * H, as);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// pass 2: feature-free dst-major reductions
// ---------------------------------------------------------------------------------------------------------
// one edge of pass 2, lane = edge
template <int H>
struct EgEdge {
    float a[H], d[H];      // alpha with the LeakyReLU-negative flag, d_alpha
    int pos;               // source-major slot
    unsigned keep;         // dropout keep bits
};
// pass 2 reads an edge in two steps so that the next chunk's loads are in flight while the current chunk is reduced:
// eg_fetch (the record {d_alpha, a_src[j]}, csr2csc and perm of dst-sorted edge e -- all contiguous over a chunk),
// then eg_finish (the row statistics of its destination row, alpha recomputed as phase A does, the keep bits)
template <int H>
struct EgRaw {
    int pos, pe;
    float d[H], as[H];
};
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_fetch(EgRaw<H>& r, int e, bool live, const int32_t* __restrict__ perm,
                                         const int32_t* __restrict__ csr2csc, const float* __restrict__ rec)
{
    r.pos = r.pe = 0;
#pragma unroll
    for (int h = 0; h < H; ++h) r.d[h] = r.as[h] = 0.f;
    if (!live) return;
    r.pos = csr2csc[e];
    load_vecH<H>(rec + int64_t(e) * 2 * H, r.d);
    load_vecH<H>(rec + int64_t(e) * 2 * H + H, r.as);
    if (DROPOUT) r.pe = perm[e];
}
// the items kernel holds the next chunk in shared memory rather than in registers: eg_fetch_async copies it (lane =
// edge, every lane copies and later reads only its own entries, one commit group per chunk), eg_take reads it back
template <int H>
struct EgStage {
    float rec[32][2 * H];
    int pos[32], pe[32];
};
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(st_smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_fetch_async(EgStage<H>& s, int e, bool live, const int32_t* __restrict__ perm,
                                               const int32_t* __restrict__ csr2csc, const float* __restrict__ rec,
                                               int lane)
{
    if (live) {
#pragma unroll
        for (int k = 0; k < H / 2; ++k) cp_async16(&s.rec[lane][4 * k], rec + int64_t(e) * 2 * H + 4 * k);
        cp_async4(&s.pos[lane], csr2csc + e);
        if (DROPOUT) cp_async4(&s.pe[lane], perm + e);
    }
    cp_async_commit();
}
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_take(EgRaw<H>& r, const EgStage<H>& s, bool live, int lane)
{
    r.pos = r.pe = 0;
#pragma unroll
    for (int h = 0; h < H; ++h) r.d[h] = r.as[h] = 0.f;
    if (!live) return;
#pragma unroll
    for (int k = 0; k < H / 4; ++k) {
        const float4 d4 = *reinterpret_cast<const float4*>(&s.rec[lane][4 * k]);
        const float4 a4 = *reinterpret_cast<const float4*>(&s.rec[lane][H + 4 * k]);
        r.d[4 * k] = d4.x; r.d[4 * k + 1] = d4.y; r.d[4 * k + 2] = d4.z; r.d[4 * k + 3] = d4.w;
        r.as[4 * k] = a4.x; r.as[4 * k + 1] = a4.y; r.as[4 * k + 2] = a4.z; r.as[4 * k + 3] = a4.w;
    }
    r.pos = s.pos[lane];
    if (DROPOUT) r.pe = s.pe[lane];
}
// the row statistics of destination row i into L1, so that eg_finish of the next chunk does not wait on DRAM for them
template <int H>
__device__ __forceinline__ void eg_prefetch_row(int64_t i, const float* __restrict__ a_dst,
                                                const float* __restrict__ rowmax, const float* __restrict__ rowsum)
{
    asm volatile("prefetch.global.L1 [%0];" ::"l"(a_dst + i * H));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(rowmax + i * H));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(rowsum + i * H));
}
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_finish(EgEdge<H>& x, const EgRaw<H>& r, bool live, int64_t row,
                                          const float* __restrict__ a_dst, const float* __restrict__ rowmax,
                                          const float* __restrict__ rowsum, float slope, KeepMask keep)
{
    x.pos = r.pos;
    x.keep = 0xffu;
#pragma unroll
    for (int h = 0; h < H; ++h) {
        x.a[h] = 0.f;
        x.d[h] = r.d[h];
    }
    if (!live) return;
    RowStat<H> st;
    load_row_stat<H>(st, row, a_dst, rowmax, rowsum);
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float z = r.as[h] + st.adst[h];
        x.a[h] = __uint_as_float(__float_as_uint(edge_alpha(z, slope, st.m[h], st.inv[h])) | (z > 0.f ? 0u : NEG_FLAG));
    }
    if (DROPOUT) x.keep = keep.bits(r.pe, H);
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
// the final slot: alpha_used = alpha * keep, dz.  eg_ld < 0 marks 32-byte-aligned slots (stored with store_vecH_wide)
// of stride -eg_ld
template <int H>
__device__ __forceinline__ void eg_store(const EgEdge<H>& x, const float (&o)[H], float keep_scale, float* alpha_used,
                                         float* dz, int64_t eg_ld)
{
    float au[H];
#pragma unroll
    for (int h = 0; h < H; ++h)
        au[h] = __uint_as_float(__float_as_uint(x.a[h]) & ~NEG_FLAG) * ((x.keep >> h) & 1 ? keep_scale : 0.f);
    if (eg_ld < 0) {
        store_vecH_wide<H>(alpha_used - int64_t(x.pos) * eg_ld, au);
        store_vecH_wide<H>(dz - int64_t(x.pos) * eg_ld, o);
    } else {
        store_vecH<H>(alpha_used + int64_t(x.pos) * eg_ld, au);
        store_vecH<H>(dz + int64_t(x.pos) * eg_ld, o);
    }
}
// second sweep of a row (or hub chunk) whose t is known: the edges are read again, one chunk ahead as in the first
// sweep; alpha_used and dz go to the slots, da_dst is summed lane-locally
template <int H, bool DROPOUT>
__device__ __forceinline__ void eg_sweep2(int64_t row, int beg, int end, const int32_t* __restrict__ perm,
                                          const int32_t* __restrict__ csr2csc, const float* __restrict__ a_dst,
                                          const float* __restrict__ rowmax, const float* __restrict__ rowsum,
                                          KeepMask keep, float keep_scale, float slope, const float (&t)[H],
                                          const float* __restrict__ rec, float* alpha_used, float* dz, int64_t eg_ld,
                                          float (&dad)[H], int lane)
{
    EgRaw<H> r0, r1;
    eg_fetch<H, DROPOUT>(r0, beg + lane, beg + lane < end, perm, csr2csc, rec);
    for (int base = beg; base < end; base += 32) {
        const bool more = base + 32 < end;
        if (more) eg_fetch<H, DROPOUT>(r1, base + 32 + lane, base + 32 + lane < end, perm, csr2csc, rec);
        if (base + lane < end) {
            EgEdge<H> x;
            eg_finish<H, DROPOUT>(x, r0, true, row, a_dst, rowmax, rowsum, slope, keep);
            float o[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const EgHead v = eg_head<H>(x, h, true, slope, keep_scale);
                o[h] = v.sl * (v.u - v.alpha * t[h]);
                dad[h] += o[h];
            }
            eg_store<H>(x, o, keep_scale, alpha_used, dz, eg_ld);
        }
        if (more) r0 = r1;
    }
}

// one warp per edge-balanced work item over rowptr; the chunk and pack sequence of gat_bwd_dst_items_pack, with the
// next chunk's records (eg_fetch_async, into a per-warp shared-memory stage) and row statistics in flight while the
// current one is finished and reduced
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS, 2)
gat_bwd_dst_eg_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                     const int32_t* __restrict__ csr2csc, const float* __restrict__ a_dst,
                     const float* __restrict__ rowmax, const float* __restrict__ rowsum, const float* __restrict__ rec,
                     gnnfd_item_plan_t items, int hub_threshold, float slope, KeepMask keep, float keep_scale,
                     float* alpha_used, float* dz, int64_t eg_ld, float* __restrict__ da_dst)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * ROW_WARPS + warp;
    __shared__ __align__(16) EgStage<H> stage_sh[ROW_WARPS][2];
    if (item >= items.n_items) return;
    EgStage<H>* stage = stage_sh[warp];
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    auto on_empty = [&](int r) {
        if (lane < H) da_dst[int64_t(r) * H + lane] = 0.f;
    };
    BwdChunk c0, c1;
    int k0 = 0, k1 = 0, la = 0, lb = 0, lo0 = 0, lo1 = 0;
    int sa0 = 0, sb0 = 0, sa1 = 0, sb1 = 0;
    int kind0 = cur.next_any(rowptr, lane, c0.row, c0.beg, c0.n, c0.first, c0.last, k0, la, lb, on_empty);
    if (!kind0) return;
    if (kind0 == 2) pack_lane_segment(c0.beg, k0, la, lb, lane, lo0, sa0, sb0);
    int b = 0;                   // stage of c0
    eg_fetch_async<H, DROPOUT>(stage[0], c0.beg + lane, lane < c0.n, perm, csr2csc, rec, lane);
    float trow[H];               // running t = sum alpha*d_alpha of the current (multi-chunk) row
    int row_beg = c0.beg;        // first edge of the current row
#pragma unroll
    for (int h = 0; h < H; ++h) trow[h] = 0.f;
    while (true) {
        const int kind1 = cur.next_any(rowptr, lane, c1.row, c1.beg, c1.n, c1.first, c1.last, k1, la, lb, on_empty);
        lo1 = 0;
        if (kind1 == 2) pack_lane_segment(c1.beg, k1, la, lb, lane, lo1, sa1, sb1);
        if (kind1) {
            if (lane < c1.n) eg_prefetch_row<H>(c1.row + lo1, a_dst, rowmax, rowsum);
            eg_fetch_async<H, DROPOUT>(stage[b ^ 1], c1.beg + lane, lane < c1.n, perm, csr2csc, rec, lane);
        } else {
            cp_async_commit();   // an empty group, so that c0's group is always the one before the newest
        }
        cp_async_wait_pending(1);
        EgEdge<H> x0;
        {
            EgRaw<H> r0;
            eg_take<H, DROPOUT>(r0, stage[b], lane < c0.n, lane);
            eg_finish<H, DROPOUT>(x0, r0, lane < c0.n, c0.row + lo0, a_dst, rowmax, rowsum, slope, keep);
        }
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
                eg_sweep2<H, DROPOUT>(c0.row, row_beg, c0.beg + c0.n, perm, csr2csc, a_dst, rowmax, rowsum, keep,
                                      keep_scale, slope, trow, rec, alpha_used, dz, eg_ld, dad, lane);
#pragma unroll
                for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
                if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
            }
        }
        if (!kind1) break;
        b ^= 1;
        c0 = c1;
        kind0 = kind1;
        k0 = k1;
        sa0 = sa1;
        sb0 = sb1;
        lo0 = lo1;
    }
}

// hub rows, step 1: one warp per chunk -- partial t of the chunk
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_dst_eg_hub1(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                    const int32_t* __restrict__ csr2csc, const float* __restrict__ a_dst,
                    const float* __restrict__ rowmax, const float* __restrict__ rowsum, const float* __restrict__ rec,
                    gnnfd_hub_plan_t plan, float slope, KeepMask keep, float keep_scale, float* __restrict__ part_t)
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
    EgRaw<H> r0, r1;
    eg_fetch<H, DROPOUT>(r0, beg + lane, beg + lane < end, perm, csr2csc, rec);
    for (int base = beg; base < end; base += 32) {
        const bool more = base + 32 < end;
        if (more) eg_fetch<H, DROPOUT>(r1, base + 32 + lane, base + 32 + lane < end, perm, csr2csc, rec);
        const bool live = base + lane < end;
        EgEdge<H> x;
        eg_finish<H, DROPOUT>(x, r0, live, i, a_dst, rowmax, rowsum, slope, keep);
#pragma unroll
        for (int h = 0; h < H; ++h) trow[h] += warp_sum(eg_head<H>(x, h, live, slope, keep_scale).u);
        if (more) r0 = r1;
    }
    if (lane == 0) store_vecH<H>(part_t + int64_t(c) * H, trow);
}

// hub rows, step 2: the row's total t (chunk order), second sweep, partial da_dst
template <int H, bool DROPOUT>
__global__ void __launch_bounds__(ROW_THREADS)
gat_bwd_dst_eg_hub2(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                    const int32_t* __restrict__ csr2csc, const float* __restrict__ a_dst,
                    const float* __restrict__ rowmax, const float* __restrict__ rowsum, const float* __restrict__ rec,
                    gnnfd_hub_plan_t plan, float slope, KeepMask keep, float keep_scale,
                    const float* __restrict__ t_total, float* alpha_used, float* dz, int64_t eg_ld,
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
    eg_sweep2<H, DROPOUT>(i, beg, end, perm, csr2csc, a_dst, rowmax, rowsum, keep, keep_scale, slope, t, rec,
                          alpha_used, dz, eg_ld, dad, lane);
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
    if (lane == 0) store_vecH<H>(part_dad + int64_t(c) * H, dad);
}

struct EgArgs {
    const float *a_dst, *rowmax, *rowsum, *rec;
};
template <class GE, bool DROPOUT>
static void launch_dst_eg(const gnnfd_graph_t* g, const EgArgs& in, float slope, KeepMask keep, float ks,
                          float* alpha_used, float* dz, int64_t eg_ld, float* da_dst, float* part_t, float* part_dad,
                          float* t_total, cudaStream_t st)
{
    constexpr int H = GE::H;
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + ROW_WARPS - 1) / ROW_WARPS);
    gat_bwd_dst_eg_items<H, DROPOUT><<<grid, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, in.a_dst, in.rowmax,
                                                                    in.rowsum, in.rec, g->items_dst, thr, slope, keep,
                                                                    ks, alpha_used, dz, eg_ld, da_dst);
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const unsigned gh = (unsigned)((pl.n_hub + ROW_WARPS - 1) / ROW_WARPS);
        const unsigned gc = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
        gat_bwd_dst_eg_hub1<H, DROPOUT><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, in.a_dst,
                                                                     in.rowmax, in.rowsum, in.rec, pl, slope, keep, ks,
                                                                     part_t);
        gat_hub_chunk_sum<H, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_t, t_total);
        gat_bwd_dst_eg_hub2<H, DROPOUT><<<gc, ROW_THREADS, 0, st>>>(g->rowptr, g->perm, g->csr2csc, in.a_dst,
                                                                     in.rowmax, in.rowsum, in.rec, pl, slope, keep, ks,
                                                                     t_total, alpha_used, dz, eg_ld, part_dad);
        gat_hub_chunk_sum<H, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_dad, da_dst);
        g_launches += 4;
    }
}

// workspace of the two-pass form: the records {d_alpha, a_src[j]} [E',2H] in CSR order, then the hub_dst partials
size_t gat_bwd_dst_srcmajor_ws_bytes(const gnnfd_graph_t* g, int H)
{
    size_t b = carve_bytes(size_t(g->n_edges) * 2 * H, 4);
    if (g->hub_dst.n_hub > 0)
        b += 2 * carve_bytes(size_t(g->hub_dst.n_chunk) * H, 4) + carve_bytes(size_t(g->hub_dst.n_hub) * H, 4);
    return b;
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
    const int64_t ld = (dz == alpha_used + H) ? 2 * H : H;
    // 32-byte-aligned slots take one 256-bit store per vector; eg_store reads that from the sign of eg_ld
    const bool wide = ((reinterpret_cast<uintptr_t>(alpha_used) | reinterpret_cast<uintptr_t>(dz)) & 31) == 0;
    const int64_t eg_ld = wide ? -ld : ld;
    const size_t need = gat_bwd_dst_srcmajor_ws_bytes(g, H);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gat_bwd_dst: workspace %zu < %zu", ws_bytes, need);
    char* p = reinterpret_cast<char*>(ws);
    float* rec = carve<float>(p, size_t(g->n_edges) * 2 * H);
    float *part_t = nullptr, *part_dad = nullptr, *t_total = nullptr;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        part_t = carve<float>(p, size_t(pl.n_chunk) * H);
        part_dad = carve<float>(p, size_t(pl.n_chunk) * H);
        t_total = carve<float>(p, size_t(pl.n_hub) * H);
    }
    if (g->n_edges > 0) {
        constexpr int SMEM = DaGeo<GE>::CTA_BYTES;
        GNNFD_CUDA(cudaFuncSetAttribute(gat_bwd_dalpha_src_stream<GE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        const int thr = g->hub_src.n_hub > 0 ? g->hub_src.threshold : INT_MAX;
        const unsigned grid = (unsigned)((g->items_src.n_items + DA_WARPS - 1) / DA_WARPS);
        gat_bwd_dalpha_src_stream<GE><<<grid, DA_THREADS, SMEM, st>>>(g->colptr, g->csc_row, g->csc_eid, xw, a_src,
                                                                      d_out, g->items_src, thr, rec);
        g_launches += 1;
        if (g->hub_src.n_hub > 0) {
            constexpr int HW = da_hub_warps<GE>();
            const unsigned gc = (unsigned)((g->hub_src.n_chunk + HW - 1) / HW);
            gat_bwd_dalpha_src_hub<GE><<<gc, 32 * HW, 0, st>>>(g->colptr, g->csc_row, g->csc_eid, xw, a_src, d_out,
                                                                   g->hub_src, rec);
            g_launches += 1;
        }
    }
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    const EgArgs in{a_dst, rowmax, rowsum, rec};
    if (p_drop > 0.f)
        launch_dst_eg<GE, true>(g, in, slope, keep, ks, alpha_used, dz, eg_ld, da_dst, part_t, part_dad, t_total, st);
    else
        launch_dst_eg<GE, false>(g, in, slope, keep, ks, alpha_used, dz, eg_ld, da_dst, part_t, part_dad, t_total, st);
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

// The source-major head-mean passes -- this two-pass backward and the three-pass forward (gat_fwd_msg.cu) -- apply to
// the head mean on a graph whose CSC positions are the edge-gradient slots (not the indirect multi-GPU receive layout),
// whose CSC twin is complete (csc_eid included) with a work-item plan over colptr, and whose sources and destinations
// are one node set.
bool gat_srcmajor_applies(const gnnfd_graph_t* g, int concat)
{
    return !concat && !g->edge_grads_indirect && g->n_src == g->n_dst && g->colptr && g->csc_row && g->csc_eid &&
           g->items_src.n_items > 0 && g->items_src.item_start;
}
bool gat_bwd_dst_srcmajor_applies(const gnnfd_graph_t* g, int concat) { return gat_srcmajor_applies(g, concat); }

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
    if (H == 8 && C == 32 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst_srcmajor<Geo<8, 32, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope,
                                                          keep_mask, p_drop, seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    if (H == 8 && C == 128 && xw_dtype == GNNFD_F32)
        return launch_bwd_dst_srcmajor<Geo<8, 128, float>>(g, xw, a_src, a_dst, rowmax, rowsum, d_out, negative_slope,
                                                           keep_mask, p_drop, seed, alpha_used, dz, da_dst, ws, ws_bytes, st);
    GNNFD_REQUIRE(false, GNNFD_ERR_UNSUPPORTED, "gat_bwd_dst: (heads=%d, out_channels=%d, dtype=%d) is not built; "
                  "available: (8,64,f32), (8,64,bf16), (8,32,f32), (8,128,f32), (4,32,f32)", H, C, xw_dtype);
    return GNNFD_ERR_UNSUPPORTED;
}

}  // namespace gnnfd
