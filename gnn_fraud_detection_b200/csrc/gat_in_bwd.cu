// Input-space backward of the GAT layer, edge pass (see in_common.cuh for the algebra): the autograd mirror of
// edge_update / softmax / aggregate (loss.backward() at src/train.py:142) without projected features:
//     d_alpha[e,h] = Gd[i,h,:] . x[j,:]          Gd = dO W_r^T / H from gnnfd_in_bwd_gd (one 4*F-byte row per destination)
//     u = alpha * d_alpha (dropout-scaled), t = sum_row u, dz = slope' * (u - alpha t), da_dst[i] = sum_row dz
// dz is written in SOURCE-MAJOR order (slot csr2csc[e]) so that da_src = per-source sums (gnnfd_in_bwd_dasrc) reads it
// contiguously.  The weight gradient comes from the saved Z image (in_gemm.cu), so a first layer needs no alpha_used.
// A hidden layer needs dx = dxw W, and dxw is what gnnfd_gat_bwd_src computes from (alpha_used, dz) slot records: the REC
// variant (KP = 64) stores alpha_used = alpha * keep / (1-p) beside dz, as the 64-byte record [alpha_used | dz] at slot
// csr2csc[e] that gnnfd_gat_bwd_dst writes (two 256-bit stores), and nothing else changes.
// alpha (with the LeakyReLU region in its sign bit) and the row-end flags are what the forward's attention pass saved: the
// staging of a chunk (lane = edge) is two coalesced loads, no logit gathers, no exp, no row statistics.
// Same warp-stream structure as gat_bwd_dst.cu (work items, staging one chunk ahead, packs of short rows, hub rows in
// chunks with a deterministic merge); x rows arrive through the per-warp bulk-copy ring, and the destination's Gd row
// is prefetched by the copy engine into a per-warp shared-memory buffer while the previous row is processed.
#include "in_common.cuh"
#include "gat_phase_bwd.cuh"


#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;
int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who);

namespace in {
constexpr int IN_UNROLL_BWD = 4;
bool in_x_ok(const float* x, int64_t ldx, int KP);   // gat_in_fwd.cu


constexpr int BWD_SLOTS = 6;      // 6 row slots: with the Gd buffer that still fits 4 CTAs (16 warps) per SM in shared memory
using BwdRing = InRingT<BWD_SLOTS>;

// Staging of one chunk (lane = edge) from what the forward's attention pass saved: alpha (sign bit = LeakyReLU negative
// region) and jflag (source id | row end).  No logit gathers, no exp, no row statistics.
// bits layout per staged edge: [0,8) LeakyReLU-positive, [8,16) dropout keep, [16,21) first lane of the row, [21,26) last lane
// of the row (packs only), bit 26 = this edge is the last of its row.
template <bool DROPOUT>
__device__ __forceinline__ void stage_bwd_chunk(const BwdChunk& c, bool pack, const float* __restrict__ alpha,
                                                const int32_t* __restrict__ jflag, const int32_t* __restrict__ perm, KeepMask keep,
                                                float* p_s, int* j_s, int* bits_s, int lane)
{
    int jf = 0, bits = 0;
    float w[H];
    if (lane < c.n) {
        const int e = c.beg + lane;
        jf = jflag[e];
        load_vecH<H>(alpha + int64_t(e) * H, w);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            bits |= int((__float_as_uint(w[h]) >> 31) ^ 1u) << h;
            w[h] = fabsf(w[h]);
        }
        if (DROPOUT) bits |= int(keep.bits(perm[e], H)) << 8;
        else bits |= 0xff00;
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) w[h] = 0.f;
    }
    const unsigned lastmask = __ballot_sync(FULL, jf < 0);
    if (lane < c.n) {
        bits |= int(jf < 0) << 26;
        if (pack) {
            const unsigned below = lastmask & ((1u << lane) - 1u);
            const int sa = below ? 32 - __clz(below) : 0;
            const int sb = __ffs(lastmask >> lane) - 1 + lane;
            bits |= (sa << 16) | (sb << 21);
        }
    }
    store_vecH<H>(p_s + lane * H, w);
    j_s[lane] = jf & 0x7fffffff;
    bits_s[lane] = bits;
    __syncwarp();
}

// second sweep of a long row: dz = slope' * (u - alpha * t); lane-local partial of da_dst.  LD: floats per dz slot (H, or 2H
// for records, whose alpha_used half phase C has already written)
template <int LD>
__device__ __forceinline__ void in_sweep2(int beg, int end, const int32_t* __restrict__ csr2csc, const float* __restrict__ alpha,
                                          float slope, const float (&t)[H], int lane, float* __restrict__ dz, float (&dad)[H])
{
    for (int e = beg + lane; e < end; e += 32) {
        float a[H], u[H], o[H];
        const int64_t pos = csr2csc[e];          // edge gradients live in source-major order
        load_vecH<H>(alpha + int64_t(e) * H, a);
        load_vecH<H>(dz + pos * LD, u);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float sl = (__float_as_uint(a[h]) >> 31) ? slope : 1.f;
            o[h] = sl * (u[h] - fabsf(a[h]) * t[h]);
            dad[h] += o[h];
        }
        store_vecH<H>(dz + pos * LD, o);
    }
}

// phase C's store of one edge in record mode: the record [alpha_used | dz] at source-major slot pos, dz == record + H
__device__ __forceinline__ void store_record(float* __restrict__ dz, int64_t pos, const float (&alpha)[H], int bits,
                                             float keep_scale, const float (&o)[H])
{
    float au[H];
#pragma unroll
    for (int hh = 0; hh < H; ++hh) au[hh] = (bits >> (8 + hh)) & 1 ? alpha[hh] * keep_scale : 0.f;
    store_vecH_wide<H>(dz + pos * 2 * H - H, au);
    store_vecH_wide<H>(dz + pos * 2 * H, o);
}

// per-warp scratch beyond the ring: dal_s [32][H] floats, bits_s [2][32] ints, the Gd row buffer [F] floats
__host__ __device__ inline int bwd_extra_bytes(int F) { return 32 * H * 4 + 2 * 32 * 4 + F * 4; }

// Gd row of the destination being processed: fetched with one bulk copy into shared memory (no registers in flight);
// lane (h, q) then keeps the float4s 4*i + q of head h in registers
template <int N4>
struct GdBuf {
    using RG = RowGeo<N4>;
    uint32_t buf_u32, bar;
    const float* gd;
    int F, KP;
    int pending = -1, loads = 0, deferred = -1;
    // WAR hazard: the copy engine (async proxy) may overwrite the buffer while the ld.shared of take() are still in
    // flight -- __syncwarp orders instruction issue, not load completion, and an L2-resident Gd row arrives within a few
    // hundred cycles.  A prefetch that follows a take() is therefore only REQUESTED (want_later) and issued by
    // flush() after the next edge has been processed: its FMAs consume every loaded register, so the loads have landed.
    __device__ __forceinline__ void want_later(int row) { deferred = row; }
    __device__ __forceinline__ void flush(int lane)
    {
        if (deferred >= 0) {
            want(deferred, lane);
            deferred = -1;
        }
    }
    __device__ __forceinline__ void want(int row, int lane)
    {
        if (pending == row) return;
        if (lane == 0) {
            mbar_expect_tx_u32(bar, uint32_t(F) * 4u);
            bulk_g2s_u32(buf_u32, gd + int64_t(row) * F, uint32_t(F) * 4u, bar);
        }
        pending = row;
    }
    __device__ __forceinline__ void take(int row, int lane, float4 (&g)[RG::NI])
    {
        deferred = -1;
        if (pending != row) {
            if (pending >= 0) {                 // a wrong guess is in flight: let it land before the buffer is reused
                mbar_wait_u32(bar, uint32_t(loads & 1));
                ++loads;
                __syncwarp();
                pending = -1;
            }
            want(row, lane);
        }
        mbar_wait_u32(bar, uint32_t(loads & 1));
        ++loads;
        const int h = lane >> 2, q = lane & 3, n4 = KP >> 2;
#pragma unroll
        for (int i = 0; i < RG::NI; ++i)
            g[i] = RG::valid(i, q, n4) ? lds128(buf_u32 + uint32_t(h * KP + 16 * i + 4 * q) * 4u) : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();                           // every lane has read the buffer before the next copy is issued
        pending = -1;
    }
};

// HUB = false: whole rows and packs of short rows, results go to da_dst.  HUB = true: one (row, range) segment, the
// partial t of the segment goes to part_t[chunk_id]; the second sweep is a separate kernel.  REC: dz slots are records.
template <int N4, bool DROPOUT, bool HUB, bool REC>
__device__ __forceinline__ void in_bwd_stream(ChunkCursor& cur, BwdRing& ring, GdBuf<N4>& gdb, const int32_t* __restrict__ rowptr,
                                              const int32_t* __restrict__ perm, const int32_t* __restrict__ csr2csc,
                                              const float* __restrict__ alpha_g, const int32_t* __restrict__ jflag, float slope,
                                              KeepMask keep, float keep_scale, float* __restrict__ dz, float* __restrict__ da_dst,
                                              float* __restrict__ part_t, int chunk_id, int lane)
{
    using RG = RowGeo<N4>;
    constexpr bool PACK = !HUB;     // the row stream also hands out packs of short rows; a hub segment is part of one row
    const int h = lane >> 2, q = lane & 3, n4 = gdb.KP >> 2;
    float* dal_s = reinterpret_cast<float*>(ring.extra);
    int* bits_s = reinterpret_cast<int*>(ring.extra + 32 * H * 4);
    auto on_empty = [&](int r) {
        if (!HUB && lane < H) da_dst[int64_t(r) * H + lane] = 0.f;
    };
    BwdChunk c0, c1;
    int kind0 = 0, kind1 = 0, k0 = 0, k1 = 0, la = 0, lb = 0;
    int b0 = 0;
    auto next = [&](BwdChunk& c, int& kk) -> int {
        if (PACK) return cur.next_any(rowptr, lane, c.row, c.beg, c.n, c.first, c.last, kk, la, lb, on_empty);
        return cur.next(rowptr, c.row, c.beg, c.n, c.first, c.last, on_empty) ? 1 : 0;
    };
    auto phase_a = [&](const BwdChunk& c, int kind, int kk, int buf) {
        (void)kk;
        stage_bwd_chunk<DROPOUT>(c, PACK && kind == 2, alpha_g, jflag, perm, keep, ring.p_s + buf * 32 * H, ring.j_s + buf * 32,
                                 bits_s + buf * 32, lane);
    };
    kind0 = next(c0, k0);
    if (!kind0) return;
    gdb.want(c0.row, lane);
    phase_a(c0, kind0, k0, b0);
    float4 g[RG::NI];
    gdb.take(c0.row, lane, g);
    if (PACK && kind0 == 2 && k0 > 1) gdb.want_later(c0.row + 1);
    int issued0 = 0, issued1 = 0;
    float trow[H];
    int row_beg = c0.beg;
#pragma unroll
    for (int hh = 0; hh < H; ++hh) trow[hh] = 0.f;
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        {
            const int kk = min(ring.room(), c0.n - issued0);
            if (kk > 0) { ring.issue_many(j0 + issued0, kk, lane); issued0 += kk; }
        }
        kind1 = next(c1, k1);
        issued1 = 0;
        if (kind1) {
            phase_a(c1, kind1, k1, b0 ^ 1);
            // the next destination row in stream order, unless a row of the current pack is still to come
            if (c1.first && gdb.pending < 0 && gdb.deferred < 0 && !(PACK && kind0 == 2 && k0 > 1)) gdb.want_later(c1.row);
        }
        if (c0.first) {
            row_beg = c0.beg;
#pragma unroll
            for (int hh = 0; hh < H; ++hh) trow[hh] = 0.f;
        }
        int rows_done = 0;
        const int* bits0 = bits_s + b0 * 32;
        // packs: lanes (= staged edges) that end a row
        const unsigned lastmask = (PACK && kind0 == 2) ? __ballot_sync(FULL, (bits0[lane] >> 26) & 1) : 0u;
        // phase B: dot products of the staged x rows with this row's Gd (lane = head, quarter); edges in groups of four:
        // one warp barrier and one (multi-lane) refill per group
        for (int t0 = 0; t0 < c0.n; t0 += 4) {
            const int cnt = min(4, c0.n - t0);
#pragma unroll IN_UNROLL_BWD
            for (int r = 0; r < 4; ++r) {
                if (r < cnt) {
                    const int t = t0 + r;
                    const uint32_t a = ring.front_at(r) + uint32_t(q) * 16u;
                    float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;     // four independent FMA chains
#pragma unroll
                    for (int i = 0; i < RG::NI; ++i)
                        if (RG::valid(i, q, n4)) {
                            const float4 v = lds128(a + uint32_t(i) * 64u);
                            ffma2_vec(d0, d1, g[i].x, g[i].y, v.x, v.y);
                            ffma2_vec(d2, d3, g[i].z, g[i].w, v.z, v.w);
                        }
                    float d = (d0 + d1) + (d2 + d3);
                    d += __shfl_xor_sync(FULL, d, 1);
                    d += __shfl_xor_sync(FULL, d, 2);
                    if (q == 0) dal_s[t * H + h] = d;
                    gdb.flush(lane);             // every lane has consumed g in the FMAs above (the shuffles are the meeting point)
                    if (PACK && t + 1 < c0.n && ((lastmask >> t) & 1u)) {
                        // row boundary inside the pack: switch to the next row's Gd, prefetch the one after it
                        ++rows_done;
                        gdb.take(c0.row + rows_done, lane, g);
                        if (rows_done + 1 < k0) gdb.want_later(c0.row + rows_done + 1);
                        else if (kind1 && c1.first) gdb.want_later(c1.row);
                    }
                }
            }
            ring.pop_many(cnt);
            int free_slots = cnt;
            const int kk = min(free_slots, c0.n - issued0);
            if (kk > 0) { ring.issue_many(j0 + issued0, kk, lane); issued0 += kk; free_slots -= kk; }
            if (kind1 && free_slots > 0) {
                const int kn = min(free_slots, c1.n - issued1);
                if (kn > 0) { ring.issue_many(j1 + issued1, kn, lane); issued1 += kn; }
            }
        }
        __syncwarp();
        // phase C: lane = edge
        {
            float alpha[H], dal[H], u[H];
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
            const int64_t pos = live ? csr2csc[c0.beg + lane] : 0;    // source-major slot of this edge
#pragma unroll
            for (int hh = 0; hh < H; ++hh) {
                const float ks = (bits >> (8 + hh)) & 1 ? keep_scale : 0.f;
                u[hh] = live ? alpha[hh] * dal[hh] * ks : 0.f;
            }
            if (PACK && kind0 == 2) {
                const int sa = (bits >> 16) & 31, sb = live ? (bits >> 21) & 31 : lane;
                const bool lastf = live && ((bits >> 26) & 1);
                float o[H], dad[H];
#pragma unroll
                for (int hh = 0; hh < H; ++hh) {
                    const float tt = seg_total(u[hh], sa, sb, lane);
                    const float sl = (bits >> hh) & 1 ? 1.f : slope;
                    o[hh] = live ? sl * (u[hh] - alpha[hh] * tt) : 0.f;
                    dad[hh] = seg_total(o[hh], sa, sb, lane);
                }
                if (live) {
                    if constexpr (REC) store_record(dz, pos, alpha, bits, keep_scale, o);
                    else store_vecH<H>(dz + pos * H, o);
                }
                const unsigned lastm = __ballot_sync(FULL, lastf);
                if (lastf) {
                    const int64_t r = c0.row + __popc(lastm & ((1u << lane) - 1u));
                    store_vecH<H>(da_dst + r * H, dad);
                }
            } else if (!HUB && c0.first && c0.last) {
                float o[H], dad[H];
#pragma unroll
                for (int hh = 0; hh < H; ++hh) {
                    const float tt = warp_sum(u[hh]);
                    const float sl = (bits >> hh) & 1 ? 1.f : slope;
                    o[hh] = live ? sl * (u[hh] - alpha[hh] * tt) : 0.f;
                    dad[hh] = warp_sum(o[hh]);
                }
                if (live) {
                    if constexpr (REC) store_record(dz, pos, alpha, bits, keep_scale, o);
                    else store_vecH<H>(dz + pos * H, o);
                }
                if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
            } else {
                if (live) {                                     // parked until t is known
                    if constexpr (REC) store_record(dz, pos, alpha, bits, keep_scale, u);
                    else store_vecH<H>(dz + pos * H, u);
                }
#pragma unroll
                for (int hh = 0; hh < H; ++hh) trow[hh] += warp_sum(u[hh]);
                if (c0.last) {
                    if (HUB) {
                        if (lane == 0) store_vecH<H>(part_t + int64_t(chunk_id) * H, trow);
                    } else {
                        __syncwarp();
                        float dad[H];
#pragma unroll
                        for (int hh = 0; hh < H; ++hh) dad[hh] = 0.f;
                        in_sweep2<REC ? 2 * H : H>(row_beg, c0.beg + c0.n, csr2csc, alpha_g, slope, trow, lane, dz, dad);
#pragma unroll
                        for (int hh = 0; hh < H; ++hh) dad[hh] = warp_sum(dad[hh]);
                        if (lane == 0) store_vecH<H>(da_dst + int64_t(c0.row) * H, dad);
                    }
                }
            }
        }
        __syncwarp();
        if (!kind1) break;
        if (c1.first) {
            gdb.take(c1.row, lane, g);
            if (PACK && kind1 == 2 && k1 > 1) gdb.want_later(c1.row + 1);
        }
        c0 = c1;
        kind0 = kind1;
        k0 = k1;
        issued0 = issued1;
        b0 ^= 1;
    }
}

template <int N4>
__device__ __forceinline__ void gdbuf_init(GdBuf<N4>& gdb, BwdRing& ring, const float* gd, int F, int KP)
{
    gdb.buf_u32 = st_smem_u32(ring.extra + 32 * H * 4 + 2 * 32 * 4);
    gdb.bar = ring.spare_bar();
    gdb.gd = gd;
    gdb.F = F;
    gdb.KP = KP;
}

constexpr int IN_BWD_CTAS = 4;

template <int N4, bool DROPOUT, bool REC>
__global__ void __launch_bounds__(IN_THREADS, IN_BWD_CTAS)
gat_in_bwd_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, const int32_t* __restrict__ csr2csc,
                 const float* __restrict__ x, int64_t ldx, int KP, const float* __restrict__ alpha,
                 const int32_t* __restrict__ jflag, const float* __restrict__ gd, gnnfd_item_plan_t items, int item_lo,
                 int item_hi, int hub_threshold, float slope, KeepMask keep, float keep_scale,
                 float* __restrict__ dz, float* __restrict__ da_dst)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = item_lo + blockIdx.x * IN_WARPS + warp;
    if (item >= item_hi) return;
    const int F = H * KP;
    BwdRing ring;
    ring.init(smem + warp * in_warp_bytes(KP, bwd_extra_bytes(F), BWD_SLOTS), x, ldx, KP, lane);
    GdBuf<N4> gdb;
    gdbuf_init(gdb, ring, gd, F, KP);
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    in_bwd_stream<N4, DROPOUT, false, REC>(cur, ring, gdb, rowptr, perm, csr2csc, alpha, jflag, slope, keep, keep_scale, dz,
                                           da_dst, nullptr, 0, lane);
}

// hub rows, step 1: one warp per chunk -- first sweep, partial t (rows outside [row_lo, row_hi) belong to another block)
template <int N4, bool DROPOUT, bool REC>
__global__ void __launch_bounds__(IN_THREADS, IN_BWD_CTAS)
gat_in_bwd_hub1(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, const int32_t* __restrict__ csr2csc,
                const float* __restrict__ x, int64_t ldx, int KP, const float* __restrict__ alpha,
                const int32_t* __restrict__ jflag, const float* __restrict__ gd, gnnfd_hub_plan_t plan, int row_lo, int row_hi,
                float slope, KeepMask keep, float keep_scale, float* __restrict__ dz, float* __restrict__ part_t)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * IN_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int i = plan.hub_row[slot];
    if (i < row_lo || i >= row_hi) return;
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    const int F = H * KP;
    BwdRing ring;
    ring.init(smem + warp * in_warp_bytes(KP, bwd_extra_bytes(F), BWD_SLOTS), x, ldx, KP, lane);
    GdBuf<N4> gdb;
    gdbuf_init(gdb, ring, gd, F, KP);
    ChunkCursor cur;
    cur.start_segment(i, beg, end);
    in_bwd_stream<N4, DROPOUT, true, REC>(cur, ring, gdb, rowptr, perm, csr2csc, alpha, jflag, slope, keep, keep_scale, dz,
                                          nullptr, part_t, c, lane);
}

// hub rows, step 2: second sweep of every chunk with the row's total t, partial da_dst
template <int LD>
__global__ void __launch_bounds__(ROW_THREADS)
gat_in_bwd_hub2(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ csr2csc, const float* __restrict__ alpha,
                gnnfd_hub_plan_t plan, float slope, const float* __restrict__ t_total, float* __restrict__ dz,
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
    load_vecH<H>(t_total + int64_t(slot) * H, t);      // the same total in every chunk of the row
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = 0.f;
    in_sweep2<LD>(beg, end, csr2csc, alpha, slope, t, lane, dz, dad);
#pragma unroll
    for (int h = 0; h < H; ++h) dad[h] = warp_sum(dad[h]);
    if (lane == 0) store_vecH<H>(part_dad + int64_t(c) * H, dad);
}

template <class Kn>
static int in_set_smem_bwd(Kn kernel, int bytes)
{
    GNNFD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return GNNFD_OK;
}

}  // namespace in
}  // namespace gnnfd

using namespace gnnfd;
using namespace gnnfd::in;

extern "C" {

int gnnfd_in_bwd_edges_workspace_bytes(const gnnfd_graph_t* g, size_t* bytes)
{
    GNNFD_REQUIRE(g && bytes, GNNFD_ERR_ARG, "in_bwd_edges_workspace_bytes: NULL argument");
    *bytes = 2 * carve_bytes(size_t(g->hub_dst.n_chunk) * H, 4) + carve_bytes(size_t(g->hub_dst.n_hub) * H, 4) + 256;
    return GNNFD_OK;
}

/* dz [E',H] (source-major order) and da_dst [n_dst,H] for the destination rows of the work items [item_lo, item_hi)
 * (= rows [row_lo, row_hi), which must be the rows those items cover; pass 0, n_items, 0, n_dst for everything).
 * gd holds the Gd rows of [gd_row0, ...) with leading dimension F.  phase bit 0: process the row block (items + first
 * hub sweep); bit 1: finish the hub rows (second sweep; after the LAST block, with the same ws).
 * alpha_used != NULL (padded K = 64 only): also alpha_used, as the interleaved [E',2H] records of gnnfd_gat_bwd_dst
 * (dz == alpha_used + H, 32-byte aligned). */
int gnnfd_in_bwd_edges(const gnnfd_graph_t* g, const float* x, int64_t ldx, int64_t K, const float* alpha,
                       const int32_t* jflag, const float* gd, int64_t gd_row0,
                       int64_t item_lo, int64_t item_hi, int64_t row_lo, int64_t row_hi, float negative_slope,
                       const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, float* alpha_used, float* dz, float* da_dst,
                       void* ws, size_t ws_bytes, int phase, gnnfd_stream_t stream)
{
    int rc = check_graph(g, true, "in_bwd_edges");
    if (rc) return rc;
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K, GNNFD_ERR_ARG, "in_bwd_edges: bad shape (K <= %d)", MAX_K);
    if (g->n_dst == 0) return GNNFD_OK;
    GNNFD_REQUIRE(x && gd && da_dst, GNNFD_ERR_ARG, "in_bwd_edges: NULL tensor");
    GNNFD_REQUIRE(g->n_edges == 0 || (alpha && jflag), GNNFD_ERR_ARG, "in_bwd_edges: NULL alpha / jflag (outputs of gnnfd_in_fwd)");
    GNNFD_REQUIRE(g->n_edges == 0 || (dz && g->csr2csc), GNNFD_ERR_ARG, "in_bwd_edges: dz / csr2csc is NULL");
    GNNFD_REQUIRE(p_drop >= 0.f && p_drop <= 0.9f, GNNFD_ERR_ARG, "in_bwd_edges: dropout p must be in [0,0.9]");
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG, "in_bwd_edges: no work-item plan over rowptr");
    GNNFD_REQUIRE(item_lo >= 0 && item_lo <= item_hi && item_hi <= g->items_dst.n_items && row_lo >= 0 && row_lo <= row_hi &&
                      row_hi <= g->n_dst && gd_row0 >= 0 && gd_row0 <= row_lo,
                  GNNFD_ERR_ARG, "in_bwd_edges: bad item / row range");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(gd) & 15) == 0, GNNFD_ERR_ARG, "in_bwd_edges: gd must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const Dims d((int)K);
    const bool rec = alpha_used != nullptr;
    GNNFD_REQUIRE(!rec || d.KP == 64, GNNFD_ERR_UNSUPPORTED,
                  "in_bwd_edges: alpha_used records are built for K <= 64 padded to 64 only (K = %lld)", (long long)K);
    GNNFD_REQUIRE(!rec || g->n_edges == 0 || (dz == alpha_used + H && (reinterpret_cast<uintptr_t>(alpha_used) & 31) == 0),
                  GNNFD_ERR_ARG, "in_bwd_edges: alpha_used / dz must be the halves of one 32-byte aligned [E',2H] buffer");
    const bool drop = p_drop > 0.f;              // explicit mask, or (mask == NULL) the counter-based RNG keyed on seed
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, dropout_seed, &ks);
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    GNNFD_REQUIRE(in_x_ok(x, ldx, d.KP), GNNFD_ERR_ARG,
                  "in_bwd_edges: x rows must be 16-byte aligned and zero-padded to %d floats (gnnfd_in_pad_x)", d.KP);
    const int smem = IN_WARPS * in_warp_bytes(d.KP, bwd_extra_bytes(d.F), BWD_SLOTS);
    const float* gd0 = gd - gd_row0 * d.F;          // indexed by global destination row
    const gnnfd_hub_plan_t& pl = g->hub_dst;
    float *part_t = nullptr, *part_dad = nullptr, *t_total = nullptr;
    if (pl.n_hub > 0) {
        size_t need = 0;
        gnnfd_in_bwd_edges_workspace_bytes(g, &need);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "in_bwd_edges: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        part_t = carve<float>(p, size_t(pl.n_chunk) * H);
        part_dad = carve<float>(p, size_t(pl.n_chunk) * H);
        t_total = carve<float>(p, size_t(pl.n_hub) * H);
    }
    if ((phase & 1) && item_hi > item_lo) {
        const unsigned grid = (unsigned)((item_hi - item_lo + IN_WARPS - 1) / IN_WARPS);
        const unsigned gc = (unsigned)((pl.n_chunk + IN_WARPS - 1) / IN_WARPS);
#define GNNFD_IN_BWD(NN, DD, RR)                                                                                       \
    rc = in_set_smem_bwd(gat_in_bwd_items<NN, DD, RR>, smem);                                                          \
    if (rc) return rc;                                                                                                 \
    gat_in_bwd_items<NN, DD, RR><<<grid, IN_THREADS, smem, st>>>(g->rowptr, g->perm, g->csr2csc, x, ldx, d.KP, alpha, jflag, gd0, \
                                                                 g->items_dst, (int)item_lo, (int)item_hi, thr, negative_slope,  \
                                                                 keep, ks, dz, da_dst)
#define GNNFD_IN_HUB1(NN, DD, RR)                                                                                      \
    rc = in_set_smem_bwd(gat_in_bwd_hub1<NN, DD, RR>, smem);                                                           \
    if (rc) return rc;                                                                                                 \
    gat_in_bwd_hub1<NN, DD, RR><<<gc, IN_THREADS, smem, st>>>(g->rowptr, g->perm, g->csr2csc, x, ldx, d.KP, alpha, jflag, gd0, pl, \
                                                              (int)row_lo, (int)row_hi, negative_slope, keep, ks, dz, part_t)
#define GNNFD_IN_BWD_ALL(NN, RR)                                                                                       \
    if (drop) { GNNFD_IN_BWD(NN, true, RR); } else { GNNFD_IN_BWD(NN, false, RR); }                                    \
    g_launches += 1;                                                                                                   \
    if (pl.n_hub > 0) {                                                                                                \
        if (drop) { GNNFD_IN_HUB1(NN, true, RR); } else { GNNFD_IN_HUB1(NN, false, RR); }                              \
        g_launches += 1;                                                                                               \
    }
        if (d.KP == 168) { GNNFD_IN_BWD_ALL(42, false) }
        else if (d.KP == 64 && rec) { GNNFD_IN_BWD_ALL(16, true) }
        else if (d.KP == 64) { GNNFD_IN_BWD_ALL(16, false) }
        else { GNNFD_IN_BWD_ALL(0, false) }
#undef GNNFD_IN_BWD_ALL
#undef GNNFD_IN_HUB1
#undef GNNFD_IN_BWD
    }
    if ((phase & 2) && pl.n_hub > 0) {
        const unsigned gh = (unsigned)((pl.n_hub + ROW_WARPS - 1) / ROW_WARPS);
        const unsigned gc2 = (unsigned)((pl.n_chunk + ROW_WARPS - 1) / ROW_WARPS);
        gat_hub_chunk_sum<H, false><<<gh, ROW_THREADS, 0, st>>>(pl, part_t, t_total);
        if (rec)
            gat_in_bwd_hub2<2 * H><<<gc2, ROW_THREADS, 0, st>>>(g->rowptr, g->csr2csc, alpha, pl, negative_slope, t_total, dz,
                                                                part_dad);
        else
            gat_in_bwd_hub2<H><<<gc2, ROW_THREADS, 0, st>>>(g->rowptr, g->csr2csc, alpha, pl, negative_slope, t_total, dz, part_dad);
        gat_hub_chunk_sum<H, true><<<gh, ROW_THREADS, 0, st>>>(pl, part_dad, da_dst);
        g_launches += 3;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // extern "C"
