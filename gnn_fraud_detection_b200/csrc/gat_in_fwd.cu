// Input-space forward of the first GAT layer (see in_common.cuh for the algebra):
//   gnnfd_in_logits   a_src / a_dst straight from x (u = W_h^T att precomputed), + max |x| for the fp16-pair scale
//   gnnfd_in_prepare  per-call constants: scales, the W images of the two dense stages
//   gnnfd_in_fwd      two passes.  ATTENTION pass (lane = edge): LeakyReLU + segment softmax -> normalised alpha [E',H] with
//                     the LeakyReLU region in its sign bit, jflag [E'] = source id | row-end flag, rowmax / rowsum; kept
//                     for the backward.  FEATURE pass: alpha-weighted gather-sum of INPUT rows x[j] (K*4 bytes per edge
//                     instead of the 2 KB projected row), lane = feature group with the accumulators of all heads, written
//                     as the fp16-pair tensor-core image Z that gnnfd_in_out (in_gemm.cu) multiplies with W.
// Replaces, for the reference's first layer (src/models/gat.py:39,80; tgn.py:43,94), the same PyG stages as
// gnnfd_project_fwd + gnnfd_gat_fwd: lin_src / (x*att).sum(-1) / edge_update / message / aggregate.
// Same warp-stream structure as gat_fwd.cu: one warp per edge-balanced work item, the staging of a chunk (lane = edge) one
// chunk ahead, rows delivered by the bulk-copy engine into a per-warp ring; packs of short rows; hub rows split into
// chunks whose partial sums are added in chunk order (deterministic).
#include "in_common.cuh"
#include "gat_stream.cuh"
#include "gat_alpha.cuh"

#include <atomic>
#include <climits>

namespace gnnfd {
extern std::atomic<long long> g_launches;
int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who);
int in_build_gd_image(const float* W, int K, void* prep, cudaStream_t st);   // in_gemm.cu

namespace in {
constexpr int IN_UNROLL_FWD = 1;     // the row epilogue (image write) sits inside the edge loop: unrolling it 4x thrashes the i-cache

// ---- u = W_h^T att  ([2H][KP]) --------------------------------------------------------------------------------------
__global__ void in_u_kernel(const float* __restrict__ W, const float* __restrict__ att_src, const float* __restrict__ att_dst,
                            int K, int KP, float* __restrict__ u)
{
    const int o = blockIdx.x;                 // 0..2H-1
    const int h = o % H;
    const float* att = (o < H ? att_src : att_dst) + h * C;
    for (int k = threadIdx.x; k < KP; k += blockDim.x) {
        float s = 0.f;
        if (k < K)
            for (int c = 0; c < C; ++c) s = fmaf(W[int64_t(h * C + c) * K + k], att[c], s);
        u[o * KP + k] = s;
    }
}

// a_src[n,h] = x[n,:] . u[h,:], a_dst[n,h] = x[n,:] . u[H+h,:].  The CTA streams tiles of 64 consecutive rows through
// shared memory (ONE bulk copy per tile, double-buffered); lane = (head h, quarter q) as in the edge kernels: 44 + 44
// u values in registers, per row 11 shared loads, 88 FMAs and two 2-step quad reductions.  Also max |x|.
constexpr int LG_ROWS = 64, LG_WARPS = 8;
// the a_src rows go to a_src (peers.mode 0) or into the same rows of a buffer on every rank (PeerRows, in_common.cuh)
template <int N4>
__global__ void __launch_bounds__(LG_WARPS * 32, 2)
in_logits_kernel(const float* __restrict__ x, int64_t ldx, int64_t N, int KP, const float* __restrict__ u,
                 float* __restrict__ a_src, float* __restrict__ a_dst, unsigned* __restrict__ xmax_bits, PeerRows peers)
{
    using RG = RowGeo<N4>;
    extern __shared__ __align__(128) uint8_t lsm[];
    __shared__ uint64_t full[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int h = lane >> 2, q = lane & 3;
    const int n4 = KP >> 2;
    const uint32_t rowb = uint32_t(KP) * 4u;
    const bool dense = (ldx == KP);                    // a tile is one contiguous block
    float4 us[RG::NI], ud[RG::NI];
#pragma unroll
    for (int i = 0; i < RG::NI; ++i) {
        us[i] = ud[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RG::valid(i, q, n4)) {
            us[i] = *reinterpret_cast<const float4*>(u + h * KP + 16 * i + 4 * q);
            ud[i] = *reinterpret_cast<const float4*>(u + (H + h) * KP + 16 * i + 4 * q);
        }
    }
    if (tid == 0) {
        st_mbar_init(&full[0], 1);
        st_mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t n_tiles = (N + LG_ROWS - 1) / LG_ROWS;
    const uint32_t buf_bytes = LG_ROWS * rowb;
    auto load_tile = [&](int64_t t, int b) {           // thread 0
        const int64_t r0 = t * LG_ROWS;
        const int rows = int(N - r0 < LG_ROWS ? N - r0 : LG_ROWS);
        const uint32_t bar = st_smem_u32(&full[b]);
        mbar_expect_tx_u32(bar, uint32_t(rows) * rowb);
        if (dense) bulk_g2s_u32(st_smem_u32(lsm) + b * buf_bytes, x + r0 * ldx, uint32_t(rows) * rowb, bar);
        else
            for (int r = 0; r < rows; ++r) bulk_g2s_u32(st_smem_u32(lsm) + b * buf_bytes + r * rowb, x + (r0 + r) * ldx, rowb, bar);
    };
    float mx = 0.f;
    int64_t it = 0;
    if (tid == 0 && blockIdx.x < n_tiles) load_tile(blockIdx.x, 0);
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
        const int b = int(it & 1);
        if (tid == 0 && t + gridDim.x < n_tiles) load_tile(t + gridDim.x, b ^ 1);   // buffer b^1 was released by the barrier below
        mbar_wait_u32(st_smem_u32(&full[b]), uint32_t((it >> 1) & 1));
        const int64_t r0 = t * LG_ROWS;
        const int rows = int(N - r0 < LG_ROWS ? N - r0 : LG_ROWS);
        for (int r = warp; r < rows; r += LG_WARPS) {
            const uint32_t a = st_smem_u32(lsm) + b * buf_bytes + r * rowb;
            float ds = 0.f, dd = 0.f;
#pragma unroll
            for (int i = 0; i < RG::NI; ++i)
                if (RG::valid(i, q, n4)) {
                    const float4 v = lds128(a + uint32_t(4 * i + q) * 16u);
                    ds = fmaf(us[i].x, v.x, fmaf(us[i].y, v.y, fmaf(us[i].z, v.z, fmaf(us[i].w, v.w, ds))));
                    dd = fmaf(ud[i].x, v.x, fmaf(ud[i].y, v.y, fmaf(ud[i].z, v.z, fmaf(ud[i].w, v.w, dd))));
                    mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
                }
            ds += __shfl_xor_sync(FULL, ds, 1); dd += __shfl_xor_sync(FULL, dd, 1);
            ds += __shfl_xor_sync(FULL, ds, 2); dd += __shfl_xor_sync(FULL, dd, 2);
            if (q == 0) a_dst[(r0 + r) * H + h] = dd;
            if (peers.mode == 0) {
                if (q == 0) a_src[(r0 + r) * H + h] = ds;
            } else {
                // lanes 0 and 16 collect heads 0-3 / 4-7 (every lane of a quad holds its head's sum) and store 16 bytes
                const int b = lane & 16;
                float4 v;
                v.x = __shfl_sync(FULL, ds, b);
                v.y = __shfl_sync(FULL, ds, b + 4);
                v.z = __shfl_sync(FULL, ds, b + 8);
                v.w = __shfl_sync(FULL, ds, b + 12);
                if ((lane & 15) == 0) {
                    const int64_t off = (peers.row_off + r0 + r) * H + (b >> 2);
                    if (peers.mode == 2) multimem_st_v4(peers.mc + off, v);
                    else
                        for (int g = 0; g < peers.n; ++g) *reinterpret_cast<float4*>(peers.ptr[g] + off) = v;
                }
            }
        }
        __syncthreads();                                // every warp is done with buffer b
    }
    mx = warp_max(mx);
    if (lane == 0 && mx > 0.f) atomicMax(xmax_bits, __float_as_uint(mx));   // non-negative floats order like their bits
}

// x16 [N, KP] = x [N, K] zero-padded to KP = round_up(K, 8) floats per row (16-byte aligned rows for the bulk copies)
__global__ void in_pad_kernel(const float* __restrict__ x, int64_t ldx, int64_t N, int K, int KP, float* __restrict__ x16)
{
    const int n4 = KP >> 2;
    const int64_t total = N * n4;
    for (int64_t idx = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; idx < total; idx += int64_t(gridDim.x) * blockDim.x) {
        const int64_t n = idx / n4;
        const int k = int(idx - n * n4) * 4;
        const float* p = x + n * ldx + k;
        float4 v;
        v.x = (k < K) ? p[0] : 0.f;
        v.y = (k + 1 < K) ? p[1] : 0.f;
        v.z = (k + 2 < K) ? p[2] : 0.f;
        v.w = (k + 3 < K) ? p[3] : 0.f;
        *reinterpret_cast<float4*>(x16 + n * KP + k) = v;
    }
}

// scal[0] = sx, [1] = sw, [2] = 1/(sx*sw*H), [3] = 1/sx;  one block
__global__ void in_scales_kernel(const float* __restrict__ W, int64_t n_w, const float* __restrict__ xmax, float* __restrict__ scal)
{
    __shared__ float red[32];
    float m = 0.f;
    for (int64_t i = threadIdx.x; i < n_w; i += blockDim.x) m = fmaxf(m, fabsf(W[i]));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        m = warp_max(m);
        if (threadIdx.x == 0) {
            const float sx = pow2_scale(*xmax), sw = pow2_scale(m);
            scal[0] = sx;
            scal[1] = sw;
            scal[2] = 1.f / (sx * sw * float(H));
            scal[3] = 1.f / sx;
        }
    }
}

// W image of out = Z W_r: k-block kb = features [64kb, 64kb+64), rows = c; element (c, f=(h,k)) = W[h*C+c, k] * sw
__global__ void in_wout_image_kernel(const float* __restrict__ W, int K, int KP, int NKB, const float* __restrict__ scal,
                                     uint8_t* __restrict__ img)
{
    const int kb = blockIdx.x;
    const float sw = scal[1];
    for (int idx = threadIdx.x; idx < C * 64; idx += blockDim.x) {
        const int c = idx >> 6, e = idx & 63;
        const int f = kb * 64 + e, h = f / KP, k = f - h * KP;
        float v = 0.f;
        if (h < H && k < K) v = W[int64_t(h * C + c) * K + k] * sw;
        const __half hi = __float2half_rn(v);
        const __half lo = __float2half_rn(v - __half2float(hi));
        const uint32_t off = plane_off(c, e);
        *reinterpret_cast<__half*>(img + size_t(kb) * 16384 + off) = hi;
        *reinterpret_cast<__half*>(img + size_t(kb) * 16384 + 8192 + off) = lo;
    }
}

// ---- sinks: what happens when a row (or a hub chunk) is complete --------------------------------------------------------
// lane l holds acc[h*NI + i] = features 2*(l + 32 i), +1 of head h's aggregated input (FeatGeo)
template <int N4>
struct ZSink {      // write the row of the fp16-pair image (the weights arrive normalised)
    using FG = FeatGeo<N4>;
    static constexpr int NA = H * FG::NI;
    uint8_t* zimg; const float* scal; int KP, NKB;
    __device__ __forceinline__ void write_row(int row, float2 (&acc)[NA], int lane) const
    {
        const int n2 = KP >> 1;
        const float f = scal[0];
        const uint32_t rr = uint32_t(row) & (TILE - 1);
        uint8_t* base = zimg + size_t(row >> 7) * size_t(NKB) * KBLOCK + (rr >> 3) * 1024u + (rr & 7u) * 128u;
#pragma unroll
        for (int i = 0; i < FG::NI; ++i)
            if (FG::valid(i, lane, n2)) {
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    // 2 consecutive features = 4 bytes per plane; the 32 lanes of one store cover 64 consecutive features
                    const uint32_t ft = uint32_t(h * KP + 64 * i + 2 * lane), kb = ft >> 6, e = ft & 63u;
                    __half2 hi, lo;
                    split_h2(acc[h * FG::NI + i].x * f, acc[h * FG::NI + i].y * f, hi, lo);
                    uint8_t* p = base + size_t(kb) * KBLOCK + (((e >> 3) ^ (rr & 7u)) << 4) + (e & 7u) * 2u;
                    *reinterpret_cast<__half2*>(p) = hi;
                    *reinterpret_cast<__half2*>(p + PLANE) = lo;
                }
            }
    }
    __device__ __forceinline__ void finish_norm(int row, float2 (&acc)[NA], int lane) const { write_row(row, acc, lane); }
    __device__ __forceinline__ void empty(int row, int lane) const
    {
        float2 acc[NA];
#pragma unroll
        for (int i = 0; i < NA; ++i) acc[i] = make_float2(0.f, 0.f);
        write_row(row, acc, lane);                         // the row statistics of an empty row are written by the alpha pass
    }
};
template <int N4>
struct ZPartialSink {   // hub chunk c: partial accumulator (the weights are normalised, so partials simply add)
    using FG = FeatGeo<N4>;
    static constexpr int NA = H * FG::NI;
    static constexpr int PART_ACC = NA * 32 * 2;          // floats of one partial accumulator set
    float* part_acc; int c;
    __device__ __forceinline__ void finish_partial(float2 (&acc)[NA], int lane) const
    {
        float2* p = reinterpret_cast<float2*>(part_acc + int64_t(c) * PART_ACC);
#pragma unroll
        for (int i = 0; i < NA; ++i) p[i * 32 + lane] = acc[i];
    }
    __device__ __forceinline__ void finish_norm(int, float2 (&)[NA], int) const {}
    __device__ __forceinline__ void empty(int, int) const {}
};

template <int NA>
__device__ __forceinline__ void acc_zero(float2 (&acc)[NA])
{
#pragma unroll
    for (int i = 0; i < NA; ++i) acc[i] = make_float2(0.f, 0.f);
}

// =====================================================================================================================
// Pass 1: attention coefficients.  alpha [E',H] in CSR order, NORMALISED, before dropout; the sign bit of alpha[e,h] says
// that the logit was in LeakyReLU's negative region (the backward needs that and nothing else of the logits), and
// jflag[e] = col[e] | (e is the last edge of its row) << 31.  The feature passes (forward and backward) then stream
// edges without any softmax state: no logit gathers, no exp, no scans, no row statistics in their registers.
// The kernels run the attention pass of gat_alpha.cuh (PROJ = false) at H = 8, without dropout: the feature passes apply it.
// =====================================================================================================================
__global__ void __launch_bounds__(IN_THREADS)
in_alpha_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
               const float* __restrict__ a_dst, gnnfd_item_plan_t items, int hub_threshold, float slope,
               AlphaOut out, float* __restrict__ rowmax, float* __restrict__ rowsum)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * IN_WARPS + warp;
    if (item >= items.n_items) return;
    alpha_items_body<H, false, false>(rowptr, col, a_src, a_dst, items.item_start[item], items.item_start[item + 1],
                                      hub_threshold, slope, out, rowmax, rowsum, lane);
}

// hub rows: (1) statistics of every 512-edge chunk, (2) one thread per (hub row, head) folds them in chunk order, (3) write sweep
__global__ void __launch_bounds__(IN_THREADS)
in_alpha_hub_stats(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
                   const float* __restrict__ a_dst, gnnfd_hub_plan_t plan, float slope, float* __restrict__ part_ms)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * IN_WARPS + warp;
    if (c >= plan.n_chunk) return;
    alpha_hub_stats_body<H>(rowptr, col, a_src, a_dst, plan, c, slope, part_ms, lane);
}
__global__ void in_alpha_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part_ms, float* __restrict__ rowmax,
                                   float* __restrict__ rowsum)
{
    if (threadIdx.x >= H) return;
    alpha_hub_merge_body<H>(plan, blockIdx.x, threadIdx.x, part_ms, rowmax, rowsum);
}
__global__ void __launch_bounds__(IN_THREADS)
in_alpha_hub_write(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ a_src,
                   const float* __restrict__ a_dst, gnnfd_hub_plan_t plan, float slope, const float* __restrict__ rowmax,
                   const float* __restrict__ rowsum, AlphaOut out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * IN_WARPS + warp;
    if (c >= plan.n_chunk) return;
    alpha_hub_write_body<H, false, false>(rowptr, col, a_src, a_dst, plan, c, slope, rowmax, rowsum, out, lane);
}

// =====================================================================================================================
// Pass 2: Z[i,h,:] = sum_e alpha_used[e,h] x[col[e],:].  The stream needs only the edge range of its rows: per chunk of <= 32
// edges lane = edge loads alpha (32 B) and jflag (4 B) -- coalesced, nothing depends on a gathered value -- one chunk ahead
// of the feature traffic; dropout is applied while staging.  Row ends come from the flag bit, so packs and single rows
// are the same code.
// =====================================================================================================================
struct FeatChunk {
    int row, beg, n;
    unsigned lastmask;      // staged edges that end a row
};

template <bool DROPOUT>
__device__ __forceinline__ void stage_chunk(FeatChunk& c, const float* __restrict__ alpha, const int32_t* __restrict__ jflag,
                                            const int32_t* __restrict__ perm, KeepMask keep, float keep_scale, float* p_s, int* j_s,
                                            int lane)
{
    int jf = 0;
    float w[H];
    if (lane < c.n) {
        const int e = c.beg + lane;
        jf = jflag[e];
        load_vecH<H>(alpha + int64_t(e) * H, w);
        unsigned kbits = 0xffu;
        if (DROPOUT) kbits = keep.bits(perm[e], H);
#pragma unroll
        for (int h = 0; h < H; ++h) w[h] = ((kbits >> h) & 1u) ? fabsf(w[h]) * (DROPOUT ? keep_scale : 1.f) : 0.f;
    } else {
#pragma unroll
        for (int h = 0; h < H; ++h) w[h] = 0.f;
    }
    store_vecH<H>(p_s + lane * H, w);
    j_s[lane] = jf & 0x7fffffff;
    c.lastmask = __ballot_sync(FULL, jf < 0);
    __syncwarp();
}

// HUB: one (row, range) segment whose partial sum goes to the sink at the end; else whole rows and packs of rows,
// finished at the flags
template <int N4, bool DROPOUT, bool HUB, class Sink>
__device__ __forceinline__ void in_fwd_stream(ChunkCursor& cur, InRing& ring, const Sink& sink, const int32_t* __restrict__ rowptr,
                                              const int32_t* __restrict__ perm, int n4, const float* __restrict__ alpha,
                                              const int32_t* __restrict__ jflag, KeepMask keep, float keep_scale, int lane)
{
    using FG = FeatGeo<N4>;
    constexpr int NA = H * FG::NI;
    (void)n4;
    auto on_empty = [&](int r) { sink.empty(r, lane); };
    FeatChunk c0, c1;
    int b0 = 0;
    auto next = [&](FeatChunk& c) -> bool {
        bool first, last;
        int k, la, lb;
        if (!HUB) return cur.next_any(rowptr, lane, c.row, c.beg, c.n, first, last, k, la, lb, on_empty) != 0;
        return cur.next(rowptr, c.row, c.beg, c.n, first, last, on_empty);
    };
    if (!next(c0)) return;
    stage_chunk<DROPOUT>(c0, alpha, jflag, perm, keep, keep_scale, ring.p_s + b0 * 32 * H, ring.j_s + b0 * 32, lane);
    int issued0 = 0, issued1 = 0;
    float2 acc[NA];
    acc_zero(acc);
    while (true) {
        const int* j0 = ring.j_s + b0 * 32;
        const int* j1 = ring.j_s + (b0 ^ 1) * 32;
        {
            const int k0 = min(ring.room(), c0.n - issued0);
            if (k0 > 0) { ring.issue_many(j0 + issued0, k0, lane); issued0 += k0; }
        }
        const bool more = next(c1);
        issued1 = 0;
        if (more) stage_chunk<DROPOUT>(c1, alpha, jflag, perm, keep, keep_scale, ring.p_s + (b0 ^ 1) * 32 * H, ring.j_s + (b0 ^ 1) * 32, lane);
        const uint32_t p0 = st_smem_u32(ring.p_s + b0 * 32 * H);
        const unsigned lastmask = HUB ? 0u : c0.lastmask;
        // edges in groups of four: one warp barrier and one (multi-lane) refill per group
        for (int t0 = 0; t0 < c0.n; t0 += 4) {
            const int cnt = min(4, c0.n - t0);
#pragma unroll IN_UNROLL_FWD
            for (int r = 0; r < 4; ++r) {
                if (r < cnt) {
                    const int t = t0 + r;
                    const uint32_t a = ring.front_at(r) + uint32_t(lane) * 8u;
                    const float4 w0 = lds128(p0 + uint32_t(t) * (H * 4u)), w1 = lds128(p0 + uint32_t(t) * (H * 4u) + 16u);   // broadcast
                    const float w[H] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
                    // no validity predicate here: a lane beyond the row's end reads the bytes that follow the slot (inside this
                    // warp's shared memory) into accumulators that the sinks never write out -- cheaper than a divergent tail
#pragma unroll
                    for (int i = 0; i < FG::NI; ++i) {
                        const float2 v = lds64(a + uint32_t(i) * 256u);
#pragma unroll
                        for (int hh = 0; hh < H; ++hh) ffma2_bcast(acc[hh * FG::NI + i].x, acc[hh * FG::NI + i].y, w[hh], v.x, v.y);
                    }
                    if ((lastmask >> t) & 1u) {           // last edge of a row (weights are normalised)
                        sink.finish_norm(c0.row + __popc(lastmask & ((1u << t) - 1u)), acc, lane);
                        acc_zero(acc);
                    }
                }
            }
            ring.pop_many(cnt);
            int free_slots = cnt;
            const int k0 = min(free_slots, c0.n - issued0);
            if (k0 > 0) { ring.issue_many(j0 + issued0, k0, lane); issued0 += k0; free_slots -= k0; }
            if (more && free_slots > 0) {
                const int k1 = min(free_slots, c1.n - issued1);
                if (k1 > 0) { ring.issue_many(j1 + issued1, k1, lane); issued1 += k1; }
            }
        }
        if (!more) break;
        c0 = c1;
        issued0 = issued1;
        b0 ^= 1;
    }
    if constexpr (HUB) sink.finish_partial(acc, lane);
}

constexpr int FWD_EXTRA = 0;
constexpr int IN_FWD_CTAS = 5;

template <int N4, bool DROPOUT>
__global__ void __launch_bounds__(IN_THREADS, IN_FWD_CTAS)
gat_in_fwd_items(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, const float* __restrict__ x, int64_t ldx,
                 const float* __restrict__ alpha, const int32_t* __restrict__ jflag, gnnfd_item_plan_t items, int hub_threshold,
                 KeepMask keep, float keep_scale, ZSink<N4> sink)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * IN_WARPS + warp;
    if (item >= items.n_items) return;
    InRing ring;
    ring.init(smem + warp * in_warp_bytes(sink.KP, FWD_EXTRA), x, ldx, sink.KP, lane);
    ChunkCursor cur;
    cur.start_rows(items.item_start[item], items.item_start[item + 1], hub_threshold);
    in_fwd_stream<N4, DROPOUT, false>(cur, ring, sink, rowptr, perm, sink.KP >> 2, alpha, jflag, keep, keep_scale, lane);
}

// one warp per (hub row, chunk): partial accumulators
template <int N4, bool DROPOUT>
__global__ void __launch_bounds__(IN_THREADS, IN_FWD_CTAS)
gat_in_fwd_hub_chunks(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, const float* __restrict__ x, int64_t ldx,
                      int KP, const float* __restrict__ alpha, const int32_t* __restrict__ jflag, gnnfd_hub_plan_t plan,
                      KeepMask keep, float keep_scale, float* __restrict__ part_acc)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * IN_WARPS + warp;
    if (c >= plan.n_chunk) return;
    const int slot = plan.chunk_hub[c];
    const int i = plan.hub_row[slot];
    const int beg = rowptr[i] + (c - plan.hub_chunk_ptr[slot]) * plan.chunk;
    const int end = min(rowptr[i + 1], beg + plan.chunk);
    InRing ring;
    ring.init(smem + warp * in_warp_bytes(KP, FWD_EXTRA), x, ldx, KP, lane);
    ChunkCursor cur;
    cur.start_segment(i, beg, end);
    ZPartialSink<N4> sink{part_acc, c};
    in_fwd_stream<N4, DROPOUT, true>(cur, ring, sink, rowptr, perm, KP >> 2, alpha, jflag, keep, keep_scale, lane);
}

// one CTA per hub row: warp w sums chunks w, w+8, ..., the eight warp sums are added in warp order -- a fixed order, so the
// result is deterministic
template <int N4>
__global__ void __launch_bounds__(ROW_THREADS)
gat_in_fwd_hub_merge(gnnfd_hub_plan_t plan, const float* __restrict__ part_acc, ZSink<N4> sink)
{
    constexpr int NA = ZSink<N4>::NA;
    constexpr int PART_ACC = ZPartialSink<N4>::PART_ACC;
    extern __shared__ __align__(16) float msm[];               // [ROW_WARPS][PART_ACC]
    float2* st_acc = reinterpret_cast<float2*>(msm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int i = plan.hub_row[slot];
    const int c0 = plan.hub_chunk_ptr[slot], c1 = plan.hub_chunk_ptr[slot + 1];
    float2 acc[NA];
    acc_zero(acc);
    auto add = [&](const float2* __restrict__ pacc) {
#pragma unroll
        for (int k = 0; k < NA; ++k) {
            const float2 v = pacc[k * 32 + lane];
            acc[k].x += v.x; acc[k].y += v.y;
        }
    };
    for (int c = c0 + warp; c < c1; c += ROW_WARPS) add(reinterpret_cast<const float2*>(part_acc + int64_t(c) * PART_ACC));
#pragma unroll
    for (int k = 0; k < NA; ++k) st_acc[warp * (PART_ACC / 2) + k * 32 + lane] = acc[k];
    __syncthreads();
    if (warp != 0) return;
    for (int w = 1; w < ROW_WARPS; ++w) add(st_acc + w * (PART_ACC / 2));
    sink.finish_norm(i, acc, lane);
}

template <class Kn>
static int in_set_smem(Kn kernel, int bytes)
{
    GNNFD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return GNNFD_OK;
}

// x as the edge kernels need it: 16-byte aligned rows of at least KP floats
bool in_x_ok(const float* x, int64_t ldx, int KP) { return (reinterpret_cast<uintptr_t>(x) & 15) == 0 && ldx % 4 == 0 && ldx >= KP; }

// attention pass: alpha / jflag for every edge, rowmax / rowsum for every row
static int launch_in_alpha(const gnnfd_graph_t* g, const float* a_src, const float* a_dst, float slope, float* alpha, int32_t* jflag,
                           float* rowmax, float* rowsum, void* ws, size_t ws_bytes, cudaStream_t st)
{
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const unsigned grid = (unsigned)((g->items_dst.n_items + IN_WARPS - 1) / IN_WARPS);
    const AlphaOut out{alpha, jflag, nullptr, KeepMask(), 1.f};
    in_alpha_items<<<grid, IN_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, g->items_dst, thr, slope, out, rowmax, rowsum);
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const size_t need = carve_bytes(size_t(pl.n_chunk) * 2 * H, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "in_fwd: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        float* part_ms = carve<float>(p, size_t(pl.n_chunk) * 2 * H);
        const unsigned gc = (unsigned)((pl.n_chunk + IN_WARPS - 1) / IN_WARPS);
        in_alpha_hub_stats<<<gc, IN_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, pl, slope, part_ms);
        in_alpha_hub_merge<<<(unsigned)pl.n_hub, 32, 0, st>>>(pl, part_ms, rowmax, rowsum);
        in_alpha_hub_write<<<gc, IN_THREADS, 0, st>>>(g->rowptr, g->col, a_src, a_dst, pl, slope, rowmax, rowsum, out);
        g_launches += 3;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

template <int N4>
static int launch_in_fwd(const gnnfd_graph_t* g, const float* x, int64_t ldx, const Dims& d, const float* alpha, const int32_t* jflag,
                         const uint8_t* keep_mask, float p_drop, uint64_t seed, const float* scal, void* zimg, void* ws,
                         size_t ws_bytes, cudaStream_t st)
{
    const bool drop = p_drop > 0.f;              // explicit mask, or (mask == NULL) the counter-based RNG keyed on seed
    float ks = 1.f;
    const KeepMask keep = make_keep(keep_mask, p_drop, seed, &ks);
    const int thr = g->hub_dst.n_hub > 0 ? g->hub_dst.threshold : INT_MAX;
    const int smem = IN_WARPS * in_warp_bytes(d.KP, FWD_EXTRA);
    const unsigned grid = (unsigned)((g->items_dst.n_items + IN_WARPS - 1) / IN_WARPS);
    ZSink<N4> sink{reinterpret_cast<uint8_t*>(zimg), scal, d.KP, d.NKB};
    int rc = GNNFD_OK;
#define GNNFD_IN_FWD(DD)                                                                                               \
    rc = in_set_smem(gat_in_fwd_items<N4, DD>, smem);                                                                  \
    if (rc) return rc;                                                                                                 \
    gat_in_fwd_items<N4, DD><<<grid, IN_THREADS, smem, st>>>(g->rowptr, g->perm, x, ldx, alpha, jflag, g->items_dst, thr, keep, ks, \
                                                             sink)
    if (drop) { GNNFD_IN_FWD(true); } else { GNNFD_IN_FWD(false); }
#undef GNNFD_IN_FWD
    g_launches += 1;
    if (g->hub_dst.n_hub > 0) {
        constexpr int PART_ACC = ZPartialSink<N4>::PART_ACC;
        const gnnfd_hub_plan_t& pl = g->hub_dst;
        const size_t need = carve_bytes(size_t(pl.n_chunk) * 2 * H, 4) + carve_bytes(size_t(pl.n_chunk) * PART_ACC, 4);
        GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "in_fwd: workspace %zu < %zu", ws_bytes, need);
        char* p = reinterpret_cast<char*>(ws);
        carve<float>(p, size_t(pl.n_chunk) * 2 * H);           // (the attention pass's chunk statistics)
        float* part_acc = carve<float>(p, size_t(pl.n_chunk) * PART_ACC);
        const unsigned gc = (unsigned)((pl.n_chunk + IN_WARPS - 1) / IN_WARPS);
        if (drop) {
            rc = in_set_smem(gat_in_fwd_hub_chunks<N4, true>, smem);
            if (rc) return rc;
            gat_in_fwd_hub_chunks<N4, true><<<gc, IN_THREADS, smem, st>>>(g->rowptr, g->perm, x, ldx, d.KP, alpha, jflag, pl, keep, ks, part_acc);
        } else {
            rc = in_set_smem(gat_in_fwd_hub_chunks<N4, false>, smem);
            if (rc) return rc;
            gat_in_fwd_hub_chunks<N4, false><<<gc, IN_THREADS, smem, st>>>(g->rowptr, g->perm, x, ldx, d.KP, alpha, jflag, pl, keep, ks, part_acc);
        }
        const int msm = ROW_WARPS * PART_ACC * 4;
        rc = in_set_smem(gat_in_fwd_hub_merge<N4>, msm);
        if (rc) return rc;
        gat_in_fwd_hub_merge<N4><<<(unsigned)pl.n_hub, ROW_THREADS, msm, st>>>(pl, part_acc, sink);
        g_launches += 2;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace in
}  // namespace gnnfd

using namespace gnnfd;
using namespace gnnfd::in;

extern "C" {

int gnnfd_in_supported(int64_t K, int H_, int C_, int concat)
{
    return (K >= 1 && K <= MAX_K && H_ == H && C_ == C && !concat) ? 1 : 0;
}

int gnnfd_in_sizes(int64_t n_dst, int64_t K, size_t* prep_bytes_out, size_t* zimg_bytes_out, int64_t* gd_ld_out,
                   int64_t* x_ld_out)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && n_dst >= 0, GNNFD_ERR_ARG, "in_sizes: K must be in [1,%d]", MAX_K);
    const Dims d((int)K);
    if (prep_bytes_out) *prep_bytes_out = prep_bytes(d);
    if (zimg_bytes_out) *zimg_bytes_out = zimg_bytes(n_dst, d) + 1024;
    if (gd_ld_out) *gd_ld_out = d.F;
    if (x_ld_out) *x_ld_out = d.KP;
    return GNNFD_OK;
}

/* x16 [N, x_ld] (x_ld = gnnfd_in_sizes' x_ld) = x zero-padded: 16-byte aligned rows for the bulk-copy gathers. */
int gnnfd_in_pad_x(const float* x, int64_t ldx, int64_t N, int64_t K, float* x16, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && ldx >= K && N >= 0, GNNFD_ERR_ARG, "in_pad_x: bad shape");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(x && x16 && (reinterpret_cast<uintptr_t>(x16) & 15) == 0, GNNFD_ERR_ARG, "in_pad_x: NULL or misaligned tensor");
    const Dims d((int)K);
    int64_t blocks = (N * (d.KP / 4) + 255) / 256;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    in_pad_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, N, d.K, d.KP, x16);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* a_src / a_dst [N,H] for rows [0,N) of x, and xmax[0] = max(xmax[0], max |x|) (caller zeroes xmax before the first call;
 * across GPUs the per-rank maxima are max-reduced before gnnfd_in_prepare).  x: padded rows (gnnfd_in_pad_x layout). */
static int in_logits_launch(const float* x, int64_t ldx, int64_t N, int64_t K, const float* W, const float* att_src,
                            const float* att_dst, float* a_src, float* a_dst, float* xmax, void* prep, const PeerRows& peers,
                            cudaStream_t st)
{
    const Dims d((int)K);
    GNNFD_REQUIRE(N == 0 || in_x_ok(x, ldx, d.KP), GNNFD_ERR_ARG,
                  "in_logits: x rows must be 16-byte aligned and zero-padded to %d floats (gnnfd_in_pad_x)", d.KP);
    float* u = reinterpret_cast<float*>(reinterpret_cast<char*>(prep) + prep_off_u(d));
    in_u_kernel<<<2 * H, 192, 0, st>>>(W, att_src, att_dst, d.K, d.KP, u);
    g_launches += 1;
    if (N > 0) {
        const int64_t n_tiles = (N + LG_ROWS - 1) / LG_ROWS;
        const int64_t cap = int64_t(sm_count()) * 2;
        const unsigned blocks = (unsigned)(n_tiles < cap ? n_tiles : cap);
        const int smem = 2 * LG_ROWS * d.KP * 4;
        unsigned* xb = reinterpret_cast<unsigned*>(xmax);
        int rc;
        if (d.KP == 168) {
            rc = in_set_smem(in_logits_kernel<42>, smem);
            if (rc) return rc;
            in_logits_kernel<42><<<blocks, LG_WARPS * 32, smem, st>>>(x, ldx, N, d.KP, u, a_src, a_dst, xb, peers);
        } else if (d.KP == 64) {
            rc = in_set_smem(in_logits_kernel<16>, smem);
            if (rc) return rc;
            in_logits_kernel<16><<<blocks, LG_WARPS * 32, smem, st>>>(x, ldx, N, d.KP, u, a_src, a_dst, xb, peers);
        } else {
            rc = in_set_smem(in_logits_kernel<0>, smem);
            if (rc) return rc;
            in_logits_kernel<0><<<blocks, LG_WARPS * 32, smem, st>>>(x, ldx, N, d.KP, u, a_src, a_dst, xb, peers);
        }
        g_launches += 1;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int gnnfd_in_logits(const float* x, int64_t ldx, int64_t N, int64_t K, const float* W, const float* att_src,
                    const float* att_dst, float* a_src, float* a_dst, float* xmax, void* prep, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && N >= 0, GNNFD_ERR_ARG, "in_logits: bad shape (K <= %d)", MAX_K);
    GNNFD_REQUIRE(W && att_src && att_dst && xmax && prep, GNNFD_ERR_ARG, "in_logits: NULL argument");
    GNNFD_REQUIRE(N == 0 || (x && a_src && a_dst), GNNFD_ERR_ARG, "in_logits: NULL tensor");
    PeerRows peers{};
    return in_logits_launch(x, ldx, N, K, W, att_src, att_dst, a_src, a_dst, xmax, prep, peers, (cudaStream_t)stream);
}

int gnnfd_in_logits_bcast(const float* x, int64_t ldx, int64_t N, int64_t K, const float* W, const float* att_src,
                          const float* att_dst, const gnnfd_peers_t* a_src_all, int64_t row_offset, int use_multicast,
                          float* a_dst, float* xmax, void* prep, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && N >= 0 && row_offset >= 0, GNNFD_ERR_ARG, "in_logits_bcast: bad shape (K <= %d)", MAX_K);
    GNNFD_REQUIRE(W && att_src && att_dst && xmax && prep && a_src_all, GNNFD_ERR_ARG, "in_logits_bcast: NULL argument");
    GNNFD_REQUIRE(N == 0 || (x && a_dst), GNNFD_ERR_ARG, "in_logits_bcast: NULL tensor");
    PeerRows peers;
    const int rc = peer_rows_from(a_src_all, row_offset, use_multicast, "in_logits_bcast", peers);
    if (rc) return rc;
    return in_logits_launch(x, ldx, N, K, W, att_src, att_dst, nullptr, a_dst, xmax, prep, peers, (cudaStream_t)stream);
}

/* scales + W images of the two dense stages into prep (gnnfd_in_sizes gives its size). */
int gnnfd_in_prepare(const float* W, int64_t K, const float* xmax, void* prep, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && W && xmax && prep, GNNFD_ERR_ARG, "in_prepare: bad argument");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(prep) & 1023) == 0, GNNFD_ERR_ARG, "in_prepare: prep must be 1024-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const Dims d((int)K);
    char* p = reinterpret_cast<char*>(prep);
    float* scal = reinterpret_cast<float*>(p);
    in_scales_kernel<<<1, 1024, 0, st>>>(W, int64_t(H) * C * K, xmax, scal);
    in_wout_image_kernel<<<d.NKB, 256, 0, st>>>(W, d.K, d.KP, d.NKB, scal, reinterpret_cast<uint8_t*>(p + prep_off_wout(d)));
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return in_build_gd_image(W, d.K, prep, st);
}

int gnnfd_in_fwd_workspace_bytes(const gnnfd_graph_t* g, size_t* bytes)
{
    GNNFD_REQUIRE(g && bytes, GNNFD_ERR_ARG, "in_fwd_workspace_bytes: NULL argument");
    const size_t nc = (size_t)g->hub_dst.n_chunk;
    *bytes = carve_bytes(nc * 2 * H, 4) + carve_bytes(nc * size_t(ZPartialSink<0>::PART_ACC), 4) + 256;
    return GNNFD_OK;
}

/* Aggregation in input space.  Pass 1 writes the attention coefficients alpha [E',H] (CSR order, normalised, sign bit =
 * LeakyReLU negative region), jflag [E'] (source id | row-end flag) and rowmax / rowsum [n_dst,H]; pass 2 streams the edges
 * and writes zimg (fp16-pair image of Z, rows = destinations).  alpha and jflag are what the backward reads. */
int gnnfd_in_fwd(const gnnfd_graph_t* g, const float* x, int64_t ldx, int64_t K, const float* a_src, const float* a_dst,
                 float negative_slope, const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, const void* prep, void* zimg,
                 float* rowmax, float* rowsum, float* alpha, int32_t* jflag, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    int rc = check_graph(g, false, "in_fwd");
    if (rc) return rc;
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K, GNNFD_ERR_ARG, "in_fwd: bad shape (K <= %d)", MAX_K);
    GNNFD_REQUIRE(g->n_dst == 0 || (x && a_src && a_dst && prep && zimg && rowmax && rowsum), GNNFD_ERR_ARG, "in_fwd: NULL tensor");
    GNNFD_REQUIRE(g->n_edges == 0 || (alpha && jflag), GNNFD_ERR_ARG, "in_fwd: NULL alpha / jflag");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(alpha) & 15) == 0, GNNFD_ERR_ARG, "in_fwd: alpha must be 16-byte aligned");
    GNNFD_REQUIRE(p_drop >= 0.f && p_drop <= 0.9f, GNNFD_ERR_ARG, "in_fwd: dropout p must be in [0,0.9] on the input-space path");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(zimg) & 1023) == 0, GNNFD_ERR_ARG, "in_fwd: zimg must be 1024-byte aligned");
    if (g->n_dst == 0) return GNNFD_OK;
    const Dims d((int)K);
    GNNFD_REQUIRE(in_x_ok(x, ldx, d.KP), GNNFD_ERR_ARG,
                  "in_fwd: x rows must be 16-byte aligned and zero-padded to %d floats (gnnfd_in_pad_x)", d.KP);
    GNNFD_REQUIRE(g->items_dst.n_items > 0 && g->items_dst.item_start, GNNFD_ERR_ARG,
                  "in_fwd: the graph has no work-item plan over rowptr (gnnfd_item_plan)");
    cudaStream_t st = (cudaStream_t)stream;
    const float* scal = reinterpret_cast<const float*>(prep);
    // rows of the last tile beyond n_dst are read by the node-reduction GEMM (dW): they must be zero, not stale
    if (g->n_dst % TILE) {
        const size_t last = size_t(g->n_dst / TILE) * d.NKB * KBLOCK;
        GNNFD_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(zimg) + last, 0, size_t(d.NKB) * KBLOCK, st));
    }
    rc = launch_in_alpha(g, a_src, a_dst, negative_slope, alpha, jflag, rowmax, rowsum, ws, ws_bytes, st);
    if (rc) return rc;
    if (d.KP == 168) return launch_in_fwd<42>(g, x, ldx, d, alpha, jflag, keep_mask, p_drop, dropout_seed, scal, zimg, ws, ws_bytes, st);
    if (d.KP == 64) return launch_in_fwd<16>(g, x, ldx, d, alpha, jflag, keep_mask, p_drop, dropout_seed, scal, zimg, ws, ws_bytes, st);
    return launch_in_fwd<0>(g, x, ldx, d, alpha, jflag, keep_mask, p_drop, dropout_seed, scal, zimg, ws, ws_bytes, st);
}

}  // extern "C"
