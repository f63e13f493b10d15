// Dense stages of the input-space GAT layer (in_common.cuh) on the 5th-gen tensor cores, fed by the bulk-copy engine.
//
//   in_out_gemm   out[n, C]  = epi( Z[n, F] @ W_r[F, C] )         K-major A = the fp16-pair image written by gnnfd_in_fwd
//   in_dw_gemm    dWr[F, C]  = Z[n, F]^T @ dO[n, C]               MN-major A = the SAME image, reduction over nodes
//
// Both read Z as ready-made 128B-swizzled shared-memory tiles: one cp.async.bulk per k-block (32 KB: fp16 hi plane +
// fp16 lo plane), completion on an mbarrier, no operand-staging warps.  Error-compensated fp16 arithmetic:
// v*s = hi + lo with s a power of two chosen so that max|v|*s is in [2^11, 2^12); the three products hi*hi, hi*lo,
// lo*hi are accumulated in fp32 in TMEM (kind::f16), which carries 22 mantissa bits per operand -- the same accuracy
// class as the 3xTF32 projection (project_tc.cu) at half the operand bytes.  One elected thread issues the MMAs;
// tcgen05.commit releases smem stages / hands accumulators to the epilogue warps.
//
// Replaces, for the reference's first layer (src/models/gat.py:39,80), the dense part of GATConv.forward
// (lin_src + head mean + bias) and of its autograd mirror (dW), cf. gnnfd_project_fwd / gnnfd_project_bwd.
#include "in_common.cuh"

#include <atomic>

namespace gnnfd {
extern std::atomic<long long> g_launches;
int check_graph(const gnnfd_graph_t* g, bool need_csc, const char* who);
size_t in_param_ws_bytes(int64_t N, int64_t K);                                                                     // project_simt.cu
int in_param_grads_simt(const float* x, int64_t ldx, const float* W, const float* da_src, const float* da_dst,
                        const float* d_out, int64_t N, int64_t K, float* datt_src, float* datt_dst, float* dbias,
                        float* Gm, void* ws, size_t ws_bytes, cudaStream_t st);

namespace in {

// ---- PTX wrappers ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(st_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(st_smem_u32(smem_dst)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(st_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version = 1 [46,48), layout type [61,64) = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= uint64_t((saddr & 0x3FFFF) >> 4);
    d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= uint64_t(1) << 46;
    d |= uint64_t(2) << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor), kind::f16: D = F32 [4,6) = 1, A = F16 [7,10) = 0, B = F16 [10,13) = 0,
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N, int a_mn, int b_mn)
{
    return (1u << 4) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

// ======================================================================================================================
// out = epi(Z W_r):  persistent, one CTA per SM, 6 warps: bulk-copy producer, MMA issuer, 4 epilogue warps
// ======================================================================================================================
constexpr int G1_STAGES = 4;
constexpr uint32_t G1_A = KBLOCK;                  // 32 KB: hi + lo planes of one k-block of one 128-row tile
constexpr uint32_t G1_B = 16384;                   // hi + lo [64 x 128 B] of the W image
constexpr uint32_t G1_STAGE = G1_A + G1_B;
constexpr int G1_THREADS = 192;
constexpr int G1_STG_LD = 36;
constexpr size_t G1_SMEM = size_t(G1_STAGES) * G1_STAGE + 4 * 32 * G1_STG_LD * 4 + 1024;

struct OutEpi {
    const float* bias;
    const float* scale;
    const float* shift;
    const float* residual;
    int act;
};
__device__ __forceinline__ float out_act(float v, int act)
{
    if (act == GNNFD_ACT_RELU) return fmaxf(v, 0.f);
    if (act == GNNFD_ACT_ELU) return v > 0.f ? v : expm1f(v);
    return v;
}

// PM: where the finished rows go besides `out` (PeerRows::mode; 0: `out` only, 1 / 2: also row (row_off + r) on every rank,
// `out` optional)
template <int PM>
__global__ void __launch_bounds__(G1_THREADS, 1)
in_out_gemm(const uint8_t* __restrict__ zimg, const uint8_t* __restrict__ wimg, const float* __restrict__ scal, int64_t n,
            int NKB, OutEpi ep, float* __restrict__ out, PeerRows peers)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full[G1_STAGES], empty[G1_STAGES], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int64_t n_tiles = (n + TILE - 1) / TILE;

    if (tid == 0) {
        for (int s = 0; s < G1_STAGES; ++s) {
            st_mbar_init(&full[s], 1);
            st_mbar_init(&empty[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            st_mbar_init(&acc_full[s], 1);
            st_mbar_init(&acc_empty[s], 4);
        }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ---------------- producer: one 32 KB copy of Z and one 16 KB copy of W per k-block -----------------------
        int64_t step = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            for (int kb = 0; kb < NKB; ++kb, ++step) {
                const int s = int(step % G1_STAGES);
                const int64_t u = step / G1_STAGES;
                if (u > 0) st_mbar_wait(&empty[s], uint32_t((u - 1) & 1));
                if (elect_one()) {
                    uint8_t* stage = smem + size_t(s) * G1_STAGE;
                    st_mbar_expect_tx(&full[s], G1_STAGE);
                    st_bulk_g2s(stage, zimg + (size_t(t) * NKB + kb) * KBLOCK, G1_A, &full[s]);
                    st_bulk_g2s(stage + G1_A, wimg + size_t(kb) * G1_B, G1_B, &full[s]);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issue --------------------------------------------------------------------------------
        constexpr uint32_t IDESC = make_idesc_f16(128, C, 0, 0);
        int64_t step = 0, j = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
            const int buf = int(j & 1);
            if ((j >> 1) > 0) {
                st_mbar_wait(&acc_empty[buf], uint32_t(((j >> 1) - 1) & 1));
                tc_fence_after();
            }
            for (int kb = 0; kb < NKB; ++kb, ++step) {
                const int s = int(step % G1_STAGES);
                st_mbar_wait(&full[s], uint32_t((step / G1_STAGES) & 1));
                tc_fence_after();
                const uint32_t a_hi = st_smem_u32(smem + size_t(s) * G1_STAGE), a_lo = a_hi + PLANE;
                const uint32_t b_hi = a_hi + G1_A, b_lo = b_hi + 8192;
                // two accumulators per tile (even / odd k-blocks) halve the length of the round-toward-zero chain
                const uint32_t d = tmem_base + uint32_t(buf * 128 + (kb & 1) * 64);
                if (elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint32_t ko = ks * 32;            // 16 fp16 = 32 bytes inside the swizzled row
                        const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                        const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                        umma_f16(d, dah, dbh, IDESC, (kb >= 2 || ks > 0) ? 1u : 0u);
                        umma_f16(d, dah, dbl, IDESC, 1u);
                        umma_f16(d, dal, dbh, IDESC, 1u);
                    }
                    umma_commit(&empty[s]);
                    if (kb == NKB - 1) umma_commit(&acc_full[buf]);
                }
                __syncwarp();
            }
        }
    } else {
        // ---------------- epilogue: warps 2..5 -> TMEM lane quadrants 2,3,0,1 -----------------------------------------
        const int quad = warp & 3;
        float* stg = reinterpret_cast<float*>(smem + size_t(G1_STAGES) * G1_STAGE) + (warp - 2) * (32 * G1_STG_LD);
        const float inv = scal[2];
        int64_t j = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
            const int buf = int(j & 1);
            st_mbar_wait(&acc_full[buf], uint32_t((j >> 1) & 1));
            tc_fence_after();
            const int64_t m0 = t * TILE + quad * 32;
#pragma unroll 1
            for (int ch = 0; ch < C / 32; ++ch) {
                uint32_t v0[32], v1[32];
                tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(buf * 128 + ch * 32), v0);
                if (NKB > 1) {
                    tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(buf * 128 + 64 + ch * 32), v1);
#pragma unroll
                    for (int c = 0; c < 32; ++c) v0[c] = __float_as_uint(__uint_as_float(v0[c]) + __uint_as_float(v1[c]));
                }
                __syncwarp();
#pragma unroll
                for (int c = 0; c < 32; c += 4)
                    *reinterpret_cast<float4*>(stg + lane * G1_STG_LD + c) =
                        make_float4(__uint_as_float(v0[c]), __uint_as_float(v0[c + 1]), __uint_as_float(v0[c + 2]),
                                    __uint_as_float(v0[c + 3]));
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + (lane >> 3), cq = ch * 32 + (lane & 7) * 4;
                    const int64_t gm = m0 + r;
                    const float4 o = *reinterpret_cast<const float4*>(stg + r * G1_STG_LD + (lane & 7) * 4);
                    if (gm < n) {
                        float ov[4] = {o.x * inv, o.y * inv, o.z * inv, o.w * inv};
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            float v = ov[k] + (ep.bias ? ep.bias[cq + k] : 0.f);
                            if (ep.scale) v = fmaf(v, ep.scale[cq + k], ep.shift[cq + k]);
                            v = out_act(v, ep.act);
                            if (ep.residual) v += ep.residual[gm * C + cq + k];
                            ov[k] = v;
                        }
                        const float4 o4 = make_float4(ov[0], ov[1], ov[2], ov[3]);
                        if (PM == 0 || out) *reinterpret_cast<float4*>(out + gm * C + cq) = o4;
                        const int64_t po = (peers.row_off + gm) * C + cq;
                        if (PM == 1)
                            for (int g = 0; g < peers.n; ++g) *reinterpret_cast<float4*>(peers.ptr[g] + po) = o4;
                        else if (PM == 2)
                            multimem_st_v4(peers.mc + po, o4);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc(tmem_base, 256);
    }
}

// ======================================================================================================================
// xw = x W^T (+ logits) for the projected-feature path, A from a CACHED fp16-pair image of x
// ======================================================================================================================
// The projection of project_tc.cu stages x through registers (hi/lo split by four producer warps), which is what bounds it
// (ncu: 2.4 TB/s, tensor pipe 49 %).  For the first layer x is static across training steps, so its split image is built
// once (gnnfd_project_image_build, like the CSR) and every step's GEMM is fed by the copy engine alone.  Each ROW carries
// its own power-of-two scale (rows of very different magnitude keep 22 bits each); it is undone in the epilogue.
// Per 128-row tile: A = NKBX k-blocks (96 KB for K = 166) resident in shared memory; the W image streams through a
// 3-stage ring in (n-tile of 128 columns, k-block) order; accumulators: 2 x 128 TMEM columns (epilogue of n-tile t
// overlaps the MMAs of t+1).  Epilogue as in project_tc_ws.cuh: thread = row, per-head logit dots from the TMEM tile,
// coalesced stores through shared memory.
constexpr int P1_BN = 128;                          // columns per n-tile
constexpr int P1_NT_PROJ = (H * C) / P1_BN;         // 4
constexpr int P1_BSTAGES = 2;
constexpr uint32_t P1_B = 2 * P1_BN * 128;          // 32 KB: hi + lo [128 rows x 128 B]
constexpr int P1_MAX_KB = 3;                        // K <= 192
constexpr int P1_EPI_WARPS = 8;                     // two per TMEM lane quadrant: each takes 64 of the 128 columns (= one head)
constexpr int P1_THREADS = 64 + 32 * P1_EPI_WARPS;
constexpr size_t P1_SMEM = size_t(P1_MAX_KB) * KBLOCK + size_t(P1_BSTAGES) * P1_B + P1_EPI_WARPS * 32 * G1_STG_LD * 4 + 1024;

// LOGITS: the projection (n_nt = 4 n-tiles of 128 = the 8 heads; per-head logit dots).  !LOGITS: plain C = A B^T with n_nt
// n-tiles, the first n_valid columns stored (n_valid % 32 == 0) -- used for Gd = dO W_r^T (K = 64, 1344 columns).
template <bool LOGITS>
__global__ void __launch_bounds__(P1_THREADS, 1)
in_proj_gemm(const uint8_t* __restrict__ ximg, const float* __restrict__ row_scale, const uint8_t* __restrict__ wimg,
             const float* __restrict__ scal, int64_t n, int NKBX, int n_nt, int ld_out, int n_valid, float out_scale,
             const float* __restrict__ att_src, const float* __restrict__ att_dst, float* __restrict__ xw,
             float* __restrict__ a_src, float* __restrict__ a_dst)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;                                         // [P1_MAX_KB][KBLOCK]
    uint8_t* sB = smem + size_t(P1_MAX_KB) * KBLOCK;            // [P1_BSTAGES][P1_B]
    __shared__ uint64_t a_full, a_empty, b_full[P1_BSTAGES], b_empty[P1_BSTAGES], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    if (tid == 0) {
        st_mbar_init(&a_full, 1);
        st_mbar_init(&a_empty, 1);
        for (int s = 0; s < P1_BSTAGES; ++s) { st_mbar_init(&b_full[s], 1); st_mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { st_mbar_init(&acc_full[s], 1); st_mbar_init(&acc_empty[s], P1_EPI_WARPS); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const int P1_NT = n_nt;

    if (warp == 0) {
        // ---------------- producer --------------------------------------------------------------------------------
        int64_t j = 0, bstep = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
            if (j > 0) st_mbar_wait(&a_empty, uint32_t((j - 1) & 1));
            if (elect_one()) {
                st_mbar_expect_tx(&a_full, uint32_t(NKBX) * KBLOCK);
                st_bulk_g2s(sA, ximg + size_t(t) * NKBX * KBLOCK, uint32_t(NKBX) * KBLOCK, &a_full);
            }
            __syncwarp();
            for (int nt = 0; nt < P1_NT; ++nt)
                for (int kb = 0; kb < NKBX; ++kb, ++bstep) {
                    const int s = int(bstep % P1_BSTAGES);
                    const int64_t u = bstep / P1_BSTAGES;
                    if (u > 0) st_mbar_wait(&b_empty[s], uint32_t((u - 1) & 1));
                    if (elect_one()) {
                        st_mbar_expect_tx(&b_full[s], P1_B);
                        st_bulk_g2s(sB + size_t(s) * P1_B, wimg + (size_t(nt) * NKBX + kb) * P1_B, P1_B, &b_full[s]);
                    }
                    __syncwarp();
                }
        }
    } else if (warp == 1) {
        // ---------------- MMA issue --------------------------------------------------------------------------------
        constexpr uint32_t IDESC = make_idesc_f16(128, P1_BN, 0, 0);
        int64_t j = 0, bstep = 0, astep = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
            st_mbar_wait(&a_full, uint32_t(j & 1));
            for (int nt = 0; nt < P1_NT; ++nt, ++astep) {
                const int buf = int(astep & 1);
                if ((astep >> 1) > 0) st_mbar_wait(&acc_empty[buf], uint32_t(((astep >> 1) - 1) & 1));
                tc_fence_after();
                const uint32_t d = tmem_base + uint32_t(buf * P1_BN);
                for (int kb = 0; kb < NKBX; ++kb, ++bstep) {
                    const int s = int(bstep % P1_BSTAGES);
                    st_mbar_wait(&b_full[s], uint32_t((bstep / P1_BSTAGES) & 1));
                    tc_fence_after();
                    const uint32_t a_hi = st_smem_u32(sA + size_t(kb) * KBLOCK), a_lo = a_hi + PLANE;
                    const uint32_t b_hi = st_smem_u32(sB + size_t(s) * P1_B), b_lo = b_hi + P1_BN * 128;
                    if (elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint32_t ko = ks * 32;
                            const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                            const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                            umma_f16(d, dah, dbh, IDESC, (kb | ks) ? 1u : 0u);
                            umma_f16(d, dah, dbl, IDESC, 1u);
                            umma_f16(d, dal, dbh, IDESC, 1u);
                        }
                        umma_commit(&b_empty[s]);
                        if (kb == NKBX - 1) {
                            umma_commit(&acc_full[buf]);
                            if (nt == P1_NT - 1) umma_commit(&a_empty);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ---------------- epilogue: warps 2..9 -> TMEM lane quadrant warp & 3, column half (warp - 2) >> 2 ------------------
        const int quad = warp & 3, half = (warp - 2) >> 2;
        float* stg = reinterpret_cast<float*>(smem + size_t(P1_MAX_KB) * KBLOCK + size_t(P1_BSTAGES) * P1_B) + (warp - 2) * (32 * G1_STG_LD);
        const float inv_w = out_scale / scal[1];
        int64_t astep = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const int64_t m0 = t * TILE + quad * 32;
            const int64_t row = m0 + lane;
            const float inv = row < n ? inv_w / row_scale[row] : 0.f;
            for (int nt = 0; nt < P1_NT; ++nt, ++astep) {
                const int buf = int(astep & 1);
                st_mbar_wait(&acc_full[buf], uint32_t((astep >> 1) & 1));
                tc_fence_after();
                float ps = 0.f, pd = 0.f;
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    const int ch = 2 * half + cc;
                    const int col0 = nt * P1_BN + ch * 32;
                    if (col0 >= n_valid) break;
                    uint32_t v[32];
                    tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(buf * P1_BN + ch * 32), v);
#pragma unroll
                    for (int c = 0; c < 32; c += 4) {
                        const float f0 = __uint_as_float(v[c]) * inv, f1 = __uint_as_float(v[c + 1]) * inv;
                        const float f2 = __uint_as_float(v[c + 2]) * inv, f3 = __uint_as_float(v[c + 3]) * inv;
                        v[c] = __float_as_uint(f0); v[c + 1] = __float_as_uint(f1); v[c + 2] = __float_as_uint(f2); v[c + 3] = __float_as_uint(f3);
                        if (LOGITS) {
                            const float4 as4 = __ldg(reinterpret_cast<const float4*>(att_src + col0 + c));
                            const float4 ad4 = __ldg(reinterpret_cast<const float4*>(att_dst + col0 + c));
                            ps = fmaf(f0, as4.x, ps); pd = fmaf(f0, ad4.x, pd);
                            ps = fmaf(f1, as4.y, ps); pd = fmaf(f1, ad4.y, pd);
                            ps = fmaf(f2, as4.z, ps); pd = fmaf(f2, ad4.z, pd);
                            ps = fmaf(f3, as4.w, ps); pd = fmaf(f3, ad4.w, pd);
                        }
                    }
                    if (LOGITS && cc == 1 && row < n) {             // this warp's two chunks are one 64-wide head
                        const int hh = col0 / 64;
                        a_src[row * H + hh] = ps;
                        a_dst[row * H + hh] = pd;
                    }
                    __syncwarp();
#pragma unroll
                    for (int c = 0; c < 32; c += 4)
                        *reinterpret_cast<float4*>(stg + lane * G1_STG_LD + c) =
                            make_float4(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), __uint_as_float(v[c + 2]), __uint_as_float(v[c + 3]));
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int r = 4 * i + (lane >> 3), cq = (lane & 7) * 4;
                        const int64_t gm = m0 + r;
                        if (gm < n)
                            *reinterpret_cast<float4*>(xw + gm * ld_out + col0 + cq) = *reinterpret_cast<const float4*>(stg + r * G1_STG_LD + cq);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc(tmem_base, 256);
    }
}

// x [N,K] -> fp16-pair image (NKBX k-blocks of 64 features per 128-row tile) with a per-row power-of-two scale; warp = row
__global__ void __launch_bounds__(256)
in_ximg_kernel(const float* __restrict__ x, int64_t ldx, int64_t N, int K, int NKBX, uint8_t* __restrict__ ximg,
               float* __restrict__ row_scale)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t n = int64_t(blockIdx.x) * 8 + warp; n < N; n += int64_t(gridDim.x) * 8) {
        const float* row = x + n * ldx;
        float v[P1_MAX_KB][2];
        float mx = 0.f;
#pragma unroll
        for (int kb = 0; kb < P1_MAX_KB; ++kb) {
            const int k = kb * 64 + 2 * lane;
            v[kb][0] = (kb < NKBX && k < K) ? row[k] : 0.f;
            v[kb][1] = (kb < NKBX && k + 1 < K) ? row[k + 1] : 0.f;
            mx = fmaxf(mx, fmaxf(fabsf(v[kb][0]), fabsf(v[kb][1])));
        }
        mx = warp_max(mx);
        const float sc = pow2_scale(mx);
        if (lane == 0) row_scale[n] = sc;
        const uint32_t rr = uint32_t(n) & (TILE - 1);
        uint8_t* base = ximg + size_t(n >> 7) * size_t(NKBX) * KBLOCK + plane_off(int(rr), 2 * lane);
#pragma unroll
        for (int kb = 0; kb < P1_MAX_KB; ++kb)
            if (kb < NKBX) {
                __half2 hi, lo;
                split_h2(v[kb][0] * sc, v[kb][1] * sc, hi, lo);
                *reinterpret_cast<__half2*>(base + size_t(kb) * KBLOCK) = hi;
                *reinterpret_cast<__half2*>(base + size_t(kb) * KBLOCK + PLANE) = lo;
            }
    }
}
// W [512, K] -> B images in (n-tile of 128 output columns, k-block) order: [hi 128 x 128 B | lo], scaled by sw; also scal[1] = sw
__global__ void in_wproj_image_kernel(const float* __restrict__ W, int K, int NKBX, float* __restrict__ scal, uint8_t* __restrict__ img)
{
    __shared__ float red[32];
    __shared__ float sw_s;
    float m = 0.f;
    for (int i = threadIdx.x; i < H * C * K; i += blockDim.x) m = fmaxf(m, fabsf(W[i]));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        m = warp_max(m);
        if (threadIdx.x == 0) { sw_s = pow2_scale(m); if (blockIdx.x == 0) scal[1] = sw_s; }
    }
    __syncthreads();
    const float sw = sw_s;
    const int nt = blockIdx.x / NKBX, kb = blockIdx.x % NKBX;
    uint8_t* dst = img + size_t(blockIdx.x) * P1_B;
    for (int idx = threadIdx.x; idx < P1_BN * 64; idx += blockDim.x) {
        const int r = idx >> 6, e = idx & 63, k = kb * 64 + e;
        const float v = k < K ? W[int64_t(nt * P1_BN + r) * K + k] * sw : 0.f;
        const __half hi = __float2half_rn(v);
        const __half lo = __float2half_rn(v - __half2float(hi));
        const uint32_t off = plane_off(r, e);
        *reinterpret_cast<__half*>(dst + off) = hi;
        *reinterpret_cast<__half*>(dst + P1_BN * 128 + off) = lo;
    }
}

// W image of Gd = dO W_r^T: n-tile nt = features [128 nt, 128 nt + 128), rows = feature f = h*KP + k, 64 columns = c;
// element = W[(h*C + c)*K + k] * sw  (fp16 hi | lo, K-major in c)
__global__ void in_wgd_image_kernel(const float* __restrict__ W, int K, int KP, int F, const float* __restrict__ scal,
                                    uint8_t* __restrict__ img)
{
    const int nt = blockIdx.x;
    const float sw = scal[1];
    uint8_t* dst = img + size_t(nt) * P1_B;
    for (int idx = threadIdx.x; idx < P1_BN * 64; idx += blockDim.x) {
        const int r = idx >> 6, c = idx & 63, f = nt * P1_BN + r;
        float v = 0.f;
        if (f < F) {
            const int h = f / KP, k = f - h * KP;
            if (k < K) v = W[int64_t(h * C + c) * K + k] * sw;
        }
        const __half hi = __float2half_rn(v);
        const __half lo = __float2half_rn(v - __half2float(hi));
        const uint32_t off = plane_off(r, c);
        *reinterpret_cast<__half*>(dst + off) = hi;
        *reinterpret_cast<__half*>(dst + P1_BN * 128 + off) = lo;
    }
}
}  // namespace in
int in_build_gd_image(const float* W, int K, void* prep, cudaStream_t st)
{
    const in::Dims d(K);
    char* p = reinterpret_cast<char*>(prep);
    in::in_wgd_image_kernel<<<(d.F + 127) / 128, 256, 0, st>>>(W, d.K, d.KP, d.F, reinterpret_cast<const float*>(p),
                                                              reinterpret_cast<uint8_t*>(p + in::prep_off_wgd(d)));
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}
namespace in {

// ======================================================================================================================
// dWr partials:  P[slab][f][c] = sum_{i in slab} Z[i,f] * dO[i,c]   (both operands MN-major, reduction over nodes)
// ======================================================================================================================
// A CTA owns a slab of node tiles and HALF of the feature M-tiles (TMEM holds 6 accumulators of 128 x 64).  Per node
// tile the four producer warps split dO (fp32 -> scaled fp16 hi/lo, swizzled) once; the bulk-copy warp streams the Z
// k-block pairs (64 KB: one M = 128 tile of features); the issuer runs 8 k-steps x 3 MMAs per M-tile.  Every FLUSH
// node tiles the accumulators are drained into the CTA's private fp32 partial with RED.ADD (L2-resident), which bounds
// the round-toward-zero accumulation chain; partials are summed in slab order afterwards (deterministic).
constexpr int G3_THREADS = 192;
constexpr uint32_t G3_A = 2 * KBLOCK;              // 64 KB: two consecutive k-blocks (128 features), hi + lo each
constexpr uint32_t G3_B = 2 * PLANE;               // 32 KB: dO tile, hi + lo planes
constexpr int G3_FLUSH = 4;   // node tiles per accumulation chain (chain = G3_FLUSH x 8 k-steps x 3 MMAs)
constexpr int G3_STG_LD = 33;
constexpr size_t G3_SMEM = 2 * size_t(G3_A) + 2 * size_t(G3_B) + 4 * 32 * G3_STG_LD * 4 + 1024;

__global__ void __launch_bounds__(G3_THREADS, 1)
in_dw_gemm(const uint8_t* __restrict__ zimg, const float* __restrict__ d_out, const float* __restrict__ dmax, int64_t n,
           int NKB, int F, int64_t tiles_per_slab, float* __restrict__ P, int64_t p_slab_stride)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;                              // [2][G3_A]
    uint8_t* sB = smem + 2 * size_t(G3_A);           // [2][G3_B]
    __shared__ uint64_t a_full[2], a_empty[2], b_full[2], b_empty[2], acc_full, acc_empty;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int slab = blockIdx.x >> 1, half = blockIdx.x & 1;
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    const int64_t t0 = int64_t(slab) * tiles_per_slab;
    const int64_t t1 = (t0 + tiles_per_slab < n_tiles) ? t0 + tiles_per_slab : n_tiles;
    const int nt = t1 > t0 ? int(t1 - t0) : 0;
    const int MT = (NKB + 1) / 2, MT0 = (MT + 1) / 2;
    const int m_base = half ? MT0 : 0;
    const int my_mt = half ? MT - MT0 : MT0;

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            st_mbar_init(&a_full[s], 1);
            st_mbar_init(&a_empty[s], 1);
            st_mbar_init(&b_full[s], 4);
            st_mbar_init(&b_empty[s], 1);
        }
        st_mbar_init(&acc_full, 1);
        st_mbar_init(&acc_empty, 4);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (my_mt > 0 && nt > 0) {
        if (warp == 0) {
            // ---------------- A producer: one 64 KB copy (two k-blocks of the image) per (node tile, M-tile) -------------
            int64_t step = 0;
            for (int i = 0; i < nt; ++i) {
                for (int mm = 0; mm < my_mt; ++mm, ++step) {
                    const int s = int(step & 1);
                    if (step >= 2) st_mbar_wait(&a_empty[s], uint32_t(((step >> 1) - 1) & 1));
                    const int kb0 = 2 * (m_base + mm);
                    const uint32_t bytes = (kb0 + 1 < NKB) ? G3_A : uint32_t(KBLOCK);   // odd NKB: the last pair is half
                    if (elect_one()) {
                        st_mbar_expect_tx(&a_full[s], bytes);
                        st_bulk_g2s(sA + size_t(s) * G3_A, zimg + (size_t(t0 + i) * NKB + kb0) * KBLOCK, bytes, &a_full[s]);
                    }
                    __syncwarp();
                }
            }
        } else if (warp == 1) {
            // ---------------- MMA issue ------------------------------------------------------------------------------
            constexpr uint32_t IDESC = make_idesc_f16(128, C, 1, 1);
            int64_t step = 0;
            for (int i = 0; i < nt; ++i) {
                const int bb = i & 1;
                st_mbar_wait(&b_full[bb], uint32_t((i >> 1) & 1));
                if (i > 0 && i % G3_FLUSH == 0) st_mbar_wait(&acc_empty, uint32_t(((i / G3_FLUSH) - 1) & 1));
                tc_fence_after();
                const uint32_t b_hi = st_smem_u32(sB + size_t(bb) * G3_B), b_lo = b_hi + PLANE;
                const bool restart = (i % G3_FLUSH) == 0;
                for (int mm = 0; mm < my_mt; ++mm, ++step) {
                    const int s = int(step & 1);
                    st_mbar_wait(&a_full[s], uint32_t((step >> 1) & 1));
                    tc_fence_after();
                    // stage layout: [k-block 2m: hi | lo][k-block 2m+1: hi | lo]; the two 64-feature atoms of the M = 128
                    // operand are KBLOCK bytes apart (LBO), consecutive 8-node groups 1024 bytes (SBO)
                    const uint32_t a_hi = st_smem_u32(sA + size_t(s) * G3_A), a_lo = a_hi + PLANE;
                    const uint32_t d = tmem_base + uint32_t(mm * 64);
                    if (elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks) {         // 16 nodes per k-step = two 8-node groups
                            const uint32_t ko = ks * 2048;
                            const uint64_t dah = make_desc(a_hi + ko, KBLOCK, 1024), dal = make_desc(a_lo + ko, KBLOCK, 1024);
                            const uint64_t dbh = make_desc(b_hi + ko, PLANE, 1024), dbl = make_desc(b_lo + ko, PLANE, 1024);
                            umma_f16(d, dah, dbh, IDESC, (restart && ks == 0) ? 0u : 1u);
                            umma_f16(d, dah, dbl, IDESC, 1u);
                            umma_f16(d, dal, dbh, IDESC, 1u);
                        }
                        umma_commit(&a_empty[s]);
                        if (mm == my_mt - 1) {
                            umma_commit(&b_empty[bb]);
                            if ((i + 1) % G3_FLUSH == 0 || i == nt - 1) umma_commit(&acc_full);
                        }
                    }
                    __syncwarp();
                }
            }
        } else {
            // ---------------- dO producers (warps 2..5, 32 nodes each) + accumulator flush (TMEM quadrants 2,3,0,1) ------
            const int w = warp - 2, quad = warp & 3;
            const float sd = pow2_scale(*dmax);
            float* stg = reinterpret_cast<float*>(smem + 2 * size_t(G3_A) + 2 * size_t(G3_B)) + w * (32 * G3_STG_LD);
            float* Ps = P + int64_t(slab) * p_slab_stride;
            int flushes = 0;
            for (int i = 0; i < nt; ++i) {
                const int bb = i & 1;
                if (i >= 2) st_mbar_wait(&b_empty[bb], uint32_t(((i >> 1) - 1) & 1));
                uint8_t* b_hi = sB + size_t(bb) * G3_B;
                const int64_t node0 = (t0 + i) * TILE + w * 32;
                // lane owns channels 2*lane, 2*lane+1 of every node row: coalesced 256-byte row reads
                float2 v[32];
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    const int64_t node = node0 + r;
                    v[r] = (node < n) ? __ldg(reinterpret_cast<const float2*>(d_out + node * C) + lane) : make_float2(0.f, 0.f);
                }
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    __half2 hi, lo;
                    split_h2(v[r].x * sd, v[r].y * sd, hi, lo);
                    const uint32_t off = plane_off(w * 32 + r, 2 * lane);
                    *reinterpret_cast<__half2*>(b_hi + off) = hi;
                    *reinterpret_cast<__half2*>(b_hi + PLANE + off) = lo;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&b_full[bb]);
                if ((i + 1) % G3_FLUSH == 0 || i == nt - 1) {
                    st_mbar_wait(&acc_full, uint32_t(flushes & 1));
                    tc_fence_after();
                    ++flushes;
                    for (int mm = 0; mm < my_mt; ++mm) {
                        const int f0 = (m_base + mm) * 128 + quad * 32;          // this warp's 32 feature rows
#pragma unroll 1
                        for (int ch = 0; ch < C / 32; ++ch) {
                            uint32_t acc[32];
                            tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(mm * 64 + ch * 32), acc);
                            __syncwarp();
#pragma unroll
                            for (int c = 0; c < 32; ++c) stg[lane * G3_STG_LD + c] = __uint_as_float(acc[c]);
                            __syncwarp();
                            // fire-and-forget fp32 reductions into this CTA's private partial: 128-byte coalesced
#pragma unroll 8
                            for (int r = 0; r < 32; ++r)
                                if (f0 + r < F) atomicAdd(Ps + int64_t(f0 + r) * C + ch * 32 + lane, stg[r * G3_STG_LD + lane]);
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc(tmem_base, 512);
    }
}

// dW[o = h*C + c, k] = inv * sum_slab P[slab][f = h*KP + k][c] + att_src[o] * Gm[h][k] + att_dst[o] * Gm[H + h][k]
__global__ void in_dw_finalize(const float* __restrict__ P, int n_slabs, int64_t p_slab_stride, const float* __restrict__ scal,
                               const float* __restrict__ dmax, const float* __restrict__ Gm, const float* __restrict__ att_src,
                               const float* __restrict__ att_dst, int K, int KP, float* __restrict__ dW)
{
    const float inv = 1.f / (scal[0] * pow2_scale(*dmax) * float(H));
    const int total = H * C * K;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        // c fastest across threads: the partials are read as 256-byte runs
        const int c = idx % C, hk = idx / C, k = hk % K, h = hk / K;
        const int64_t pf = int64_t(h * KP + k) * C + c;
        float s = 0.f;
        for (int sl = 0; sl < n_slabs; ++sl) s += P[int64_t(sl) * p_slab_stride + pf];
        const int o = h * C + c;
        dW[int64_t(o) * K + k] = s * inv + att_src[o] * Gm[h * K + k] + att_dst[o] * Gm[(H + h) * K + k];
    }
}

__global__ void in_absmax_kernel(const float* __restrict__ a, int64_t n, unsigned* __restrict__ out_bits)
{
    float m = 0.f;
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
        m = fmaxf(m, fabsf(a[i]));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out_bits, __float_as_uint(m));
}

// da_src[j,h] = sum of dz over the out-edges of source j (dz rows are in source-major order): thread per (j, h)
__global__ void in_dasrc_kernel(const int32_t* __restrict__ colptr, const float* __restrict__ dz, int64_t n_src,
                                float* __restrict__ da_src)
{
    const int64_t idx = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
    const int64_t j = idx / H;
    const int h = int(idx % H);
    if (j >= n_src) return;
    const int beg = colptr[j], end = colptr[j + 1];
    float s0 = 0.f, s1 = 0.f;
    int p = beg;
    for (; p + 1 < end; p += 2) {
        s0 += dz[int64_t(p) * H + h];
        s1 += dz[int64_t(p + 1) * H + h];
    }
    if (p < end) s0 += dz[int64_t(p) * H + h];
    da_src[j * H + h] = s0 + s1;
}

static int dw_slabs(int64_t n_tiles)
{
    int64_t s = sm_count() / 2;
    if (s > n_tiles) s = n_tiles;
    if (s < 1) s = 1;
    return (int)s;
}
static size_t dw_partial_floats(const Dims& d) { return size_t((d.NKB + 1) / 2) * 128 * C; }

}  // namespace in
}  // namespace gnnfd

using namespace gnnfd;
using namespace gnnfd::in;

template <int PM>
static int in_out_launch(const void* zimg, int64_t n, int64_t K, const void* prep, const OutEpi& ep, float* out,
                         const PeerRows& peers, cudaStream_t st)
{
    const Dims d((int)K);
    const char* p = reinterpret_cast<const char*>(prep);
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    const unsigned grid = (unsigned)(n_tiles < sm_count() ? n_tiles : sm_count());
    GNNFD_CUDA(cudaFuncSetAttribute(in_out_gemm<PM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G1_SMEM));
    in_out_gemm<PM><<<grid, G1_THREADS, G1_SMEM, st>>>(reinterpret_cast<const uint8_t*>(zimg),
                                                       reinterpret_cast<const uint8_t*>(p + prep_off_wout(d)),
                                                       reinterpret_cast<const float*>(p), n, d.NKB, ep, out, peers);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

extern "C" {

/* out [n, C] = act((Z W_r / H + bias) * post_scale + post_shift) + residual   (cf. gnnfd_gat_fwd_fused) */
int gnnfd_in_out(const void* zimg, int64_t n, int64_t K, const void* prep, const float* bias, int act,
                 const float* post_scale, const float* post_shift, const float* residual, float* out,
                 gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && n >= 0, GNNFD_ERR_ARG, "in_out: bad shape");
    if (n == 0) return GNNFD_OK;
    GNNFD_REQUIRE(zimg && prep && out, GNNFD_ERR_ARG, "in_out: NULL tensor");
    GNNFD_REQUIRE((post_scale == nullptr) == (post_shift == nullptr), GNNFD_ERR_ARG,
                  "in_out: post_scale and post_shift must be given together");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(zimg) & 1023) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, GNNFD_ERR_ARG,
                  "in_out: zimg must be 1024-byte and out 16-byte aligned");
    const OutEpi ep{bias, post_scale, post_shift, residual, act};
    return in_out_launch<0>(zimg, n, K, prep, ep, out, PeerRows{}, (cudaStream_t)stream);
}

/* gnnfd_in_out fused with the all-gather of the output rows: every finished 16-byte piece of row r also goes to row
 * (row_offset + r) of h_all [n_pos, C] on every rank (one multimem.st, or one store per peer).  out (own rows) may be NULL. */
int gnnfd_in_out_bcast(const void* zimg, int64_t n, int64_t K, const void* prep, const float* bias, int act,
                       const float* post_scale, const float* post_shift, const float* residual,
                       const gnnfd_peers_t* h_all, int64_t row_offset, int use_multicast, float* out,
                       gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && n >= 0, GNNFD_ERR_ARG, "in_out_bcast: bad shape");
    PeerRows peers;
    const int rc = peer_rows_from(h_all, row_offset, use_multicast, "in_out_bcast", peers);
    if (rc) return rc;
    if (n == 0) return GNNFD_OK;
    GNNFD_REQUIRE(zimg && prep, GNNFD_ERR_ARG, "in_out_bcast: NULL tensor");
    GNNFD_REQUIRE((post_scale == nullptr) == (post_shift == nullptr), GNNFD_ERR_ARG,
                  "in_out_bcast: post_scale and post_shift must be given together");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(zimg) & 1023) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, GNNFD_ERR_ARG,
                  "in_out_bcast: zimg must be 1024-byte and out 16-byte aligned");
    GNNFD_REQUIRE(!use_multicast || (reinterpret_cast<uintptr_t>(h_all->multicast) & 15) == 0, GNNFD_ERR_ARG,
                  "in_out_bcast: the multicast address must be 16-byte aligned");
    const OutEpi ep{bias, post_scale, post_shift, residual, act};
    cudaStream_t st = (cudaStream_t)stream;
    return use_multicast ? in_out_launch<2>(zimg, n, K, prep, ep, out, peers, st) : in_out_launch<1>(zimg, n, K, prep, ep, out, peers, st);
}

/* gd [n, F] = d_out [n, C] @ W_r^T / H  (F = gnnfd_in_sizes' gd_ld): the per-destination vectors whose dot product with
 * x[j] is d_alpha.  Row-range agnostic: call it on a block of rows to bound the size of gd.  d_out is first split into its
 * fp16-pair image (per-row scale) so that the GEMM is fed by the copy engine; ws: gnnfd_in_bwd_gd_workspace_bytes(n). */
int gnnfd_in_bwd_gd_workspace_bytes(int64_t n, size_t* bytes)
{
    GNNFD_REQUIRE(bytes && n >= 0, GNNFD_ERR_ARG, "in_bwd_gd_workspace_bytes: bad argument");
    *bytes = size_t((n + TILE - 1) / TILE) * KBLOCK + carve_bytes(size_t(n > 0 ? n : 1), 4) + 2048;
    return GNNFD_OK;
}
int gnnfd_in_bwd_gd(const float* d_out, int64_t n, int64_t K, const void* prep, float* gd, void* ws, size_t ws_bytes,
                    gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && n >= 0, GNNFD_ERR_ARG, "in_bwd_gd: bad shape");
    if (n == 0) return GNNFD_OK;
    size_t need = 0;
    gnnfd_in_bwd_gd_workspace_bytes(n, &need);
    GNNFD_REQUIRE(d_out && prep && gd && ws && ws_bytes >= need && (reinterpret_cast<uintptr_t>(ws) & 1023) == 0, GNNFD_ERR_WORKSPACE,
                  "in_bwd_gd: NULL tensor, or workspace too small / not 1024-byte aligned");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(gd) & 15) == 0, GNNFD_ERR_ARG, "in_bwd_gd: gd must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const Dims d((int)K);
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    uint8_t* dimg = reinterpret_cast<uint8_t*>(ws);
    float* row_scale = reinterpret_cast<float*>(dimg + size_t(n_tiles) * KBLOCK);
    int64_t blocks = (n + 7) / 8;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    in_ximg_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_out, C, n, C, 1, dimg, row_scale);
    const char* p = reinterpret_cast<const char*>(prep);
    const unsigned grid = (unsigned)(n_tiles < sm_count() ? n_tiles : sm_count());
    GNNFD_CUDA(cudaFuncSetAttribute(in_proj_gemm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1_SMEM));
    in_proj_gemm<false><<<grid, P1_THREADS, P1_SMEM, st>>>(dimg, row_scale, reinterpret_cast<const uint8_t*>(p + prep_off_wgd(d)),
                                                           reinterpret_cast<const float*>(p), n, 1, (d.F + 127) / 128, d.F, d.F,
                                                           1.f / float(H), nullptr, nullptr, gd, nullptr, nullptr);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* da_src [n_src, H] = per-source sums of dz (source-major order, as gnnfd_in_bwd_edges writes it); needs the CSC twin. */
int gnnfd_in_bwd_dasrc(const gnnfd_graph_t* g, const float* dz, float* da_src, gnnfd_stream_t stream)
{
    int rc = check_graph(g, true, "in_bwd_dasrc");
    if (rc) return rc;
    if (g->n_src == 0) return GNNFD_OK;
    GNNFD_REQUIRE(da_src && (g->n_edges == 0 || dz), GNNFD_ERR_ARG, "in_bwd_dasrc: NULL tensor");
    const int64_t total = g->n_src * H;
    in_dasrc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g->colptr, dz, g->n_src, da_src);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int gnnfd_in_bwd_params_workspace_bytes(int64_t n, int64_t K, size_t* bytes)
{
    GNNFD_REQUIRE(bytes && K >= 1 && K <= MAX_K && n >= 0, GNNFD_ERR_ARG, "in_bwd_params_workspace_bytes: bad argument");
    const Dims d((int)K);
    const int S = dw_slabs((n + TILE - 1) / TILE);
    *bytes = in_param_ws_bytes(n, K) + carve_bytes(size_t(S) * dw_partial_floats(d), 4) + carve_bytes(size_t(2) * H * K, 4) + 1024;
    return GNNFD_OK;
}

/* Parameter gradients of the layer from the saved image and the logit gradients of THIS rank's n rows:
 *   dW [H*C, K], datt_src / datt_dst [H*C], dbias [C]   (x, da_src, da_dst, d_out: rows [0, n)).
 * phase bit 0: the tensor-core reduction dO^T Z into ws (needs no logit gradients -- across GPUs it runs while da_src is still
 * being exchanged); bit 1: the node reductions with da_src / da_dst and the final dW (same ws); 3 = both. */
int gnnfd_in_bwd_params(const void* zimg, const float* d_out, const float* x, int64_t ldx, int64_t n, int64_t K,
                        const float* W, const float* att_src, const float* att_dst, const float* da_src,
                        const float* da_dst, const void* prep, float* dW, float* datt_src, float* datt_dst,
                        float* dbias, void* ws, size_t ws_bytes, int phase, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && n >= 0 && ldx >= K, GNNFD_ERR_ARG, "in_bwd_params: bad shape");
    GNNFD_REQUIRE(W && att_src && att_dst && prep && dW && datt_src && datt_dst && dbias, GNNFD_ERR_ARG, "in_bwd_params: NULL argument");
    GNNFD_REQUIRE(phase >= 1 && phase <= 3, GNNFD_ERR_ARG, "in_bwd_params: phase must be 1, 2 or 3");
    GNNFD_REQUIRE(n == 0 || (zimg && d_out && x), GNNFD_ERR_ARG, "in_bwd_params: NULL tensor");
    GNNFD_REQUIRE(n == 0 || !(phase & 2) || (da_src && da_dst), GNNFD_ERR_ARG, "in_bwd_params: NULL logit gradients");
    size_t need = 0;
    gnnfd_in_bwd_params_workspace_bytes(n, K, &need);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "in_bwd_params: workspace %zu < %zu", ws_bytes, need);
    cudaStream_t st = (cudaStream_t)stream;
    const Dims d((int)K);
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    const int S = dw_slabs(n_tiles);
    char* p = reinterpret_cast<char*>(ws);
    const size_t simt_bytes = in_param_ws_bytes(n, K);
    char* q = p + ((simt_bytes + 255) & ~size_t(255));
    float* P = carve<float>(q, size_t(S) * dw_partial_floats(d));
    float* Gm = carve<float>(q, size_t(2) * H * K);
    unsigned* dmax = reinterpret_cast<unsigned*>(carve<float>(q, 16));
    const int64_t pstride = (int64_t)dw_partial_floats(d);
    if (phase & 1) {
        // the tensor-core part: slab partials of dO^T Z (needs neither da_src nor da_dst)
        GNNFD_CUDA(cudaMemsetAsync(P, 0, size_t(S) * pstride * sizeof(float), st));
        GNNFD_CUDA(cudaMemsetAsync(dmax, 0, 64, st));
        if (n > 0) {
            int64_t blocks = (n * C + 255) / 256;
            if (blocks > int64_t(sm_count()) * 8) blocks = int64_t(sm_count()) * 8;
            in_absmax_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_out, n * C, dmax);
            const int64_t tps = (n_tiles + S - 1) / S;
            GNNFD_CUDA(cudaFuncSetAttribute(in_dw_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G3_SMEM));
            in_dw_gemm<<<2 * S, G3_THREADS, G3_SMEM, st>>>(reinterpret_cast<const uint8_t*>(zimg), d_out,
                                                           reinterpret_cast<const float*>(dmax), n, d.NKB, d.F, tps, P, pstride);
            g_launches += 2;
        }
    }
    if (phase & 2) {
        // datt, dbias and G = [da_src | da_dst]^T x (node reductions over x, shared with the projected-feature path)
        int rc = in_param_grads_simt(x, ldx, W, da_src, da_dst, d_out, n, K, datt_src, datt_dst, dbias, Gm, p, simt_bytes, st);
        if (rc) return rc;
        in_dw_finalize<<<(H * C * d.K + 255) / 256, 256, 0, st>>>(P, S, pstride, reinterpret_cast<const float*>(prep),
                                                                 reinterpret_cast<const float*>(dmax), Gm, att_src, att_dst, d.K,
                                                                 d.KP, dW);
        g_launches += 1;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* Cached-image projection (projected-feature path, first layer): gnnfd_project_image_build splits x once into the fp16-pair
 * tensor-core image (+ one power-of-two scale per row); gnnfd_project_fwd_image then computes xw = x W^T and the per-head
 * logits exactly like gnnfd_project_fwd, fed by the copy engine alone.  H = 8, C = 64, K <= 192.
 * ximg: gnnfd_project_image_bytes, 1024-byte aligned; row_scale [N]; ws >= 512 KB + 1 KB, 1024-byte aligned. */
int gnnfd_project_image_bytes(int64_t N, int64_t K, size_t* ximg_bytes, size_t* ws_bytes)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && N >= 0, GNNFD_ERR_ARG, "project_image_bytes: K must be in [1,%d]", MAX_K);
    const int nkbx = int((K + 63) / 64);
    if (ximg_bytes) *ximg_bytes = size_t((N + TILE - 1) / TILE) * nkbx * KBLOCK + 1024;
    if (ws_bytes) *ws_bytes = size_t(P1_NT_PROJ) * nkbx * P1_B + 2048;
    return GNNFD_OK;
}
int gnnfd_project_image_build(const float* x, int64_t ldx, int64_t N, int64_t K, void* ximg, float* row_scale, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && ldx >= K && N >= 0, GNNFD_ERR_ARG, "project_image_build: bad shape");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(x && ximg && row_scale && (reinterpret_cast<uintptr_t>(ximg) & 1023) == 0, GNNFD_ERR_ARG,
                  "project_image_build: NULL tensor or ximg not 1024-byte aligned");
    const int nkbx = int((K + 63) / 64);
    int64_t blocks = (N + 7) / 8;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    in_ximg_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, N, (int)K, nkbx, reinterpret_cast<uint8_t*>(ximg), row_scale);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}
int gnnfd_project_fwd_image(const void* ximg, const float* row_scale, int64_t N, int64_t K, const float* W, const float* att_src,
                            const float* att_dst, float* xw, float* a_src, float* a_dst, void* ws, size_t ws_bytes,
                            gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(K >= 1 && K <= MAX_K && N >= 0 && W && att_src && att_dst, GNNFD_ERR_ARG, "project_fwd_image: bad argument");
    if (N == 0) return GNNFD_OK;
    size_t need = 0;
    gnnfd_project_image_bytes(N, K, nullptr, &need);
    GNNFD_REQUIRE(ximg && row_scale && xw && a_src && a_dst && ws && ws_bytes >= need && (reinterpret_cast<uintptr_t>(ws) & 1023) == 0,
                  GNNFD_ERR_WORKSPACE, "project_fwd_image: NULL tensor, or workspace too small / not 1024-byte aligned");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(xw) & 15) == 0, GNNFD_ERR_ARG, "project_fwd_image: xw must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int nkbx = int((K + 63) / 64);
    float* scal = reinterpret_cast<float*>(ws);
    uint8_t* wimg = reinterpret_cast<uint8_t*>(ws) + 1024;
    in_wproj_image_kernel<<<P1_NT_PROJ * nkbx, 512, 0, st>>>(W, (int)K, nkbx, scal, wimg);
    const int64_t n_tiles = (N + TILE - 1) / TILE;
    const unsigned grid = (unsigned)(n_tiles < sm_count() ? n_tiles : sm_count());
    GNNFD_CUDA(cudaFuncSetAttribute(in_proj_gemm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1_SMEM));
    in_proj_gemm<true><<<grid, P1_THREADS, P1_SMEM, st>>>(reinterpret_cast<const uint8_t*>(ximg), row_scale, wimg, scal, N, nkbx, P1_NT_PROJ,
                                                          H * C, H * C, 1.f, att_src, att_dst, xw, a_src, a_dst);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // extern "C"
