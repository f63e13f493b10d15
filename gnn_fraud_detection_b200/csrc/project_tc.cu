// (2) tensor-core projection: xw = x @ W^T on the 5th-gen tensor cores (tcgen05.mma, accumulators in
// TMEM), error-compensated 3xTF32 so the fp32 parity bar (1e-5) holds, with the per-head attention
// logits a_src/a_dst computed in the epilogue from the TMEM-resident tile.  Also the two projection
// backward GEMMs: dx = dxw @ W (transposed weight image) and dW = dxw^T @ x (split over node slabs,
// MN-major operands).
//
// Replaces lin_src(x) / (x*att).sum(-1) of GATConv.forward (reference call site src/models/gat.py:80)
// and their autograd mirror (src/train.py:142).
//
// This file holds the PTX wrappers, the weight-image builder, the slab reduction and the host launchers.
// The kernels:
//   forward  gemm_tc_ws2 (project_tc_ws2.cuh): persistent, warp-specialised, two CTAs of a cluster per
//            256 x 256 tile (cta_group::2), logits epilogue
//   dx       gemm_tc_ws (project_tc_ws.cuh): the same pipeline on one SM, plain fp32 store
//   dW       dw_tc2 (project_tc_dw2.cuh): one persistent CTA per SM and 256 output rows, fp32 partial per slab
// Data movement
//   * W (and W^T) are split once per call into tf32 hi/lo parts and laid out in global memory as ready-made
//     128B-swizzled shared-memory images, one 64 KB image per (column tile, k-block); a CTA fetches its part of
//     an image with cp.async.bulk (bulk async copy engine, mbarrier complete_tx) -- no tensor map needed.
//   * x rows have a 664-byte stride (K=166), not 16-byte aligned, so TMA cannot address them: producer warps read
//     coalesced 128-byte row segments, split them into hi/lo in registers and store them into the swizzled
//     K-major layout (conflict-free), then publish them to the async proxy with fence.proxy.async.
//   * one elected lane issues tcgen05.mma.kind::tf32 (K=8): per k-step three MMAs (hi*hi, lo*hi, hi*lo);
//     tcgen05.commit arrives on an mbarrier when they retire.
//   * epilogue: each warp reads its 32 TMEM lanes (tcgen05.ld 32x32b.x32), a thread owns a full output row so
//     the logit dot products need no shuffles; the tile is staged through shared memory and written with
//     coalesced stores.
#include "common.cuh"

#include <atomic>

namespace gnnfd {
extern std::atomic<long long> g_launches;

namespace tc {

constexpr int BM = 128;          // rows per CTA tile (UMMA M)
constexpr int BK = 32;           // tf32 elements per k-block = one 128-byte swizzle row
constexpr int UK = 8;            // tf32 UMMA K
constexpr uint32_t SPIN_LIMIT = 1u << 26;

// ---- PTX wrappers -----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (++spins > SPIN_LIMIT) __trap();   // never hang the GPU on a protocol bug
    }
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
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

// ---- descriptors ------------------------------------------------------------------------------------
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout type [61,64) (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = 2)
{
    uint64_t d = 0;
    d |= uint64_t((saddr & 0x3FFFF) >> 4);
    d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= uint64_t(1) << 46;
    d |= uint64_t(layout) << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2,
// a_major bit15, b_major bit16 (0 = K-major, 1 = MN-major), N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) |
           (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

// byte offset of element (row r, k-element kk in [0,32)) inside a K-major SWIZZLE_128B tile
__host__ __device__ __forceinline__ uint32_t kmajor_off(int r, int kk)
{
    return uint32_t(r >> 3) * 1024u + uint32_t(r & 7) * 128u + (uint32_t((kk >> 2) ^ (r & 7)) << 4) + uint32_t(kk & 3) * 4u;
}
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo)
{
    hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);   // what the tensor core keeps of an fp32 operand
    lo = v - hi;                                              // exact; its own low bits are dropped by the MMA
}

// ---- weight images -------------------------------------------------------------------------------------
// img[tile][kb][part][rows x 128 B swizzled], part 0 = hi, 1 = lo.  rows = rows_per_tile (<= 256).
// element(tile t, row r, k) = src[(t*rows + r) * s_row + k * s_k] for r < n_rows_total - t*rows, k < Kd; else 0.
__global__ void build_b_images(const float* __restrict__ src, int64_t s_row, int64_t s_k, int n_rows_total, int Kd,
                               int rows_per_tile, int n_kb, float* __restrict__ img)
{
    const int tile = blockIdx.z, kb = blockIdx.y;
    const size_t tile_elems = size_t(rows_per_tile) * BK;
    float* hi = img + ((size_t(tile) * n_kb + kb) * 2 + 0) * tile_elems;
    float* lo = img + ((size_t(tile) * n_kb + kb) * 2 + 1) * tile_elems;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < rows_per_tile * BK; idx += gridDim.x * blockDim.x) {
        const int r = idx / BK, kk = idx % BK;
        const int gr = tile * rows_per_tile + r, gk = kb * BK + kk;
        float v = 0.f;
        if (gr < n_rows_total && gk < Kd) v = src[int64_t(gr) * s_row + int64_t(gk) * s_k];
        float h, l;
        split_tf32(v, h, l);
        const uint32_t off = kmajor_off(r, kk) >> 2;
        hi[off] = h;
        lo[off] = l;
    }
}

__global__ void reduce_slabs(const float* __restrict__ P, int64_t n, int S, float* __restrict__ out)
{
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < S; ++k) s += P[int64_t(k) * n + i];
        out[i] = s;
    }
}

inline int kblocks(int64_t Kd) { return int((Kd + BK - 1) / BK); }

}  // namespace tc

}  // namespace gnnfd
#include "project_tc_ws.cuh"
#include "project_tc_ws2.cuh"
#include "project_tc_dw2.cuh"
namespace gnnfd {

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
static int g_tc_state = 0;   // 0 unknown, 1 usable, -1 not an sm_100 device
static bool tc_device_ok()
{
    if (g_tc_state == 0) {
        int dev = 0, major = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
        g_tc_state = (major == 10) ? 1 : -1;
    }
    return g_tc_state == 1;
}

bool tc_supported(int64_t N, int64_t K, int H, int C)
{
    (void)N;
    return tc_device_ok() && (C == 32 || C == 64 || C == 128) && (H * C) % 256 == 0 && K >= 1 && K <= 4096;
}

// images for the forward (W: D rows x K) + for dx (W^T: K rows x D, one tile of <= 256 rows)
size_t tc_ws_bytes(int64_t N, int64_t K, int H, int C)
{
    (void)N;
    const size_t D = size_t(H) * C;
    const size_t fwd = (D / 256) * tc::kblocks(K) * 2 * (256 * tc::BK) * sizeof(float);
    const size_t kt = size_t((K + 255) / 256);
    const size_t bwd = kt * tc::kblocks((int64_t)D) * 2 * (256 * tc::BK) * sizeof(float);
    const size_t dwp = (size_t(N / 2048 > 74 ? 74 : (N / 2048 < 1 ? 1 : N / 2048))) * D * size_t(K) * sizeof(float) + 2048;
    return fwd + bwd + dwp + 4096;
}

// the forward GEMM with the logits epilogue for heads of HC columns.  bf16 feature storage (2e-2 relative tolerance)
// takes one TF32 pass (FAST) instead of the compensated three.
template <int HC, bool BF16>
static int launch_fwd_tc(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst, int64_t N,
                         int64_t K, int H, int D, void* xw, float* a_src, float* a_dst, void* ws, cudaStream_t st)
{
    constexpr int BN = 256;
    const int n_kb = tc::kblocks(K), n_tiles = D / BN;
    float* img = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    float* xf = BF16 ? nullptr : reinterpret_cast<float*>(xw);
    __nv_bfloat16* xb = BF16 ? reinterpret_cast<__nv_bfloat16*>(xw) : nullptr;
    tc::build_b_images<<<dim3(8, n_kb, n_tiles), 256, 0, st>>>(W, K, 1, D, (int)K, BN, n_kb, img);
    const int64_t tiles = int64_t(n_tiles) * ((N + 2 * tc::BM - 1) / (2 * tc::BM));
    int64_t clusters = sm_count() / 2;
    if (tiles < clusters) clusters = tiles;
    const unsigned grid = (unsigned)(2 * clusters);
    GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc_ws2<BF16, BF16, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)tc::WS2_SMEM));
    tc::gemm_tc_ws2<BF16, BF16, HC><<<grid, tc::WS2_THREADS, tc::WS2_SMEM, st>>>(
        x, ldx, N, (int)K, img, n_kb, n_tiles, xf, xb, D, att_src, att_dst, a_src, a_dst, H);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int project_fwd_tc(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst, int64_t N,
                   int64_t K, int H, int C, int xw_dtype, void* xw, float* a_src, float* a_dst, void* ws, size_t ws_bytes,
                   cudaStream_t st)
{
    GNNFD_REQUIRE(tc_supported(N, K, H, C), GNNFD_ERR_UNSUPPORTED, "project_fwd_tc: unsupported shape");
    GNNFD_REQUIRE(xw_dtype == GNNFD_F32 || C == 64, GNNFD_ERR_UNSUPPORTED, "project_fwd: bf16 xw needs C == 64");
    GNNFD_REQUIRE(ws && ws_bytes >= tc_ws_bytes(N, K, H, C), GNNFD_ERR_WORKSPACE, "project_fwd_tc: workspace too small");
    if (N == 0) return GNNFD_OK;
    const int D = H * C;
    if (xw_dtype == GNNFD_BF16) return launch_fwd_tc<64, true>(x, ldx, W, att_src, att_dst, N, K, H, D, xw, a_src, a_dst, ws, st);
    if (C == 32) return launch_fwd_tc<32, false>(x, ldx, W, att_src, att_dst, N, K, H, D, xw, a_src, a_dst, ws, st);
    if (C == 128) return launch_fwd_tc<128, false>(x, ldx, W, att_src, att_dst, N, K, H, D, xw, a_src, a_dst, ws, st);
    return launch_fwd_tc<64, false>(x, ldx, W, att_src, att_dst, N, K, H, D, xw, a_src, a_dst, ws, st);
}

// dx[N,K] = dxw[N,D] @ W[D,K]:  A = dxw (K-major in D), B rows = k (W^T), reduction over D
constexpr int DX_BN = 256;   // TODO(perf): a BN=64/128 instantiation for the K=64 hidden layers
size_t dx_tc_ws_bytes(int64_t K, int D)
{
    return size_t((K + DX_BN - 1) / DX_BN) * tc::kblocks(D) * 2 * (DX_BN * tc::BK) * sizeof(float) + 2048;
}
int project_bwd_dx_tc(const float* dxw, const float* W, int64_t N, int64_t K, int D, float* dx, int64_t lddx, void* ws,
                      size_t ws_bytes, cudaStream_t st)
{
    if (N == 0) return GNNFD_OK;
    constexpr int BN = DX_BN;
    const int n_kb = tc::kblocks(D), n_tiles = int((K + BN - 1) / BN);
    const size_t need = dx_tc_ws_bytes(K, D);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "project_bwd_dx_tc: workspace %zu < %zu", ws_bytes, need);
    float* img = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    // B row r = input feature k, reduction index = output column o: element = W[o*K + k]
    tc::build_b_images<<<dim3(8, n_kb, n_tiles), 256, 0, st>>>(W, 1, K, (int)K, D, BN, n_kb, img);
    const int64_t tiles = int64_t(n_tiles) * ((N + tc::BM - 1) / tc::BM);
    const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
    GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::WS_SMEM));
    tc::gemm_tc_ws<<<grid, tc::WS_THREADS, tc::WS_SMEM, st>>>(dxw, D, N, D, img, n_kb, n_tiles, dx, lddx, (int)K);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

// dW[D,K] = dxw^T @ x over node slabs (partials reduced in slab order => deterministic)
static int dw_slabs(int64_t N)
{
    int64_t s = N / 2048;
    if (s > 74) s = 74;        // D = 512: 2 tiles of 256 output rows x 74 slabs = one CTA on each of the 148 SMs
    if (s < 1) s = 1;
    return (int)s;
}
size_t dw_tc_ws_bytes(int64_t N, int64_t K, int D) { return size_t(dw_slabs(N)) * D * K * sizeof(float) + 1024; }
bool dw_tc_supported(int64_t K, int D) { return tc_device_ok() && K <= 256 && D % 256 == 0; }   // dw_tc2: 256 rows per CTA

template <int NG>
static int launch_dw(const float* dxw, const float* x, int64_t ldx, int64_t N, int64_t K, int D, float* P, int S,
                     int64_t rps, cudaStream_t st)
{
    const int kpad = int((K + 15) / 16 * 16);
    const bool vec2 = (NG % 2 == 0) && (K % 2 == 0) && (ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(x) & 7) == 0;
    const size_t smem = tc::dw2_smem<NG>();
    if (vec2) {
        GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc2<NG, (NG % 2 == 0)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::dw_tc2<NG, (NG % 2 == 0)><<<dim3(D / 256, S), tc::DW2_THREADS, smem, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
    } else {
        GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc2<NG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::dw_tc2<NG, false><<<dim3(D / 256, S), tc::DW2_THREADS, smem, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
    }
    return GNNFD_OK;
}

int project_bwd_dw_tc(const float* dxw, const float* x, int64_t ldx, int64_t N, int64_t K, int D, float* dW, void* ws,
                      size_t ws_bytes, cudaStream_t st)
{
    GNNFD_REQUIRE(dw_tc_supported(K, D), GNNFD_ERR_UNSUPPORTED, "project_bwd_dw_tc: K=%lld D=%d not supported", (long long)K, D);
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(dxw) & 15) == 0, GNNFD_ERR_ARG, "project_bwd_dw_tc: dxw must be 16-byte aligned");
    const int S = dw_slabs(N);
    GNNFD_REQUIRE(ws && ws_bytes >= dw_tc_ws_bytes(N, K, D), GNNFD_ERR_WORKSPACE, "project_bwd_dw_tc: workspace too small");
    float* P = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
    const int64_t rps = ((N + S - 1) / S + tc::BK - 1) / tc::BK * tc::BK;
    const int ng = int((K + 31) / 32);
    GNNFD_CUDA(cudaMemsetAsync(P, 0, size_t(S) * D * K * sizeof(float), st));
    int rc;
    switch (ng) {
        case 1: rc = launch_dw<1>(dxw, x, ldx, N, K, D, P, S, rps, st); break;
        case 2: rc = launch_dw<2>(dxw, x, ldx, N, K, D, P, S, rps, st); break;
        case 3: case 4: rc = launch_dw<4>(dxw, x, ldx, N, K, D, P, S, rps, st); break;
        case 5: case 6: rc = launch_dw<6>(dxw, x, ldx, N, K, D, P, S, rps, st); break;
        default: rc = launch_dw<8>(dxw, x, ldx, N, K, D, P, S, rps, st); break;
    }
    if (rc) return rc;
    tc::reduce_slabs<<<(unsigned)((int64_t(D) * K + 255) / 256), 256, 0, st>>>(P, int64_t(D) * K, S, dW);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace gnnfd
