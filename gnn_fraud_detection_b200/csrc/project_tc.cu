// (2) tensor-core projection: xw = x @ W^T on the 5th-gen tensor cores (tcgen05.mma, accumulators in
// TMEM), error-compensated 3xTF32 so the fp32 parity bar (1e-5) holds, with the per-head attention
// logits a_src/a_dst computed in the epilogue from the TMEM-resident tile.  Also the two projection
// backward GEMMs: dx = dxw @ W (same kernel, transposed weight image) and dW = dxw^T @ x (split over
// node slabs, MN-major operands).
//
// Replaces lin_src(x) / (x*att).sum(-1) of GATConv.forward (reference call site src/models/gat.py:80)
// and their autograd mirror (src/train.py:142).
//
// Data movement
//   * W (and W^T) are split once per call into tf32 hi/lo parts and laid out in global memory as ready-made
//     128B-swizzled shared-memory images, one 64 KB image per (column half, k-block); a CTA fetches an
//     image with ONE cp.async.bulk (bulk async copy engine, mbarrier complete_tx) -- no tensor map needed.
//   * x rows have a 664-byte stride (K=166), not 16-byte aligned, so TMA cannot address them: the A tile
//     is read with coalesced 128-byte row segments, split into hi/lo in registers and stored into the
//     swizzled K-major layout (conflict-free), then published to the async proxy with fence.proxy.async.
//   * one elected thread issues tcgen05.mma.kind::tf32 (M=128, N<=256, K=8): per k-step three MMAs
//     (hi*hi, lo*hi, hi*lo); tcgen05.commit arrives on an mbarrier when the tile's MMAs retire.
//   * epilogue: each warp reads its 32 TMEM lanes (tcgen05.ld 32x32b.x32), a thread owns a full output
//     row so the 64-wide logit dot products need no shuffles; the tile is staged through shared memory
//     and written with coalesced 128-bit stores.
#include "common.cuh"

#include <atomic>
#include <cstdlib>

namespace gnnfd {
extern std::atomic<long long> g_launches;

namespace tc {

constexpr int BM = 128;          // rows per CTA tile (UMMA M)
constexpr int BK = 32;           // tf32 elements per k-block = one 128-byte swizzle row
constexpr int UK = 8;            // tf32 UMMA K
constexpr int THREADS = 128;
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

// split form: issue the load, later wait with the destination registers threaded through the wait (so the compiler
// cannot touch them while the asynchronous load may still be writing them)
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32])
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
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
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

// ---- C[M, NT*BN] = A[M, Kd] * B^T, A fp32 row-major (lda), B as prebuilt images ----------------------
// EPI 1: forward epilogue -- store xw (fp32 / bf16) and the per-head logits of heads HC columns wide; BN must be a
//        multiple of HC.
// EPI 0: plain fp32 store of the first n_valid columns (ldc).
template <int BN, int EPI, bool OUT_BF16, int HC = 64>
__global__ void __launch_bounds__(THREADS)
gemm_tc(const float* __restrict__ A, int64_t lda, int64_t M, int Kd, const float* __restrict__ b_img, int n_kb,
        float* __restrict__ Cf, __nv_bfloat16* __restrict__ Cb, int64_t ldc, int n_valid,
        const float* __restrict__ att_src, const float* __restrict__ att_dst, float* __restrict__ a_src,
        float* __restrict__ a_dst, int H)
{
    constexpr uint32_t A_BYTES = BM * 128;        // one part (hi or lo) of the A k-block
    constexpr uint32_t B_BYTES = BN * 128;        // one part of the B k-block
    constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr uint32_t IDESC = make_idesc(BM, BN, 0, 0);
    constexpr int STG_LD = 36;                    // staging row stride (floats): conflict-free float4 both ways
    static_assert(HC == 32 || HC == 64 || HC == 128, "the logits epilogue covers heads of 32, 64 or 128 columns");
    static_assert(EPI == 0 || BN % HC == 0, "a column tile holds whole heads");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA_hi = smem;
    uint8_t* sA_lo = smem + A_BYTES;
    uint8_t* sB = smem + 2 * A_BYTES;             // [hi | lo], exactly the global image
    __shared__ uint64_t bar_b, bar_mma;
    __shared__ uint32_t tmem_base_s;
    __shared__ float att_s[2][BN];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // 1-D grid, column tile fastest: the CTAs sharing an A tile are co-scheduled, so its re-read hits L2
    const int n_col_tiles = (n_valid + BN - 1) / BN;
    const int nt = blockIdx.x % n_col_tiles;
    const int64_t m0 = int64_t(blockIdx.x / n_col_tiles) * BM;
    const float* img = b_img + size_t(nt) * n_kb * 2 * (size_t(BN) * BK);

    if (tid == 0) {
        mbar_init(&bar_b, 1);
        mbar_init(&bar_mma, 1);
        fence_mbar_init();
    }
    if (EPI == 1)
        for (int i = tid; i < BN; i += THREADS) {
            att_s[0][i] = att_src[nt * BN + i];
            att_s[1][i] = att_dst[nt * BN + i];
        }
    if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;

    // A k-block loader: warp w owns rows [32w, 32w+32); lane = k element -> 128-byte coalesced row segments
    float xr[32];
    auto load_a = [&](int kb) {
        const int gk = kb * BK + lane;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int64_t gm = m0 + warp * 32 + i;
            xr[i] = (gm < M && gk < Kd) ? __ldg(A + gm * lda + gk) : 0.f;
        }
    };
    load_a(0);
    for (int kb = 0; kb < n_kb; ++kb) {
        if (kb > 0) mbar_wait(&bar_mma, (kb - 1) & 1);     // previous k-block's MMAs retired: smem is free
        if (tid == 0) {
            mbar_expect_tx(&bar_b, 2 * B_BYTES);
            bulk_g2s(sB, img + size_t(kb) * 2 * (size_t(BN) * BK), 2 * B_BYTES, &bar_b);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int r = warp * 32 + i;
            float h, l;
            split_tf32(xr[i], h, l);
            const uint32_t off = kmajor_off(r, lane);
            *reinterpret_cast<float*>(sA_hi + off) = h;
            *reinterpret_cast<float*>(sA_lo + off) = l;
        }
        fence_proxy_async();                               // generic-proxy stores -> visible to the tensor core
        __syncthreads();
        if (tid == 0) {
            mbar_wait(&bar_b, kb & 1);
            tc_fence_after();
            const int ksteps = min(BK / UK, (Kd - kb * BK + UK - 1) / UK);
            const uint32_t a_hi = smem_u32(sA_hi), a_lo = smem_u32(sA_lo), b_hi = smem_u32(sB), b_lo = smem_u32(sB + B_BYTES);
            for (int ks = 0; ks < ksteps; ++ks) {
                const uint32_t ko = ks * UK * 4;           // 32 bytes per k-step inside the swizzled row
                const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                umma_tf32(tmem_d, dah, dbh, IDESC, (kb | ks) ? 1u : 0u);
                umma_tf32(tmem_d, dal, dbh, IDESC, 1u);
                umma_tf32(tmem_d, dah, dbl, IDESC, 1u);
            }
            umma_commit(&bar_mma);
        }
        if (kb + 1 < n_kb) load_a(kb + 1);                 // global loads overlap the MMAs
    }
    mbar_wait(&bar_mma, (n_kb - 1) & 1);
    tc_fence_after();

    // ---- epilogue: warp w <-> TMEM lanes [32w, 32w+32), thread <-> one output row ----------------------
    float* stg = reinterpret_cast<float*>(smem) + warp * (32 * STG_LD);   // A/B stage memory is free now
    const int64_t row = m0 + warp * 32 + lane;
    float ps = 0.f, pd = 0.f;
#pragma unroll 1
    for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t v[32];
        tmem_ld32(tmem_d + (uint32_t(warp * 32) << 16) + ch * 32, v);
        if (EPI == 1) {
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const float f = __uint_as_float(v[c]);
                ps = fmaf(f, att_s[0][ch * 32 + c], ps);
                pd = fmaf(f, att_s[1][ch * 32 + c], pd);
            }
            if ((ch & (HC / 32 - 1)) == HC / 32 - 1) {      // HC/32 32-column chunks per head
                if (row < M) {
                    const int h = (nt * BN + ch * 32) / HC;
                    a_src[row * H + h] = ps;
                    a_dst[row * H + h] = pd;
                }
                ps = pd = 0.f;
            }
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 32; c += 4)
            *reinterpret_cast<float4*>(stg + lane * STG_LD + c) =
                make_float4(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), __uint_as_float(v[c + 2]),
                            __uint_as_float(v[c + 3]));
        __syncwarp();
        const int col0 = nt * BN + ch * 32;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + (lane >> 3), cq = (lane & 7) * 4;
            const int64_t gm = m0 + warp * 32 + r;
            const float4 o = *reinterpret_cast<const float4*>(stg + r * STG_LD + cq);
            if (gm < M) {
                if (EPI == 1) {
                    if (OUT_BF16) {
                        __nv_bfloat162 lo2 = __floats2bfloat162_rn(o.x, o.y), hi2 = __floats2bfloat162_rn(o.z, o.w);
                        uint2 pk;
                        pk.x = *reinterpret_cast<uint32_t*>(&lo2);
                        pk.y = *reinterpret_cast<uint32_t*>(&hi2);
                        *reinterpret_cast<uint2*>(Cb + gm * ldc + col0 + cq) = pk;
                    } else {
                        *reinterpret_cast<float4*>(Cf + gm * ldc + col0 + cq) = o;
                    }
                } else {
                    const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (col0 + cq + k < n_valid) Cf[gm * ldc + col0 + cq + k] = ov[k];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_d, TMEM_COLS);
}


// ---- dW partials on the tensor cores: P[slab][o][k] = sum_{n in slab} dxw[n][o] * x[n][k] -------------
// Reduction runs over nodes, so both operands are "MN-major" (the contiguous global dimension is o resp. k).
// For 32-bit MN-major operands the only swizzled layout is SWIZZLE_128B_BASE32B (layout type 1,
// cute::UMMA::Layout_MN_SW128_32B_Atom): atoms of 4 node rows x 128 bytes (32 consecutive o / k), the 32-byte
// chunk index XOR-ed with (node row % 4); LBO = stride between 32-element MN groups, SBO = stride between
// 4-node groups.  One K=8 MMA consumes two consecutive node groups.
// VEC2: x rows are 8-byte aligned (even ldx), so the B operand is read and staged as float2 pairs -- half the
// load/store instructions on the LSU pipe, which the two co-resident CTAs share.
template <int NG, bool VEC2>   // NG = number of 32-wide k groups of the B operand (N = KPAD <= 32*NG), even if VEC2
__global__ void __launch_bounds__(THREADS)
dw_tc(const float* __restrict__ dxw, int D, const float* __restrict__ x, int64_t ldx, int64_t N, int K, int kpad,
      int64_t rows_per_slab, float* __restrict__ P)
{
    constexpr uint32_t A_PART = 4 * 4 * 1024;        // 4 node groups x 4 o groups x 1 KB
    constexpr uint32_t B_PART = 4 * NG * 1024;
    constexpr uint32_t TMEM_COLS = NG * 32 <= 32 ? 32 : NG * 32 <= 64 ? 64 : NG * 32 <= 128 ? 128 : 256;
    constexpr int STG_LD = 36;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA_hi = smem;
    uint8_t* sA_lo = smem + A_PART;
    uint8_t* sB_hi = smem + 2 * A_PART;
    uint8_t* sB_lo = sB_hi + B_PART;
    __shared__ uint64_t bar_mma;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = blockIdx.x * BM;                  // o tile
    const int64_t nb = int64_t(blockIdx.y) * rows_per_slab;
    const int64_t ne = (nb + rows_per_slab < N) ? nb + rows_per_slab : N;
    const int n_kb = int((ne - nb + BK - 1) / BK);
    const uint32_t idesc = make_idesc(BM, kpad, 1, 1);

    if (tid == 0) {
        mbar_init(&bar_mma, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;

    // warp w stages node group kg = w (8 node rows) of every k-block
    float4 ar[8];
    float br[8][NG];
    auto load_blk = [&](int kb) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int64_t n = nb + int64_t(kb) * BK + warp * 8 + j;
            const bool ok = n < ne;
            ar[j] = ok ? __ldg(reinterpret_cast<const float4*>(dxw + n * D + m0) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (VEC2) {
                // lane owns the feature pairs 2*lane + 64*t', t' < NG/2 (K is even: a pair is never split by K)
#pragma unroll
                for (int t = 0; t < NG / 2; ++t) {
                    const int kf = 2 * lane + 64 * t;
                    const float2 v = (ok && kf < K) ? __ldg(reinterpret_cast<const float2*>(x + n * ldx + kf)) : make_float2(0.f, 0.f);
                    br[j][2 * t] = v.x;
                    br[j][2 * t + 1] = v.y;
                }
            } else {
#pragma unroll
                for (int t = 0; t < NG; ++t) {
                    const int kf = lane + 32 * t;
                    br[j][t] = (ok && kf < K) ? __ldg(x + n * ldx + kf) : 0.f;
                }
            }
        }
    };
    // The tensor core accumulates with round-toward-zero, so a long reduction chain drifts (measured: ~2e-5
    // relative after 3000 nodes).  Every FLUSH_KB k-blocks (512 nodes) the TMEM tile is therefore drained
    // into this CTA's private fp32 partial in global memory (L2-resident: 128 x K floats) and the
    // accumulation restarts from zero.
    constexpr int FLUSH_KB = 16;
    float* Ps = P + int64_t(blockIdx.y) * D * K;
    float* stg = reinterpret_cast<float*>(smem) + warp * (32 * STG_LD);
    auto flush = [&](bool first, bool have_acc) {
#pragma unroll 1
        for (int ch = 0; ch < NG; ++ch) {
            uint32_t v[32];
            if (have_acc) tmem_ld32(tmem_d + (uint32_t(warp * 32) << 16) + ch * 32, v);
            else {
#pragma unroll
                for (int c = 0; c < 32; ++c) v[c] = 0u;
            }
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 32; c += 4)
                *reinterpret_cast<float4*>(stg + lane * STG_LD + c) =
                    make_float4(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), __uint_as_float(v[c + 2]),
                                __uint_as_float(v[c + 3]));
            __syncwarp();
            const int kf = ch * 32 + lane;
            if (kf < K) {
                // fire-and-forget fp32 reductions (RED.ADD, round-to-nearest in L2): the partial is private to
                // this CTA, so there is no contention and the flush never waits on a load
                (void)first;
#pragma unroll 8
                for (int r = 0; r < 32; ++r) atomicAdd(Ps + int64_t(m0 + warp * 32 + r) * K + kf, stg[r * STG_LD + lane]);
            }
        }
    };

    if (n_kb > 0) load_blk(0);
    int flushed = 0;
    for (int kb = 0; kb < n_kb; ++kb) {
        if (kb > 0) mbar_wait(&bar_mma, (kb - 1) & 1);
        if (kb > 0 && kb % FLUSH_KB == 0) {
            // all MMAs so far have retired (barrier above): drain, then the staging area is rewritten below
            tc_fence_after();
            flush(flushed == 0, true);
            ++flushed;
            tc_fence_before();
            __syncthreads();
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            // node row r = 8*warp + j -> node group kq = r/4, row-in-group jr = r%4
            const uint32_t kq = uint32_t(warp * 2 + (j >> 2)), jr = uint32_t(j & 3);
            // A: o = 4*lane..4*lane+3 -> o group lane/8, 32-byte chunk (lane%8)/2, 16-byte half lane%2
            const uint32_t offA = (kq * 4u + uint32_t(lane >> 3)) * 512u + jr * 128u +
                                  ((uint32_t((lane & 7) >> 1) ^ jr) << 5) + (uint32_t(lane & 1) << 4);
            float4 h, l;
            split_tf32(ar[j].x, h.x, l.x); split_tf32(ar[j].y, h.y, l.y);
            split_tf32(ar[j].z, h.z, l.z); split_tf32(ar[j].w, h.w, l.w);
            *reinterpret_cast<float4*>(sA_hi + offA) = h;
            *reinterpret_cast<float4*>(sA_lo + offA) = l;
            if (VEC2) {
#pragma unroll
                for (int t = 0; t < NG / 2; ++t) {
                    // features f = 2*lane + 64*t, f+1: 32-feature group 2t + lane/16, position fi = (2*lane) % 32
                    const uint32_t grp = uint32_t(2 * t + (lane >> 4)), fi = uint32_t((2 * lane) & 31);
                    const uint32_t offB = (kq * uint32_t(NG) + grp) * 512u + jr * 128u + (((fi >> 3) ^ jr) << 5) + (fi & 7u) * 4u;
                    float2 hh, ll;
                    split_tf32(br[j][2 * t], hh.x, ll.x);
                    split_tf32(br[j][2 * t + 1], hh.y, ll.y);
                    *reinterpret_cast<float2*>(sB_hi + offB) = hh;
                    *reinterpret_cast<float2*>(sB_lo + offB) = ll;
                }
            } else {
#pragma unroll
                for (int t = 0; t < NG; ++t) {
                    const uint32_t offB = (kq * uint32_t(NG) + uint32_t(t)) * 512u + jr * 128u +
                                          ((uint32_t(lane >> 3) ^ jr) << 5) + uint32_t(lane & 7) * 4u;
                    float hh, ll;
                    split_tf32(br[j][t], hh, ll);
                    *reinterpret_cast<float*>(sB_hi + offB) = hh;
                    *reinterpret_cast<float*>(sB_lo + offB) = ll;
                }
            }
        }
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint32_t a_hi = smem_u32(sA_hi), a_lo = smem_u32(sA_lo), b_hi = smem_u32(sB_hi), b_lo = smem_u32(sB_lo);
            const bool restart = (kb % FLUSH_KB) == 0;
#pragma unroll
            for (int kg = 0; kg < 4; ++kg) {   // k-step = 8 nodes = two 4-node groups
                const uint64_t dah = make_desc(a_hi + kg * 4096, 512, 2048, 1), dal = make_desc(a_lo + kg * 4096, 512, 2048, 1);
                const uint64_t dbh = make_desc(b_hi + kg * NG * 1024, 512, NG * 512, 1);
                const uint64_t dbl = make_desc(b_lo + kg * NG * 1024, 512, NG * 512, 1);
                umma_tf32(tmem_d, dah, dbh, idesc, (restart && kg == 0) ? 0u : 1u);
                umma_tf32(tmem_d, dal, dbh, idesc, 1u);
                umma_tf32(tmem_d, dah, dbl, idesc, 1u);
            }
            umma_commit(&bar_mma);
        }
        if (kb + 1 < n_kb) load_blk(kb + 1);
    }
    if (n_kb > 0) {
        mbar_wait(&bar_mma, (n_kb - 1) & 1);
        tc_fence_after();
    }
    flush(flushed == 0, n_kb > 0);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_d, TMEM_COLS);
}

__global__ void reduce_slabs(const float* __restrict__ P, int64_t n, int S, float* __restrict__ out)
{
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < S; ++k) s += P[int64_t(k) * n + i];
        out[i] = s;
    }
}

template <int BN>
constexpr size_t gemm_smem_bytes() { return 2 * BM * 128 + 2 * BN * 128 + 1024; }

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
// GNNFD_GEMM_WS=0 selects the simpler one-tile-per-CTA kernel (kept for A/B measurements)
// GNNFD_GEMM_WS: 0 = simple one-tile-per-CTA kernel, 1 = persistent warp-specialised 1-SM kernel,
// 2 = 2-SM (cta_group::2) kernel
static int ws_mode()
{
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("GNNFD_GEMM_WS");
        v = e ? atoi(e) : 2;
    }
    return v;
}
static bool use_ws()
{
    return ws_mode() >= 1;
}
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
    if (ws_mode() == 2) {
        const int64_t tiles = int64_t(n_tiles) * ((N + 2 * tc::BM - 1) / (2 * tc::BM));
        int64_t clusters = sm_count() / 2;
        if (tiles < clusters) clusters = tiles;
        const unsigned grid = (unsigned)(2 * clusters);
        GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc_ws2<1, BF16, BF16, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)tc::WS2_SMEM));
        tc::gemm_tc_ws2<1, BF16, BF16, HC><<<grid, tc::WS2_THREADS, tc::WS2_SMEM, st>>>(
            x, ldx, N, (int)K, img, n_kb, n_tiles, xf, xb, D, D, att_src, att_dst, a_src, a_dst, H);
    } else if (use_ws()) {
        const int64_t tiles = int64_t(n_tiles) * ((N + tc::BM - 1) / tc::BM);
        const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
        GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc_ws<1, BF16, BF16, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)tc::WS_SMEM));
        tc::gemm_tc_ws<1, BF16, BF16, HC><<<grid, tc::WS_THREADS, tc::WS_SMEM, st>>>(
            x, ldx, N, (int)K, img, n_kb, n_tiles, xf, xb, D, D, att_src, att_dst, a_src, a_dst, H);
    } else {
        const size_t smem = tc::gemm_smem_bytes<BN>();
        dim3 grid((unsigned)(int64_t(n_tiles) * ((N + tc::BM - 1) / tc::BM)));
        GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc<BN, 1, BF16, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc<BN, 1, BF16, HC><<<grid, tc::THREADS, smem, st>>>(x, ldx, N, (int)K, img, n_kb, xf, xb, D, D, att_src,
                                                                      att_dst, a_src, a_dst, H);
    }
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
int project_bwd_dx_tc(const float* dxw, const float* W, int64_t N, int64_t K, int D, float* dx, int64_t lddx, void* ws,
                      size_t ws_bytes, cudaStream_t st)
{
    if (N == 0) return GNNFD_OK;
    constexpr int BN = 256;   // TODO(perf): a BN=64/128 instantiation for the K=64 hidden layers
    const int n_kb = tc::kblocks(D), n_tiles = int((K + BN - 1) / BN);
    const size_t need = size_t(n_tiles) * n_kb * 2 * (BN * tc::BK) * sizeof(float) + 2048;
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "project_bwd_dx_tc: workspace %zu < %zu", ws_bytes, need);
    float* img = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    // B row r = input feature k, reduction index = output column o: element = W[o*K + k]
    tc::build_b_images<<<dim3(8, n_kb, n_tiles), 256, 0, st>>>(W, 1, K, (int)K, D, BN, n_kb, img);
    if (use_ws()) {
        const int64_t tiles = int64_t(n_tiles) * ((N + tc::BM - 1) / tc::BM);
        const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
        GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc_ws<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::WS_SMEM));
        tc::gemm_tc_ws<0, false><<<grid, tc::WS_THREADS, tc::WS_SMEM, st>>>(dxw, D, N, D, img, n_kb, n_tiles, dx, nullptr, lddx,
                                                                          (int)K, nullptr, nullptr, nullptr, nullptr, 0);
        g_launches += 2;
        GNNFD_LAUNCH_CHECK();
        return GNNFD_OK;
    }
    const size_t smem = tc::gemm_smem_bytes<BN>();
    GNNFD_CUDA(cudaFuncSetAttribute(tc::gemm_tc<BN, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)(int64_t(n_tiles) * ((N + tc::BM - 1) / tc::BM)));
    tc::gemm_tc<BN, 0, false><<<grid, tc::THREADS, smem, st>>>(dxw, D, N, D, img, n_kb, dx, nullptr, lddx, (int)K, nullptr,
                                                              nullptr, nullptr, nullptr, 0);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

// dW[D,K] = dxw^T @ x over node slabs (partials reduced in slab order => deterministic)
static int dw_slabs(int64_t N)
{
    int64_t s = N / 2048;
    if (s > 74) s = 74;        // 4 o-tiles x 74 slabs = one wave of 2 CTAs on each of the 148 SMs
    if (s < 1) s = 1;
    return (int)s;
}
size_t dw_tc_ws_bytes(int64_t N, int64_t K, int D) { return size_t(dw_slabs(N)) * D * K * sizeof(float) + 1024; }
bool dw_tc_supported(int64_t K, int D) { return tc_device_ok() && K <= 256 && D % tc::BM == 0; }

template <int NG>
static int launch_dw(const float* dxw, const float* x, int64_t ldx, int64_t N, int64_t K, int D, float* P, int S,
                     int64_t rps, cudaStream_t st)
{
    const size_t smem = 2 * (16 * 1024) + 2 * (4 * NG * 1024) + 1024;
    const int kpad = int((K + 15) / 16 * 16);
    const bool vec2 = (NG % 2 == 0) && (K % 2 == 0) && (ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(x) & 7) == 0;
    static const int dw_mode = [] {
        const char* e = getenv("GNNFD_DW_TC");      // 1 = one-stage kernel (two CTAs per SM), 2 = pipelined 256-row kernel
        return e ? atoi(e) : 2;
    }();
    if (dw_mode == 2 && D % 256 == 0) {
        const size_t smem2 = tc::dw2_smem<NG>();
        if (vec2) {
            GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc2<NG, (NG % 2 == 0)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            tc::dw_tc2<NG, (NG % 2 == 0)><<<dim3(D / 256, S), tc::DW2_THREADS, smem2, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
        } else {
            GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc2<NG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            tc::dw_tc2<NG, false><<<dim3(D / 256, S), tc::DW2_THREADS, smem2, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
        }
        return GNNFD_OK;
    }
    if (vec2) {
        GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc<NG, (NG % 2 == 0)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::dw_tc<NG, (NG % 2 == 0)><<<dim3(D / tc::BM, S), tc::THREADS, smem, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
    } else {
        GNNFD_CUDA(cudaFuncSetAttribute(tc::dw_tc<NG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::dw_tc<NG, false><<<dim3(D / tc::BM, S), tc::THREADS, smem, st>>>(dxw, D, x, ldx, N, (int)K, kpad, rps, P);
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
