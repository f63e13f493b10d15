// Persistent, warp-specialised tcgen05 GEMM:  C[M, NT*256] = A[M, Kd] * B^T  (3xTF32, fp32 accumulate in TMEM).
// The projection backward's dx = dxw @ W; the forward runs the 2-SM variant (project_tc_ws2.cuh).
//
// One CTA per SM, 10 warps:
//   warps 0-3  A producers: coalesced 128-byte row segments of x -> hi/lo split -> swizzled K-major smem stage
//              (three-step register ring, next tile's rows prefetched into L2)
//   warp  4    MMA issuer (one elected lane): waits only for FULL barriers, so the tcgen05.mma's of consecutive
//              k-blocks queue back to back; tcgen05.commit releases the smem stage and, on a tile's last
//              k-block, hands the TMEM accumulator to the epilogue
//   warps 5-8  epilogue: tcgen05.ld of their TMEM lane quadrant, staged coalesced stores of the first n_valid columns
//   warp  9    B producer: cp.async.bulk of the prebuilt weight image of each k-block as soon as its stage drains
// Two smem stages (A 2x32 KB, B 2x64 KB) and two TMEM accumulators (2 x 256 columns) keep all roles busy:
// the epilogue of tile t overlaps the mainloop of tile t+1, the copies of k-block k+1 overlap the MMAs of k.
#pragma once

namespace gnnfd {
namespace tc {

constexpr int WS_THREADS = 320;
constexpr int WS_BN = 256;
constexpr uint32_t WS_A_PART = BM * 128;            // 16 KB: one part (hi or lo) of an A k-block
constexpr uint32_t WS_B_PART = WS_BN * 128;         // 32 KB
constexpr uint32_t WS_STAGE = 2 * WS_A_PART + 2 * WS_B_PART;   // 96 KB
constexpr int WS_STG_LD = 36;
constexpr size_t WS_SMEM = 2 * WS_STAGE + 4 * 32 * WS_STG_LD * 4 + 1024;

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
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(WS_THREADS, 1)
gemm_tc_ws(const float* __restrict__ A, int64_t lda, int64_t M, int Kd, const float* __restrict__ b_img, int n_kb,
           int n_col_tiles, float* __restrict__ Cf, int64_t ldc, int n_valid)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full_a[2], full_b[2], empty[2], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);     // warp-uniform for the compiler (uniform datapath)
    const int64_t m_tiles = (M + BM - 1) / BM;
    const int64_t n_tiles = m_tiles * n_col_tiles;           // tile id = m * n_col_tiles + nt  (nt fastest)

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(&full_a[s], 4);                 // one arrive per producer warp
            mbar_init(&full_b[s], 1);
            mbar_init(&empty[s], 1);
            mbar_init(&acc_full[s], 1);
            mbar_init(&acc_empty[s], 4);              // one arrive per epilogue warp
        }
        fence_mbar_init();
    }
    if (warp == 4) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp < 4) {
        // ---------------- A producers ----------------------------------------------------------------
        // software-pipelined by one step: the global loads of step i+1 are in flight while step i is split and
        // stored, so neither the DRAM/L2 latency nor the smem stores sit on the MMA critical path
        const int64_t my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
        const int64_t n_steps = my_tiles * n_kb;
        const uint32_t lda32 = uint32_t(lda);
        auto load_step = [&](int64_t step, float (&xr)[32]) {
            const int64_t t = blockIdx.x + (step / n_kb) * gridDim.x;
            const int64_t m0 = (t / n_col_tiles) * BM;
            const int kb = int(step % n_kb);
            const int gk = kb * BK + lane;
            if (kb == 0 && t + gridDim.x < n_tiles) {
                // pull the NEXT tile's rows (one contiguous block of A) into L2 while this tile is processed:
                // the 32 scalar loads per thread below then see L2 latency instead of DRAM latency
                const int64_t m1 = ((t + gridDim.x) / n_col_tiles) * BM;
                const int64_t m2 = (m1 + BM < M) ? m1 + BM : M;
                const char* pb = reinterpret_cast<const char*>(A + m1 * lda);
                const int64_t nbytes = (m2 - m1) * lda * int64_t(sizeof(float));
                for (int64_t off = int64_t(warp * 32 + lane) * 128; off < nbytes; off += 128 * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(pb + off));
            }
            // one producer warp per scheduler cannot hide instruction latency, so the interior path carries no
            // predicates and one address instruction per element (uniform 64-bit base + 32-bit offset)
            const float* base = A + (m0 + warp * 32) * lda;
            if (m0 + BM <= M && (kb + 1) * BK <= Kd) {
                uint32_t off = uint32_t(gk);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    xr[i] = __ldg(base + off);
                    off += lda32;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int64_t gm = m0 + warp * 32 + i;
                    xr[i] = (gm < M && gk < Kd) ? __ldg(base + uint32_t(i) * lda32 + uint32_t(gk)) : 0.f;
                }
            }
        };
        // swizzled K-major position of (row warp*32+i, k = lane): the lane-dependent part takes 8 values (i % 8)
        const uint32_t smem_a = smem_u32(smem) + uint32_t(warp) * 4096u;
        auto store_step = [&](int64_t step, const float (&xr)[32]) {
            const int s = int(step & 1);
            const int64_t u = step >> 1;
            if (u > 0) mbar_wait(&empty[s], uint32_t((u - 1) & 1));   // MMAs that read this stage have retired
            const uint32_t a_hi = smem_a + uint32_t(s) * WS_STAGE;
            uint32_t lp[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) lp[j] = a_hi + ((uint32_t((lane >> 2) ^ j)) << 4) + (uint32_t(lane & 3) << 2);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                float h, l;
                split_tf32(xr[i], h, l);
                const uint32_t a = lp[i & 7] + uint32_t((i >> 3) * 1024 + (i & 7) * 128);   // folded into the STS immediate
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(h) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + WS_A_PART), "f"(l) : "memory");
            }
            fence_proxy_async();
            __syncwarp();                                  // every lane's stores + proxy fence precede the arrive
            if (lane == 0) mbar_arrive(&full_a[s]);
        };
        // register ring of three steps: the loads of step i+2 are issued before step i is split and stored, so an
        // L2 (or DRAM) round trip is covered by a whole store phase plus the wait for the stage to drain
        float xa[32], xb[32], xc[32];
        if (n_steps > 0) load_step(0, xa);
        if (n_steps > 1) load_step(1, xb);
        for (int64_t step = 0; step < n_steps; step += 3) {
            if (step + 2 < n_steps) load_step(step + 2, xc);
            store_step(step, xa);
            if (step + 1 < n_steps) {
                if (step + 3 < n_steps) load_step(step + 3, xa);
                store_step(step + 1, xb);
            }
            if (step + 2 < n_steps) {
                if (step + 4 < n_steps) load_step(step + 4, xb);
                store_step(step + 2, xc);
            }
        }
    } else if (warp == 4) {
        // ---------------- MMA issue (one elected lane) ---------------------------------------------------
        {
            // the whole warp walks the loop with warp-uniform operands (descriptors live in uniform registers);
            // one elected lane issues the asynchronous instructions
            constexpr uint32_t IDESC = make_idesc(BM, WS_BN, 0, 0);
            const int64_t my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
            const int64_t n_steps = my_tiles * n_kb;
            for (int64_t step = 0; step < n_steps; ++step) {
                const int64_t j = step / n_kb;                        // CTA-local tile counter
                const int kb = int(step % n_kb);
                const int s = int(step & 1);
                const uint32_t par = uint32_t((step >> 1) & 1);
                const int buf = int(j & 1);
                if (kb == 0 && (j >> 1) > 0) {                        // accumulator buffer drained by the epilogue?
                    mbar_wait(&acc_empty[buf], uint32_t(((j >> 1) - 1) & 1));
                    tc_fence_after();
                }
                mbar_wait(&full_a[s], par);
                mbar_wait(&full_b[s], par);
                tc_fence_after();
                const uint32_t a_hi = smem_u32(smem + s * WS_STAGE), a_lo = a_hi + WS_A_PART;
                const uint32_t b_hi = a_hi + 2 * WS_A_PART, b_lo = b_hi + WS_B_PART;
                const uint32_t d = tmem_base + uint32_t(buf * WS_BN);
                const int ksteps = min(BK / UK, (Kd - kb * BK + UK - 1) / UK);
                if (elect_one()) {
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint32_t ko = ks * UK * 4;
                        const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                        const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                        umma_tf32(d, dah, dbh, IDESC, (kb | ks) ? 1u : 0u);
                        umma_tf32(d, dal, dbh, IDESC, 1u);
                        umma_tf32(d, dah, dbl, IDESC, 1u);
                    }
                    umma_commit(&empty[s]);                           // stage reusable once these MMAs retire
                    if (kb == n_kb - 1) umma_commit(&acc_full[buf]);  // ... and the tile is complete
                }
                __syncwarp();
            }
        }
    } else if (warp == 9) {
        // ---------------- B producer: cp.async.bulk of the prebuilt weight images -------------------------
        // Its own warp, so that the MMA issuer never waits for a stage to drain: the issuer only waits for FULL
        // barriers and keeps the tensor pipe queued across k-blocks.
        const int64_t my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
        const int64_t n_steps = my_tiles * n_kb;
        auto issue_b = [&](int64_t step) {
            const int64_t t = blockIdx.x + (step / n_kb) * gridDim.x;
            const int kb = int(step % n_kb), nt = int(t % n_col_tiles);
            const int s = int(step & 1);
            const int64_t u = step >> 1;
            if (u > 0) mbar_wait(&empty[s], uint32_t((u - 1) & 1));
            uint8_t* sB = smem + s * WS_STAGE + 2 * WS_A_PART;
            const float* img = b_img + (size_t(nt) * n_kb + kb) * 2 * (size_t(WS_BN) * BK);
            if (elect_one()) {
                mbar_expect_tx(&full_b[s], 2 * WS_B_PART);
                bulk_g2s(sB, img, 2 * WS_B_PART, &full_b[s]);
            }
            __syncwarp();
        };
        for (int64_t step = 0; step < n_steps; ++step) issue_b(step);
    } else {
        // ---------------- epilogue (warps 5..8 -> TMEM lane quadrants 1,2,3,0) ---------------------------
        const int quad = warp & 3;
        float* stg = reinterpret_cast<float*>(smem + 2 * WS_STAGE) + (warp - 5) * (32 * WS_STG_LD);
        int64_t j = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
            const int64_t m0 = (t / n_col_tiles) * BM;
            const int nt = int(t % n_col_tiles);
            const int buf = int(j & 1);
            mbar_wait(&acc_full[buf], uint32_t((j >> 1) & 1));
            tc_fence_after();
#pragma unroll 1
            for (int ch = 0; ch < WS_BN / 32; ++ch) {
                uint32_t v[32];
                tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(buf * WS_BN + ch * 32), v);
                const int col0 = nt * WS_BN + ch * 32;
                // staged through smem so that every store instruction writes four full 128-byte lines (writing each
                // thread's own row directly was measured 40 % slower: 16-byte fragments of 32 different lines)
                __syncwarp();
#pragma unroll
                for (int c = 0; c < 32; c += 4)
                    *reinterpret_cast<float4*>(stg + lane * WS_STG_LD + c) =
                        make_float4(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), __uint_as_float(v[c + 2]),
                                    __uint_as_float(v[c + 3]));
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + (lane >> 3), cq = (lane & 7) * 4;
                    const int64_t gm = m0 + quad * 32 + r;
                    const float4 o = *reinterpret_cast<const float4*>(stg + r * WS_STG_LD + cq);
                    if (gm < M) {
                        const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (col0 + cq + k < n_valid) Cf[gm * ldc + col0 + cq + k] = ov[k];
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
    if (warp == 4) {
        __syncwarp();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace tc
}  // namespace gnnfd
