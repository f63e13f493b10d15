// 2-SM variant of the persistent warp-specialised GEMM:  C[M, NT*256] = A[M, Kd] * B^T  (3xTF32, fp32 in TMEM).
//
// Two CTAs of a cluster (a pair of SMs) work on one 256 x 256 tile with tcgen05.mma.cta_group::2: each CTA
// produces the A operand of ITS 128 rows and holds only HALF of the B (weight) image; the tensor cores of both
// SMs read the two halves across the pair.  Per SM and tile this halves the shared-memory traffic of B (bulk-copy
// writes and operand reads), which is what bounds the 1-SM kernel (project_tc_ws.cuh), and the smaller stage
// (A 32 KB + B 32 KB) leaves room for THREE stages.
//
// Roles per CTA (11 warps):
//   warps 0-3  A producers (both CTAs): x rows -> hi/lo split -> swizzled K-major stage; arrive on the LEADER's
//              full_a barrier (remote arrive from the peer CTA)
//   warp  4    leader: MMA issuer (one elected lane), tcgen05.commit multicast to both CTAs' barriers;
//              both CTAs: TMEM allocation (cta_group::2)
//   warps 5-8  epilogue (both CTAs): own TMEM lanes -> logits -> staged coalesced stores; arrive on the leader's
//              acc_empty barrier
//   warp  9    B producer (both CTAs): cp.async.bulk of this CTA's half image, local full_b barrier
//   warp 10    peer only: forwards "my half of B has landed" to the leader's full_b barrier
#pragma once

namespace gnnfd {
namespace tc {

constexpr int WS2_THREADS = 352;
constexpr int WS2_STAGES = 3;
constexpr uint32_t WS2_A_PART = BM * 128;                 // 16 KB: hi or lo of this CTA's 128 rows
constexpr uint32_t WS2_B_PART = 128 * 128;                // 16 KB: hi or lo of this CTA's 128 weight rows
constexpr uint32_t WS2_STAGE = 2 * WS2_A_PART + 2 * WS2_B_PART;   // 64 KB
constexpr size_t WS2_SMEM = WS2_STAGES * WS2_STAGE + 4 * 32 * WS_STG_LD * 4 + 1024;

__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait with cluster-scope acquire (the arrivals may come from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity)
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
        if (++spins > SPIN_LIMIT) __trap();
    }
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma2_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum)
{
    const uint32_t z = 0;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum), "r"(z)
        : "memory");
}
// arrive (once the MMAs issued so far have retired) on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar)
{
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}

// The forward projection: stores xw (fp32, or bf16 with OUT_BF16) and the per-head logits of heads HC columns wide;
// FAST runs one TF32 pass instead of the compensated three.
template <bool OUT_BF16, bool FAST = false, int HC = 64>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(WS2_THREADS, 1)
gemm_tc_ws2(const float* __restrict__ A, int64_t lda, int64_t M, int Kd, const float* __restrict__ b_img, int n_kb,
            int n_col_tiles, float* __restrict__ Cf, __nv_bfloat16* __restrict__ Cb, int64_t ldc,
            const float* __restrict__ att_src, const float* __restrict__ att_dst, float* __restrict__ a_src,
            float* __restrict__ a_dst, int H)
{
    static_assert(HC == 32 || HC == 64 || HC == 128, "the logits epilogue covers heads of 32, 64 or 128 columns");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full_a[WS2_STAGES], full_b[WS2_STAGES], empty[WS2_STAGES], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const uint32_t rank = cluster_ctarank();                  // 0 = leader (issues the MMAs), 1 = peer
    const int64_t cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int64_t m_tiles = (M + 2 * BM - 1) / (2 * BM);      // 256-row tiles
    const int64_t n_tiles = m_tiles * n_col_tiles;            // tile id = m * n_col_tiles + nt  (nt fastest)
    const int64_t my_tiles = (n_tiles > cluster_id) ? (n_tiles - cluster_id + n_clusters - 1) / n_clusters : 0;
    const int64_t n_steps = my_tiles * n_kb;

    if (tid == 0) {
        for (int s = 0; s < WS2_STAGES; ++s) {
            mbar_init(&full_a[s], 8);                         // leader: 4 local + 4 remote producer warps
            mbar_init(&full_b[s], rank == 0 ? 2 : 1);         // leader: own expect_tx arrive + the peer's forward
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 8);                      // leader: epilogue warps of both CTAs
        }
        fence_mbar_init();
    }
    if (warp == 4) tmem_alloc2(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                       // both CTAs' barriers are initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp < 4) {
        // ---------------- A producers ----------------------------------------------------------------
        const uint32_t lda32 = uint32_t(lda);
        auto load_step = [&](int64_t step, float (&xr)[32]) {
            const int64_t t = cluster_id + (step / n_kb) * n_clusters;
            const int64_t m0 = (t / n_col_tiles) * (2 * BM) + int64_t(rank) * BM;
            const int kb = int(step % n_kb);
            const int gk = kb * BK + lane;
            if (kb == 0 && t + n_clusters < n_tiles) {
                // next tile's rows -> L2
                const int64_t m1 = ((t + n_clusters) / n_col_tiles) * (2 * BM) + int64_t(rank) * BM;
                if (m1 < M) {
                    const int64_t m2 = (m1 + BM < M) ? m1 + BM : M;
                    const char* pb = reinterpret_cast<const char*>(A + m1 * lda);
                    const int64_t nbytes = (m2 - m1) * lda * int64_t(sizeof(float));
                    for (int64_t off = int64_t(warp * 32 + lane) * 128; off < nbytes; off += 128 * 128)
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(pb + off));
                }
            }
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
        const uint32_t smem_a = smem_u32(smem) + uint32_t(warp) * 4096u;
        uint32_t full_a_leader[WS2_STAGES];
#pragma unroll
        for (int s = 0; s < WS2_STAGES; ++s) full_a_leader[s] = map_to_cta(smem_u32(&full_a[s]), 0);
        auto store_step = [&](int64_t step, const float (&xr)[32]) {
            const int s = int(step % WS2_STAGES);
            const int64_t u = step / WS2_STAGES;
            if (u > 0) mbar_wait(&empty[s], uint32_t((u - 1) & 1));   // MMAs that read this stage have retired
            const uint32_t a_hi = smem_a + uint32_t(s) * WS2_STAGE;
            uint32_t lp[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) lp[j] = a_hi + ((uint32_t((lane >> 2) ^ j)) << 4) + (uint32_t(lane & 3) << 2);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                float h, l;
                split_tf32(xr[i], h, l);
                const uint32_t a = lp[i & 7] + uint32_t((i >> 3) * 1024 + (i & 7) * 128);
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(h) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + WS2_A_PART), "f"(l) : "memory");
            }
            fence_proxy_async();
            __syncwarp();                                  // every lane's stores + proxy fence precede the arrive
            if (lane == 0) mbar_arrive_cluster(s == 0 ? full_a_leader[0] : s == 1 ? full_a_leader[1] : full_a_leader[2]);
        };
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
        // ---------------- MMA issue: leader CTA only ---------------------------------------------------
        if (rank == 0) {
            constexpr uint32_t IDESC = make_idesc(2 * BM, WS_BN, 0, 0);
            for (int64_t step = 0; step < n_steps; ++step) {
                const int64_t j = step / n_kb;
                const int kb = int(step % n_kb);
                const int s = int(step % WS2_STAGES);
                const uint32_t par = uint32_t((step / WS2_STAGES) & 1);
                const int buf = int(j & 1);
                if (kb == 0 && (j >> 1) > 0) {
                    mbar_wait_cluster(&acc_empty[buf], uint32_t(((j >> 1) - 1) & 1));
                    tc_fence_after();
                }
                mbar_wait_cluster(&full_a[s], par);
                mbar_wait_cluster(&full_b[s], par);
                tc_fence_after();
                const uint32_t a_hi = smem_u32(smem + s * WS2_STAGE), a_lo = a_hi + WS2_A_PART;
                const uint32_t b_hi = a_hi + 2 * WS2_A_PART, b_lo = b_hi + WS2_B_PART;
                const uint32_t d = tmem_base + uint32_t(buf * WS_BN);
                const int ksteps = min(BK / UK, (Kd - kb * BK + UK - 1) / UK);
                if (elect_one()) {
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint32_t ko = ks * UK * 4;
                        const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                        const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                        umma2_tf32(d, dah, dbh, IDESC, (kb | ks) ? 1u : 0u);
                        if (!FAST) {
                            umma2_tf32(d, dal, dbh, IDESC, 1u);
                            umma2_tf32(d, dah, dbl, IDESC, 1u);
                        }
                    }
                    umma2_commit_both(&empty[s]);
                    if (kb == n_kb - 1) umma2_commit_both(&acc_full[buf]);
                }
                __syncwarp();
            }
        }
    } else if (warp == 9) {
        // ---------------- B producer: this CTA's half (128 weight rows) of each k-block image -----------
        for (int64_t step = 0; step < n_steps; ++step) {
            const int64_t t = cluster_id + (step / n_kb) * n_clusters;
            const int kb = int(step % n_kb), nt = int(t % n_col_tiles);
            const int s = int(step % WS2_STAGES);
            const int64_t u = step / WS2_STAGES;
            if (u > 0) mbar_wait(&empty[s], uint32_t((u - 1) & 1));
            uint8_t* sB = smem + s * WS2_STAGE + 2 * WS2_A_PART;
            // image = [hi: 256 rows x 128 B][lo: 256 rows x 128 B]; rows 128*rank.. are a contiguous 16 KB block
            const float* img = b_img + (size_t(nt) * n_kb + kb) * 2 * (size_t(WS_BN) * BK) + size_t(rank) * (128 * BK);
            if (elect_one()) {
                mbar_expect_tx(&full_b[s], (FAST ? 1 : 2) * WS2_B_PART);
                bulk_g2s(sB, img, WS2_B_PART, &full_b[s]);
                if (!FAST) bulk_g2s(sB + WS2_B_PART, img + size_t(WS_BN) * BK, WS2_B_PART, &full_b[s]);
            }
            __syncwarp();
        }
    } else if (warp == 10) {
        // ---------------- peer: tell the leader when this CTA's half of B has landed ---------------------
        if (rank == 1) {
            for (int64_t step = 0; step < n_steps; ++step) {
                const int s = int(step % WS2_STAGES);
                mbar_wait(&full_b[s], uint32_t((step / WS2_STAGES) & 1));
                if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&full_b[s]), 0));
                __syncwarp();
            }
        }
    } else {
        // ---------------- epilogue (warps 5..8 -> TMEM lane quadrants 1,2,3,0) ---------------------------
        const int quad = warp & 3;
        float* stg = reinterpret_cast<float*>(smem + WS2_STAGES * WS2_STAGE) + (warp - 5) * (32 * WS_STG_LD);
        const uint32_t acc_empty_leader[2] = {map_to_cta(smem_u32(&acc_empty[0]), 0), map_to_cta(smem_u32(&acc_empty[1]), 0)};
        int64_t j = 0;
        for (int64_t t = cluster_id; t < n_tiles; t += n_clusters, ++j) {
            const int64_t m0 = (t / n_col_tiles) * (2 * BM) + int64_t(rank) * BM;
            const int nt = int(t % n_col_tiles);
            const int buf = int(j & 1);
            mbar_wait(&acc_full[buf], uint32_t((j >> 1) & 1));
            tc_fence_after();
            const int64_t row = m0 + quad * 32 + lane;
            float ps = 0.f, pd = 0.f;
#pragma unroll 1
            for (int ch = 0; ch < WS_BN / 32; ++ch) {
                uint32_t v[32];
                tmem_ld32(tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(buf * WS_BN + ch * 32), v);
                const int col0 = nt * WS_BN + ch * 32;
#pragma unroll
                for (int c = 0; c < 32; c += 4) {
                    const float4 as4 = __ldg(reinterpret_cast<const float4*>(att_src + col0 + c));
                    const float4 ad4 = __ldg(reinterpret_cast<const float4*>(att_dst + col0 + c));
                    ps = fmaf(__uint_as_float(v[c]), as4.x, ps); pd = fmaf(__uint_as_float(v[c]), ad4.x, pd);
                    ps = fmaf(__uint_as_float(v[c + 1]), as4.y, ps); pd = fmaf(__uint_as_float(v[c + 1]), ad4.y, pd);
                    ps = fmaf(__uint_as_float(v[c + 2]), as4.z, ps); pd = fmaf(__uint_as_float(v[c + 2]), ad4.z, pd);
                    ps = fmaf(__uint_as_float(v[c + 3]), as4.w, ps); pd = fmaf(__uint_as_float(v[c + 3]), ad4.w, pd);
                }
                if ((ch & (HC / 32 - 1)) == HC / 32 - 1) {      // HC/32 32-column chunks per head
                    if (row < M) {
                        const int h = col0 / HC;
                        a_src[row * H + h] = ps;
                        a_dst[row * H + h] = pd;
                    }
                    ps = pd = 0.f;
                }
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
                        if (OUT_BF16) {
                            __nv_bfloat162 lo2 = __floats2bfloat162_rn(o.x, o.y), hi2 = __floats2bfloat162_rn(o.z, o.w);
                            uint2 pk;
                            pk.x = *reinterpret_cast<uint32_t*>(&lo2);
                            pk.y = *reinterpret_cast<uint32_t*>(&hi2);
                            *reinterpret_cast<uint2*>(Cb + gm * ldc + col0 + cq) = pk;
                        } else {
                            *reinterpret_cast<float4*>(Cf + gm * ldc + col0 + cq) = o;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_empty_leader[buf]);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                  // no CTA leaves (or frees TMEM) while its peer may still signal it
    if (warp == 4) {
        __syncwarp();
        tmem_dealloc2(tmem_base, 512);
    }
}

}  // namespace tc
}  // namespace gnnfd
