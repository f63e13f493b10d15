// Pipelined dW partials on the tensor cores:  P[slab][o][k] = sum_{n in slab} dxw[n][o] * x[n][k]   (3xTF32)
//
// Staging the operands is bound by the load/store pipe, so ONE persistent CTA per SM owns 256 output rows (two
// M=128 accumulators in TMEM that share the B = x operand): the x tile is staged once per 256 rows rather than once
// per 128, and the staging of node block i+1.. overlaps the MMAs of block i through a three-stage mbarrier ring:
//   warps 0-7   producers: node group kq = warp/2 (4 nodes) of each 16-node stage; even warps stage the A operand
//               (dxw rows, both o-tiles, float4), odd warps the B operand (x rows, float2 pairs when aligned);
//               the global loads of the next stage are in flight while the current one is split and stored
//   warp  8     MMA issuer (one elected lane): 2 k-steps x 3 passes x 2 o-tiles per stage; tcgen05.commit frees
//               the stage; every FLUSH stages it hands both accumulators to the flush warps
//   warps 9-12  flush: TMEM -> registers -> smem transpose -> coalesced fire-and-forget RED.ADD into this CTA's
//               private fp32 partial (the tensor core accumulates round-toward-zero, so chains are kept short)
// Operands are MN-major (the reduction runs over nodes): SWIZZLE_128B_BASE32B atoms of 4 nodes x 32 elements.
#pragma once

namespace gnnfd {
namespace tc {

constexpr int DW2_BK = 16;                                  // nodes per stage
constexpr int DW2_STAGES = 3;
constexpr int DW2_THREADS = 13 * 32;
constexpr int DW2_FLUSH = 32;                               // stages (512 nodes) between accumulator drains
constexpr uint32_t DW2_A_PART = 4 * 4 * 512;                // 8 KB: one o-tile, hi or lo: 4 node groups x 4 o groups
constexpr int DW2_STG_LD = 36;
template <int NG> constexpr uint32_t dw2_b_part() { return 4u * NG * 512u; }
template <int NG> constexpr uint32_t dw2_stage() { return 4u * DW2_A_PART + 2u * dw2_b_part<NG>(); }
template <int NG> constexpr size_t dw2_smem() { return DW2_STAGES * dw2_stage<NG>() + 4 * 32 * DW2_STG_LD * 4 + 1024; }

template <int NG, bool VEC2>
__global__ void __launch_bounds__(DW2_THREADS, 1)
dw_tc2(const float* __restrict__ dxw, int D, const float* __restrict__ x, int64_t ldx, int64_t N, int K, int kpad,
       int64_t rows_per_slab, float* __restrict__ P)
{
    constexpr uint32_t B_PART = dw2_b_part<NG>();
    constexpr uint32_t STAGE = dw2_stage<NG>();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full[DW2_STAGES], empty[DW2_STAGES], acc_full, acc_empty;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int o0 = blockIdx.x * 256;                          // first of this CTA's 256 output rows
    const int64_t nb = int64_t(blockIdx.y) * rows_per_slab;
    const int64_t ne = (nb + rows_per_slab < N) ? nb + rows_per_slab : N;
    const int n_kb = (ne > nb) ? int((ne - nb + DW2_BK - 1) / DW2_BK) : 0;
    const int n_flush = (n_kb + DW2_FLUSH - 1) / DW2_FLUSH;

    if (tid == 0) {
        for (int s = 0; s < DW2_STAGES; ++s) {
            mbar_init(&full[s], 8);
            mbar_init(&empty[s], 1);
        }
        mbar_init(&acc_full, 1);
        mbar_init(&acc_empty, 4);
        fence_mbar_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;

    if (warp < 8) {
        // ---------------- producers --------------------------------------------------------------------
        const uint32_t kq = uint32_t(warp >> 1);
        const bool is_a = (warp & 1) == 0;
        const uint32_t stage0 = smem_u32(smem);
        if (is_a) {
            float4 cur[4][2], nxt[4][2];
            auto load = [&](int kb, float4 (&v)[4][2]) {
#pragma unroll
                for (int jr = 0; jr < 4; ++jr) {
                    const int64_t n = nb + int64_t(kb) * DW2_BK + kq * 4 + jr;
                    const bool ok = n < ne;
#pragma unroll
                    for (int T = 0; T < 2; ++T)
                        v[jr][T] = ok ? __ldg(reinterpret_cast<const float4*>(dxw + n * D + o0 + T * 128) + lane)
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            auto store = [&](int kb, const float4 (&v)[4][2]) {
                const int s = kb % DW2_STAGES;
                if (kb >= DW2_STAGES) mbar_wait(&empty[s], uint32_t((kb / DW2_STAGES - 1) & 1));
                const uint32_t base = stage0 + uint32_t(s) * STAGE + (kq * 4u + uint32_t(lane >> 3)) * 512u + (uint32_t(lane & 1) << 4);
#pragma unroll
                for (int jr = 0; jr < 4; ++jr) {
                    const uint32_t off = base + uint32_t(jr) * 128u + ((uint32_t((lane & 7) >> 1) ^ uint32_t(jr)) << 5);
#pragma unroll
                    for (int T = 0; T < 2; ++T) {
                        float4 h, l;
                        split_tf32(v[jr][T].x, h.x, l.x); split_tf32(v[jr][T].y, h.y, l.y);
                        split_tf32(v[jr][T].z, h.z, l.z); split_tf32(v[jr][T].w, h.w, l.w);
                        const uint32_t a = off + uint32_t(T) * 2u * DW2_A_PART;       // [T0 hi][T0 lo][T1 hi][T1 lo]
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(h.x), "f"(h.y), "f"(h.z), "f"(h.w) : "memory");
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a + DW2_A_PART), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[s]);
            };
            if (n_kb > 0) load(0, cur);
            for (int kb = 0; kb < n_kb; kb += 2) {
                if (kb + 1 < n_kb) load(kb + 1, nxt);
                store(kb, cur);
                if (kb + 1 < n_kb) {
                    if (kb + 2 < n_kb) load(kb + 2, cur);
                    store(kb + 1, nxt);
                }
            }
        } else {
            float cur[4][NG], nxt[4][NG];
            auto load = [&](int kb, float (&v)[4][NG]) {
#pragma unroll
                for (int jr = 0; jr < 4; ++jr) {
                    const int64_t n = nb + int64_t(kb) * DW2_BK + kq * 4 + jr;
                    const bool ok = n < ne;
                    if (VEC2) {
#pragma unroll
                        for (int t = 0; t < NG / 2; ++t) {
                            const int kf = 2 * lane + 64 * t;     // K is even: a pair is never split by K
                            const float2 p = (ok && kf < K) ? __ldg(reinterpret_cast<const float2*>(x + n * ldx + kf)) : make_float2(0.f, 0.f);
                            v[jr][2 * t] = p.x;
                            v[jr][2 * t + 1] = p.y;
                        }
                    } else {
#pragma unroll
                        for (int t = 0; t < NG; ++t) {
                            const int kf = lane + 32 * t;
                            v[jr][t] = (ok && kf < K) ? __ldg(x + n * ldx + kf) : 0.f;
                        }
                    }
                }
            };
            auto store = [&](int kb, const float (&v)[4][NG]) {
                const int s = kb % DW2_STAGES;
                if (kb >= DW2_STAGES) mbar_wait(&empty[s], uint32_t((kb / DW2_STAGES - 1) & 1));
                const uint32_t b_hi = stage0 + uint32_t(s) * STAGE + 4u * DW2_A_PART + kq * uint32_t(NG) * 512u;
#pragma unroll
                for (int jr = 0; jr < 4; ++jr) {
                    if (VEC2) {
#pragma unroll
                        for (int t = 0; t < NG / 2; ++t) {
                            const uint32_t grp = uint32_t(2 * t + (lane >> 4)), fi = uint32_t((2 * lane) & 31);
                            const uint32_t a = b_hi + grp * 512u + uint32_t(jr) * 128u + (((fi >> 3) ^ uint32_t(jr)) << 5) + (fi & 7u) * 4u;
                            float2 h, l;
                            split_tf32(v[jr][2 * t], h.x, l.x);
                            split_tf32(v[jr][2 * t + 1], h.y, l.y);
                            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(h.x), "f"(h.y) : "memory");
                            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a + B_PART), "f"(l.x), "f"(l.y) : "memory");
                        }
                    } else {
#pragma unroll
                        for (int t = 0; t < NG; ++t) {
                            const uint32_t a = b_hi + uint32_t(t) * 512u + uint32_t(jr) * 128u +
                                               ((uint32_t(lane >> 3) ^ uint32_t(jr)) << 5) + uint32_t(lane & 7) * 4u;
                            float h, l;
                            split_tf32(v[jr][t], h, l);
                            asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(h) : "memory");
                            asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + B_PART), "f"(l) : "memory");
                        }
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[s]);
            };
            if (n_kb > 0) load(0, cur);
            for (int kb = 0; kb < n_kb; kb += 2) {
                if (kb + 1 < n_kb) load(kb + 1, nxt);
                store(kb, cur);
                if (kb + 1 < n_kb) {
                    if (kb + 2 < n_kb) load(kb + 2, cur);
                    store(kb + 1, nxt);
                }
            }
        }
    } else if (warp == 8) {
        // ---------------- MMA issue ----------------------------------------------------------------------
        const uint32_t idesc = make_idesc(BM, kpad, 1, 1);
        for (int kb = 0; kb < n_kb; ++kb) {
            const int s = kb % DW2_STAGES;
            const bool restart = (kb % DW2_FLUSH) == 0;
            if (restart && kb > 0) {
                // hand the accumulators to the flush warps, wait until they are drained
                if (elect_one()) umma_commit(&acc_full);
                __syncwarp();
                mbar_wait(&acc_empty, uint32_t((kb / DW2_FLUSH - 1) & 1));
                tc_fence_after();
            }
            mbar_wait(&full[s], uint32_t((kb / DW2_STAGES) & 1));
            tc_fence_after();
            const uint32_t st = smem_u32(smem) + uint32_t(s) * STAGE;
            const uint32_t b_hi = st + 4u * DW2_A_PART, b_lo = b_hi + B_PART;
            if (elect_one()) {
#pragma unroll
                for (int kg = 0; kg < 2; ++kg) {               // k-step = 8 nodes = two 4-node groups
                    const uint64_t dbh = make_desc(b_hi + kg * NG * 1024, 512, NG * 512, 1);
                    const uint64_t dbl = make_desc(b_lo + kg * NG * 1024, 512, NG * 512, 1);
#pragma unroll
                    for (int T = 0; T < 2; ++T) {
                        const uint32_t a_hi = st + uint32_t(T) * 2u * DW2_A_PART, a_lo = a_hi + DW2_A_PART;
                        const uint64_t dah = make_desc(a_hi + kg * 4096, 512, 2048, 1), dal = make_desc(a_lo + kg * 4096, 512, 2048, 1);
                        const uint32_t d = tmem_d + uint32_t(T * 256);
                        umma_tf32(d, dah, dbh, idesc, (restart && kg == 0) ? 0u : 1u);
                        umma_tf32(d, dal, dbh, idesc, 1u);
                        umma_tf32(d, dah, dbl, idesc, 1u);
                    }
                }
                umma_commit(&empty[s]);
            }
            __syncwarp();
        }
        if (n_kb > 0) {
            if (elect_one()) umma_commit(&acc_full);
            __syncwarp();
        }
    } else {
        // ---------------- flush warps 9..12 -> TMEM lane quadrants 1,2,3,0 ----------------------------------
        const int quad = warp & 3;
        float* Ps = P + int64_t(blockIdx.y) * D * K;
        float* stg = reinterpret_cast<float*>(smem + DW2_STAGES * STAGE) + (warp - 9) * (32 * DW2_STG_LD);
        for (int f = 0; f < n_flush; ++f) {
            mbar_wait(&acc_full, uint32_t(f & 1));
            tc_fence_after();
#pragma unroll 1
            for (int T = 0; T < 2; ++T) {
#pragma unroll 1
                for (int ch = 0; ch < NG; ++ch) {
                    uint32_t v[32];
                    tmem_ld32(tmem_d + (uint32_t(quad * 32) << 16) + uint32_t(T * 256 + ch * 32), v);
                    __syncwarp();
#pragma unroll
                    for (int c = 0; c < 32; c += 4)
                        *reinterpret_cast<float4*>(stg + lane * DW2_STG_LD + c) =
                            make_float4(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), __uint_as_float(v[c + 2]),
                                        __uint_as_float(v[c + 3]));
                    __syncwarp();
                    const int kf = ch * 32 + lane;
                    if (kf < K) {
                        float* dst = Ps + int64_t(o0 + T * 128 + quad * 32) * K + kf;
#pragma unroll 8
                        for (int r = 0; r < 32; ++r) atomicAdd(dst + int64_t(r) * K, stg[r * DW2_STG_LD + lane]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        __syncwarp();
        tmem_dealloc(tmem_d, 512);
    }
}

}  // namespace tc
}  // namespace gnnfd
