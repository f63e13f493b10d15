// Input-space formulation of the GAT layer (concat = False, H = 8, C = 64; gradient w.r.t. x at K = 64 only).
//
// PyG's GATConv projects first (xw = x W^T, [N, H*C]) and aggregates 2 KB projected rows per edge.  When the input
// width K is smaller than H*C (166 vs 512 for the reference's first layer, src/models/gat.py:39) the same layer is
//     Z[i,h,:]  = sum_{j->i} alpha[e,h] * x[j,:]                       (per-edge gather: K*4 bytes instead of 2 KB)
//     out[i,c]  = (1/H) sum_{h,k} Z[i,h,k] * W[h*C+c,k] + bias[c]      (one [n, H*K] x [H*K, C] GEMM on the tensor cores)
//     a_src[n,h] = x[n,:] . (W_h^T att_src[h]),  a_dst likewise       (logits straight from x)
// and the backward needs no projected features either:
//     Gd[i,h,:] = (1/H) W_h^T dO[i]                                    ([n, C] x [C, H*K] GEMM)
//     d_alpha[e,h] = Gd[i,h,:] . x[j,:]      -> softmax / LeakyReLU backward -> dz, da_dst, da_src = sum_e dz
//     dW[h*C+c,k] = (1/H) sum_i dO[i,c] Z[i,h,k] + att_src[h,c] (da_src^T x)[h,k] + att_dst[h,c] (da_dst^T x)[h,k]
// Across GPUs (destination-range partition, x replicated) this removes the redundant projection of every referenced
// source row and the exchange of per-edge gradients: only [N,H] logits / logit gradients cross NVLink.
//
// Z is written ONCE, by the aggregation kernel, directly in the layout the tensor cores read: per 128-row tile and per
// 64-feature k-block two 16 KB planes (fp16 "hi" and fp16 "lo" of the power-of-two scaled value, hi + lo carries 22
// mantissa bits), each plane the canonical 128B-swizzled shared-memory image, so the GEMMs fetch a k-block with ONE
// cp.async.bulk and need no operand-staging warps.  The same image is a K-major operand (rows = nodes, out = Z W_r) and
// an MN-major operand (rows = features, dW = Z^T dO): the swizzle atom (8 rows x 128 B) is identical for both.
#pragma once
#include <cuda_fp16.h>

#include "gat_stream.cuh"

namespace gnnfd {
namespace in {

constexpr int H = 8, C = 64;
constexpr int MAX_K = 192;               // 48 float4s per row at most: 12 per lane quarter
constexpr int TILE = 128;                // rows (nodes) per image tile
constexpr int PLANE = TILE * 128;        // 16 KB: one fp16 plane of one k-block (64 features) of one tile
constexpr int KBLOCK = 2 * PLANE;        // hi plane then lo plane

struct GI { static constexpr int H = in::H, C = in::C; };   // head geometry for the helpers shared with the projected-feature kernels

struct Dims {
    int K, KP, F, NKB;
    __host__ __device__ explicit Dims(int k) : K(k), KP((k + 7) & ~7), F(H * ((k + 7) & ~7)), NKB((k + 7) >> 3) {}
};

// byte offset of (row r of the tile, element e of the k-block) inside one 128B-swizzled plane
__host__ __device__ __forceinline__ uint32_t plane_off(int r, int e)
{
    return uint32_t(r >> 3) * 1024u + uint32_t(r & 7) * 128u + ((uint32_t(e >> 3) ^ uint32_t(r & 7)) << 4) + uint32_t(e & 7) * 2u;
}

// power-of-two scale s with m*s in [2^11, 2^12): fp16 keeps 11 bits, leaves x16 headroom below 65504 (attention dropout
// rescales by 1/(1-p)) and 26 bits of range above the smallest normal
__host__ __device__ __forceinline__ float pow2_scale(float m)
{
#ifdef __CUDA_ARCH__
    const uint32_t b = __float_as_uint(m);
#else
    uint32_t b;
    memcpy(&b, &m, 4);
#endif
    const int e = int((b >> 23) & 0xffu) - 127;
    if (!(m > 0.f) || e < -100 || e > 100) return 1.f;
    const uint32_t sb = uint32_t(127 + 11 - e) << 23;
#ifdef __CUDA_ARCH__
    return __uint_as_float(sb);
#else
    float s;
    memcpy(&s, &sb, 4);
    return s;
#endif
}

// v (already scaled) -> fp16 hi + fp16 lo, hi + lo = v to 22 bits (the fp32 residual is exact)
__device__ __forceinline__ void split_h2(float v0, float v1, __half2& hi, __half2& lo)
{
    hi = __floats2half2_rn(v0, v1);
    const float2 hf = __half22float2(hi);
    lo = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
}

// Device-resident per-call constants and operand images ("prep" buffer), built by gnnfd_in_prepare:
//   float scal[8]      : [0] sx (scale of x / Z), [1] sw (scale of W), [2] 1/(sx*sw*H), [3] 1/sx
//   W image for out = Z W_r   : NKB k-blocks x (hi [64 rows x 128 B] | lo), rows = c, K-major, scaled by sw
//   W image for Gd = dO W_r^T : fp16 hi/lo, n-tiles of 128 features x 64 c (K-major in c), scaled by sw (1/H in the epilogue)
//   u [2H][KP]         : W_h^T att_src[h] (rows 0..H-1) and W_h^T att_dst[h] (rows H..2H-1)
constexpr size_t PREP_SCAL_BYTES = 256;
__host__ __device__ inline size_t prep_wout_bytes(const Dims& d) { return size_t(d.NKB) * 16384; }
__host__ __device__ inline size_t prep_wgd_bytes(const Dims& d) { return size_t((d.F + 127) / 128) * 2 /*hi, lo*/ * (128 * 128); }
__host__ __device__ inline size_t prep_u_bytes(const Dims& d) { return size_t(2 * H) * d.KP * sizeof(float); }
__host__ __device__ inline size_t prep_off_wout(const Dims&) { return 1024; }
__host__ __device__ inline size_t prep_off_wgd(const Dims& d) { return 1024 + ((prep_wout_bytes(d) + 1023) & ~size_t(1023)); }
__host__ __device__ inline size_t prep_off_u(const Dims& d) { return prep_off_wgd(d) + ((prep_wgd_bytes(d) + 1023) & ~size_t(1023)); }
__host__ __device__ inline size_t prep_bytes(const Dims& d) { return prep_off_u(d) + ((prep_u_bytes(d) + 1023) & ~size_t(1023)) + 1024; }

inline size_t zimg_bytes(int64_t n_rows, const Dims& d) { return size_t((n_rows + TILE - 1) / TILE) * d.NKB * KBLOCK; }

// Where a kernel's finished rows also go (header section 7): mode 0 = nowhere else; 1 = row (row_off + r) of the same buffer
// on every peer (one 16-byte store per peer over NVLink); 2 = one multimem.st to the multicast mapping (the NVSwitch
// replicates it to every rank)
struct PeerRows {
    int mode, n;
    int64_t row_off;
    float* ptr[GNNFD_MAX_PEERS];
    float* mc;
};
__device__ __forceinline__ void multimem_st_v4(float* p, float4 v)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// checks the caller's peer table before anything is launched and fills `pr` (mode 1 or 2)
inline int peer_rows_from(const gnnfd_peers_t* p, int64_t row_offset, int use_multicast, const char* who, PeerRows& pr)
{
    GNNFD_REQUIRE(p && row_offset >= 0, GNNFD_ERR_ARG, "%s: NULL peer table or negative row offset", who);
    GNNFD_REQUIRE(p->n_peers >= 1 && p->n_peers <= GNNFD_MAX_PEERS, GNNFD_ERR_ARG, "%s: 1..%d peers", who, GNNFD_MAX_PEERS);
    GNNFD_REQUIRE(!use_multicast || p->multicast, GNNFD_ERR_ARG, "%s: no multicast mapping given", who);
    pr = PeerRows{};
    pr.mode = use_multicast ? 2 : 1;
    pr.n = p->n_peers;
    pr.row_off = row_offset;
    pr.mc = reinterpret_cast<float*>(p->multicast);
    for (int g = 0; g < pr.n; ++g) {
        GNNFD_REQUIRE(p->ptr[g] && (reinterpret_cast<uintptr_t>(p->ptr[g]) & 15) == 0, GNNFD_ERR_ARG,
                      "%s: peer buffer %d NULL or not 16-byte aligned", who, g);
        pr.ptr[g] = reinterpret_cast<float*>(p->ptr[g]);
    }
    return GNNFD_OK;
}

}  // namespace in
}  // namespace gnnfd

namespace gnnfd {
namespace in {

// ---- lane geometry of the logits kernel and of the backward edge kernel -------------------------------------------------
// lane = (head h = lane >> 2, quarter q = lane & 3).  A staged x row is KP floats = n4 float4s; lane (h, q) owns the
// float4s 4*i + q (i = 0, 1, ...) of the row for ITS head: 44 accumulators (forward) / 44 Gd values (backward) for
// K = 166.  Per edge and lane: ceil(n4/4) conflict-free 128-bit shared loads (the four q-lanes read 64 contiguous bytes,
// the eight heads read the same addresses = broadcast) and 4 FMAs per load; the backward's dot product is finished by
// TWO shuffles over the lane's quad; everything per-head (softmax state, weights, scales) is a scalar per lane.
// N4 > 0: compile-time row width (no per-load predicate except the tail); N4 = 0: run-time n4 <= 48.
template <int N4>
struct RowGeo {
    static constexpr int NI = N4 > 0 ? (N4 + 3) / 4 : MAX_K / 16;
    __device__ static __forceinline__ bool valid(int i, int q, int n4) { return N4 > 0 ? (4 * i + q < N4) : (4 * i + q < n4); }
};

// Forward aggregation: lane = FEATURE group.  Lane l owns the float2s l + 32*i (i = 0, 1, 2) of the staged row and keeps the
// accumulators of ALL heads for them (8 x 3 float2 = 48 fp32).  Per edge the warp then reads the 672-byte row exactly once
// (3 conflict-free LDS.64 = 6 shared-memory wavefronts) plus the 8 weights (broadcast), against 44 wavefronts when every head
// re-reads the row -- the (head, quarter) layout had the forward at 81 % of the shared-memory pipe (ncu, round 2).
template <int N4>
struct FeatGeo {
    static constexpr int NI = N4 > 0 ? (2 * N4 + 31) / 32 : MAX_K / 64;       // float2s per lane
    __device__ static __forceinline__ bool valid(int i, int lane, int n2) { return N4 > 0 ? (lane + 32 * i < 2 * N4) : (lane + 32 * i < n2); }
};
__device__ __forceinline__ float2 lds64(uint32_t addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}

// ---- per-warp ring of staged x rows ------------------------------------------------------------------------------
// Rows must be 16-byte aligned and zero-padded to KP floats (ldx % 4 == 0, ldx >= KP: gnnfd_in_pad_x builds such a copy
// of an unaligned x): lane 0 hands a whole row to the bulk-copy engine (cp.async.bulk global->shared, mbarrier
// complete_tx).  Per-warp layout:  [R slots of KP*4 bytes][p_s: 2 x 32 x H floats][j_s: 2 x 32 ints][R+1 mbarriers][extra]
constexpr int IN_WARPS = 4;
constexpr int IN_THREADS = IN_WARPS * 32;
constexpr int IN_R_MAX = 8;                                // ring slots per warp: 8 (forward) or 4 (backward), a power of two
constexpr int IN_P_BYTES = 2 * 32 * H * 4, IN_J_BYTES = 2 * 32 * 4, IN_BAR_BYTES = ((IN_R_MAX + 1) * 8 + 15) / 16 * 16;

__host__ __device__ inline int in_warp_bytes(int KP, int extra, int slots = IN_R_MAX)
{
    return (slots * KP * 4 + IN_P_BYTES + IN_J_BYTES + IN_BAR_BYTES + extra + 127) / 128 * 128;
}

__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        if (++spins > (1u << 26)) __trap();   // a protocol bug must not hang the GPU
    }
}
__device__ __forceinline__ void bulk_g2s_u32(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
                 "l"(gsrc), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// packed fp32x2 FMA (sm_100 FFMA2): two FMAs per issue slot, each component rounded exactly like fmaf
__device__ __forceinline__ void ffma2_bcast(float& a0, float& a1, float w, float v0, float v1)     // a += w * v
{
    unsigned long long a, b, c;
    asm("mov.b64 %0, {%1, %1};" : "=l"(a) : "f"(w));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(v0), "f"(v1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(a0), "f"(a1));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(c));
}
__device__ __forceinline__ void ffma2_vec(float& a0, float& a1, float g0, float g1, float v0, float v1)   // a += g * v
{
    unsigned long long a, b, c;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(g0), "f"(g1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(v0), "f"(v1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(a0), "f"(a1));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(c));
}

template <int R_>
struct InRingT {
    static constexpr int IN_R = R_;            // any count <= IN_R_MAX (a power of two costs one instruction less per wait)
    uint32_t ring_u32, full_u32, slot;   // shared-space addresses / bytes per slot
    uint8_t* extra;
    float* p_s;      // [2][32*H]
    int* j_s;        // [2][32]
    int issued = 0, consumed = 0;
    const float* x;
    int64_t ldx;

    __device__ __forceinline__ void init(uint8_t* base, const float* x_, int64_t ldx_, int KP, int lane)
    {
        slot = uint32_t(KP) * 4u;
        ring_u32 = st_smem_u32(base);
        p_s = reinterpret_cast<float*>(base + IN_R * slot);
        j_s = reinterpret_cast<int*>(base + IN_R * slot + IN_P_BYTES);
        uint64_t* full = reinterpret_cast<uint64_t*>(base + IN_R * slot + IN_P_BYTES + IN_J_BYTES);
        full_u32 = st_smem_u32(full);
        extra = base + IN_R * slot + IN_P_BYTES + IN_J_BYTES + IN_BAR_BYTES;
        x = x_;
        ldx = ldx_;
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i <= IN_R; ++i) st_mbar_init(&full[i], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }
    __device__ __forceinline__ uint32_t spare_bar() const { return full_u32 + 8u * IN_R; }   // for kernel-specific use
    __device__ __forceinline__ bool has_room() const { return issued - consumed < IN_R; }
    __device__ __forceinline__ void issue(int j, int lane)
    {
        if (lane == 0) {
            const uint32_t s = uint32_t(issued) % uint32_t(IN_R);
            const uint32_t bar = full_u32 + 8u * s;
            mbar_expect_tx_u32(bar, slot);
            bulk_g2s_u32(ring_u32 + s * slot, x + int64_t(j) * ldx, slot, bar);
        }
        ++issued;
    }
    // rows j[0..cnt) in ONE divergent block: lane r < cnt hands row j[r] to the copy engine (cnt <= IN_R)
    __device__ __forceinline__ void issue_many(const int* j, int cnt, int lane)
    {
        if (lane < cnt) {
            const uint32_t n = uint32_t(issued + lane);
            const uint32_t s = n % uint32_t(IN_R);
            const uint32_t bar = full_u32 + 8u * s;
            mbar_expect_tx_u32(bar, slot);
            bulk_g2s_u32(ring_u32 + s * slot, x + int64_t(j[lane]) * ldx, slot, bar);
        }
        issued += cnt;
    }
    // wait for the oldest in-flight row; returns its shared-space address
    __device__ __forceinline__ uint32_t front() { return front_at(0); }
    // ... for the r-th oldest
    __device__ __forceinline__ uint32_t front_at(int r)
    {
        const uint32_t n = uint32_t(consumed + r);
        const uint32_t s = n % uint32_t(IN_R);
        mbar_wait_u32(full_u32 + 8u * s, (n / uint32_t(IN_R)) & 1u);
        return ring_u32 + s * slot;
    }
    __device__ __forceinline__ void pop()
    {
        __syncwarp();
        ++consumed;
    }
    // the cnt oldest rows have been consumed by every lane (their loads fed FMAs that have issued)
    __device__ __forceinline__ void pop_many(int cnt)
    {
        __syncwarp();
        consumed += cnt;
    }
    __device__ __forceinline__ int room() const { return IN_R - (issued - consumed); }
};
using InRing = InRingT<8>;

// arr[h] with a run-time h, without dynamic register indexing
__device__ __forceinline__ float pick_head(const float (&arr)[H], int h)
{
    float r = arr[0];
#pragma unroll
    for (int k = 1; k < H; ++k) r = (h == k) ? arr[k] : r;
    return r;
}

}  // namespace in
}  // namespace gnnfd
