// Lane/slot geometry shared by the forward and backward message-passing kernels.
//
// A projected feature row has D = H*C elements.  One warp owns one row; a warp-wide 128-bit load covers
// 32*VW consecutive elements (VW = 4 fp32 / 8 bf16 per lane), so a row is NS = D/(32*VW) "slots" per
// lane, each slot a fully coalesced 512-byte warp transaction.  All VW elements of a slot lie in one
// head; G = C/VW consecutive lanes share a head, HP = 32/G heads are covered by one slot instruction,
// and the head of (slot q, lane l) is q*HP + l/G.
#pragma once
#include "common.cuh"

namespace gnnfd {

template <int H_, int C_, typename XT_>
struct Geo {
    using XT = XT_;
    static constexpr int H = H_, C = C_, D = H_ * C_;
    static constexpr int VW = sizeof(XT_) == 4 ? 4 : 8;
    static constexpr int NS = D / (32 * VW);
    static constexpr int G = C / VW;
    static constexpr int HP = 32 / G;
    static_assert(D % (32 * VW) == 0, "row must be a whole number of warp-wide 128-bit loads");
    static_assert(C % VW == 0 && G >= 1 && G <= 32 && (G & (G - 1)) == 0, "C/VW must be a power of two <= 32");
    static_assert(NS * HP == H, "slots x heads-per-slot must tile the heads");
    static_assert(H % 4 == 0 && H <= 8, "logit vectors are loaded as float4s");
};

// arr[q*HP + sub] with compile-time q and run-time sub, without dynamic register indexing
template <int HP, int N>
__device__ __forceinline__ float pick(const float (&arr)[N], int q, int sub)
{
    float r = arr[q * HP];
#pragma unroll
    for (int k = 1; k < HP; ++k) r = (sub == k) ? arr[q * HP + k] : r;
    return r;
}

template <int H>
__device__ __forceinline__ void load_vecH(const float* __restrict__ p, float (&v)[H])
{
#pragma unroll
    for (int k = 0; k < H / 4; ++k) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p) + k);
        v[4 * k + 0] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
    }
}
template <int H>
__device__ __forceinline__ void store_vecH(float* __restrict__ p, const float (&v)[H])
{
#pragma unroll
    for (int k = 0; k < H / 4; ++k)
        reinterpret_cast<float4*>(p)[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}
// H floats to a 32-byte-aligned address: one 256-bit store for H = 8 (a whole sector per lane), else store_vecH
template <int H>
__device__ __forceinline__ void store_vecH_wide(float* __restrict__ p, const float (&v)[H])
{
    if constexpr (H == 8) {
        asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]),
                     "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                     : "memory");
    } else {
        store_vecH<H>(p, v);
    }
}

// one slot (VW elements) of a feature row, streamed past L1
__device__ __forceinline__ void load_slot(const float* __restrict__ row, int q, int lane, float (&v)[4])
{
    const float4 t = ldg_stream(reinterpret_cast<const float4*>(row) + lane + 32 * q);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load_slot(const __nv_bfloat16* __restrict__ row, int q, int lane, float (&v)[8])
{
    const uint4 t = ldg_stream_u4(reinterpret_cast<const uint4*>(row) + lane + 32 * q);
    v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
    v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
    v[4] = __uint_as_float(t.z << 16); v[5] = __uint_as_float(t.z & 0xffff0000u);
    v[6] = __uint_as_float(t.w << 16); v[7] = __uint_as_float(t.w & 0xffff0000u);
}

// Attention dropout (GATConv(..., dropout=p), src/models/gat.py:39): which (edge, head) coefficients survive.
// Either an explicit keep-mask [E',H] in edge_index' (PyG) order -- parity tests inject one -- or, in training, a
// counter-based RNG keyed on (seed, position in edge_index', head): stateless, so the forward and the backward kernels
// re-derive the SAME bits with no [E',H] tensor and no extra pass.  16 random bits per (edge, head): keep iff bits >= thr,
// thr = floor(p * 65536); the survivors are scaled by 65536 / (65536 - thr) (the exact keep probability).
struct KeepMask {
    const uint8_t* mask;
    uint64_t seed;
    uint32_t thr;
    const uint64_t* seed_src;     // optional device word added to the seed (gnnfd_set_dropout_seed_source): lets a step that
                                  // is replayed from a CUDA graph draw fresh masks -- the graph bumps the word, not the host
    __host__ __device__ KeepMask(const uint8_t* m = nullptr, uint64_t s = 0, uint32_t t = 0, const uint64_t* src = nullptr)
        : mask(m), seed(s), thr(t), seed_src(src) {}
    __host__ __device__ static uint64_t mix(uint64_t z)            // splitmix64 finaliser
    {
        z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
        z ^= z >> 27; z *= 0x94D049BB133111EBull;
        z ^= z >> 31;
        return z;
    }
    // bit h = coefficient (edge at position pos of edge_index', head h) is kept; H <= 8
    __host__ __device__ unsigned bits(int64_t pos, int H) const
    {
        unsigned r = 0;
        if (mask) {
            const uint8_t* kb = mask + pos * H;
            for (int h = 0; h < H; ++h) r |= unsigned(kb[h] != 0) << h;
            return r;
        }
        uint64_t sd = seed;
#ifdef __CUDA_ARCH__
        if (seed_src) sd += __ldg(reinterpret_cast<const unsigned long long*>(seed_src));
#endif
        const uint64_t c = sd + 0x9E3779B97F4A7C15ull * uint64_t(2 * pos + 1);
        const uint64_t w0 = mix(c), w1 = mix(c ^ 0xD1B54A32D192ED03ull);
        for (int h = 0; h < H; ++h) {
            const uint32_t v = uint32_t(((h < 4 ? w0 : w1) >> (16 * (h & 3))) & 0xffffu);
            r |= unsigned(v >= thr) << h;
        }
        return r;
    }
};
extern const uint64_t* g_dropout_seed_src;      // csr_radix.cu; set by gnnfd_set_dropout_seed_source
// host side: the KeepMask and the survivor scale for (explicit mask or NULL, p, seed)
inline KeepMask make_keep(const uint8_t* mask, float p_drop, uint64_t seed, float* scale)
{
    if (!(p_drop > 0.f)) { *scale = 1.f; return KeepMask(); }
    if (mask) { *scale = 1.f / (1.f - p_drop); return KeepMask(mask, 0, 0); }
    uint32_t thr = uint32_t(double(p_drop) * 65536.0);
    if (thr > 65535u) thr = 65535u;
    *scale = 65536.f / float(65536u - thr);
    return KeepMask(nullptr, seed, thr, g_dropout_seed_src);
}

constexpr int ROW_WARPS = 8;                 // warps (rows) per CTA
constexpr int ROW_THREADS = ROW_WARPS * 32;

}  // namespace gnnfd
