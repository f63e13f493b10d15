// (2) projection xw = x @ W^T with the per-head attention-logit epilogue, and the projection backward
// (dW, dx, datt_src, datt_dst, dbias) -- fp32 CUDA-core reference path.
//
// Replaces lin_src(x).view(-1,H,C), (x_src*att_src).sum(-1), (x_dst*att_dst).sum(-1) of PyG's
// GATConv.forward (reference call site src/models/gat.py:80) and their autograd mirror.  This file is the
// exact-fp32 path (GNNFD_GEMM_SIMT): it is what parity at 1e-5 is anchored on and what the tensor-core
// path (project_tc.cu, GNNFD_GEMM_TC) is cross-checked against on the device.
#include "common.cuh"

#include <atomic>

namespace gnnfd {
extern std::atomic<long long> g_launches;

constexpr int GB_M = 64, GB_N = 64, GB_K = 16, G_PAD = 4;

// C[M,Nc] = A[M,Kd] (row-major, lda) * B, B(kd,nc) = Bp[kd*sbk + nc*sbn].
// EPI: 0 = plain store (fp32, ldc); 1 = forward epilogue (xw store fp32/bf16 + a_src/a_dst, needs Ccols==GB_N)
template <bool B_KCONTIG, int EPI, bool OUT_BF16>
__global__ void __launch_bounds__(256)
gemm_simt(const float* __restrict__ A, int64_t lda, const float* __restrict__ Bp, int64_t sbk, int64_t sbn,
          int64_t M, int Nc, int Kd, float* __restrict__ Cf, __nv_bfloat16* __restrict__ Cb, int64_t ldc,
          const float* __restrict__ att_src, const float* __restrict__ att_dst, float* __restrict__ a_src,
          float* __restrict__ a_dst, int H)
{
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t m0 = int64_t(blockIdx.x) * GB_M;
    const int n0 = blockIdx.y * GB_N;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < Kd; k0 += GB_K) {
        // A tile: 64 rows x 16 k, k fastest across threads (contiguous in global)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = (tid >> 4) + 16 * i, kk = tid & 15;
            const int64_t gm = m0 + r;
            const int gk = k0 + kk;
            As[kk][r] = (gm < M && gk < Kd) ? A[gm * lda + gk] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int kk, c;
            if (B_KCONTIG) { kk = tid & 15; c = (tid >> 4) + 16 * i; }
            else           { c = tid & 63;  kk = (tid >> 6) + 4 * i; }
            const int gk = k0 + kk, gn = n0 + c;
            Bs[kk][c] = (gk < Kd && gn < Nc) ? Bp[int64_t(gk) * sbk + int64_t(gn) * sbn] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GB_K; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }

    if (EPI == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t gm = m0 + ty * 4 + i;
            if (gm >= M) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int gn = n0 + tx * 4 + j;
                if (gn < Nc) Cf[gm * ldc + gn] = acc[i][j];
            }
        }
    } else {
        // one head per column tile (C == GB_N): logits are a 64-wide dot product of this tile's rows
        const int h = blockIdx.y;
        float as4[4], ad4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            as4[j] = att_src[n0 + tx * 4 + j];
            ad4[j] = att_dst[n0 + tx * 4 + j];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t gm = m0 + ty * 4 + i;
            float ps = 0.f, pd = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                ps = fmaf(acc[i][j], as4[j], ps);
                pd = fmaf(acc[i][j], ad4[j], pd);
            }
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) {   // the 16 tx lanes of a row are a half-warp
                ps += __shfl_xor_sync(FULL, ps, o);
                pd += __shfl_xor_sync(FULL, pd, o);
            }
            if (gm < M) {
                if (tx == 0) {
                    a_src[gm * H + h] = ps;
                    a_dst[gm * H + h] = pd;
                }
                if (OUT_BF16) {
                    __nv_bfloat162 lo = __floats2bfloat162_rn(acc[i][0], acc[i][1]);
                    __nv_bfloat162 hi = __floats2bfloat162_rn(acc[i][2], acc[i][3]);
                    uint2 v;
                    v.x = *reinterpret_cast<uint32_t*>(&lo);
                    v.y = *reinterpret_cast<uint32_t*>(&hi);
                    *reinterpret_cast<uint2*>(Cb + gm * ldc + n0 + tx * 4) = v;
                } else {
                    *reinterpret_cast<float4*>(Cf + gm * ldc + n0 + tx * 4) =
                        make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                }
            }
        }
    }
}

// dW partials: P[s][m][k] = sum_{n in slice s} dxw[n][m] * x[n][k]     (m < D, k < K)
__global__ void __launch_bounds__(256)
dw_partial(const float* __restrict__ dxw, int64_t D, const float* __restrict__ x, int64_t ldx, int64_t N, int K,
           int64_t rows_per_slice, float* __restrict__ P)
{
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.x * GB_M, c0 = blockIdx.y * GB_N;
    const int64_t nb = int64_t(blockIdx.z) * rows_per_slice;
    const int64_t ne = (nb + rows_per_slice < N) ? nb + rows_per_slice : N;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int64_t n0 = nb; n0 < ne; n0 += GB_K) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = tid & 63, kk = (tid >> 6) + 4 * i;
            const int64_t gn = n0 + kk;
            As[kk][c] = (gn < ne && m0 + c < D) ? dxw[gn * D + m0 + c] : 0.f;
            Bs[kk][c] = (gn < ne && c0 + c < K) ? x[gn * ldx + c0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GB_K; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* Ps = P + int64_t(blockIdx.z) * D * K;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= D) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gk = c0 + tx * 4 + j;
            if (gk < K) Ps[int64_t(gm) * K + gk] = acc[i][j];
        }
    }
}

// out[i] = sum_s P[s][i]  (fixed order => deterministic)
__global__ void reduce_slices(const float* __restrict__ P, int64_t n, int S, float* __restrict__ out)
{
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        // eight independent partial sums keep eight loads in flight; the combine order is fixed => deterministic
        float s[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) s[u] = 0.f;
        int k = 0;
        for (; k + 8 <= S; k += 8) {
#pragma unroll
            for (int u = 0; u < 8; ++u) s[u] += P[int64_t(k + u) * n + i];
        }
        for (; k < S; ++k) s[0] += P[int64_t(k) * n + i];
        out[i] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
    }
}

// datt partials: for column t of xw (head h = t / C):  Ps[s][t] = sum_n da_src[n,h]*xw[n,t], Pd likewise.
template <bool XW_BF16>
__global__ void __launch_bounds__(512)
datt_partial(const void* __restrict__ xw_, const float* __restrict__ da_src, const float* __restrict__ da_dst,
             int64_t N, int D, int H, int C, int64_t rows_per_slice, float* __restrict__ P)
{
    const int64_t nb = int64_t(blockIdx.x) * rows_per_slice;
    const int64_t ne = (nb + rows_per_slice < N) ? nb + rows_per_slice : N;
    for (int t = threadIdx.x; t < D; t += blockDim.x) {
        const int h = t / C;
        float s = 0.f, d = 0.f;
        for (int64_t n = nb; n < ne; ++n) {
            float v;
            if (XW_BF16) v = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(xw_)[n * D + t]);
            else         v = reinterpret_cast<const float*>(xw_)[n * D + t];
            s = fmaf(da_src[n * H + h], v, s);
            d = fmaf(da_dst[n * H + h], v, d);
        }
        P[(int64_t(blockIdx.x) * 2 + 0) * D + t] = s;
        P[(int64_t(blockIdx.x) * 2 + 1) * D + t] = d;
    }
}
// column sums of a [N,Wd] matrix, sliced; thread = column, sixteen independent row loads in flight
__global__ void colsum_partial(const float* __restrict__ A, int64_t N, int Wd, int64_t rows_per_slice, float* __restrict__ P)
{
    const int64_t nb = int64_t(blockIdx.x) * rows_per_slice;
    const int64_t ne = (nb + rows_per_slice < N) ? nb + rows_per_slice : N;
    for (int t = threadIdx.x; t < Wd; t += blockDim.x) {
        float s = 0.f;
        for (int64_t n = nb; n < ne; n += 16) {
            float v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (n + u < ne) ? __ldg(A + (n + u) * Wd + t) : 0.f;
#pragma unroll
            for (int u = 0; u < 16; ++u) s += v[u];
        }
        P[int64_t(blockIdx.x) * Wd + t] = s;
    }
}

// logits from a stored xw (used when C != 64 so the GEMM epilogue cannot own a whole head)
template <bool XW_BF16>
__global__ void alpha_dots(const void* __restrict__ xw_, const float* __restrict__ att_src,
                           const float* __restrict__ att_dst, int64_t N, int H, int C, float* __restrict__ a_src,
                           float* __restrict__ a_dst)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
    if (w >= N * H) return;
    const int64_t n = w / H;
    const int h = int(w % H);
    float s = 0.f, d = 0.f;
    for (int c = lane; c < C; c += 32) {
        float v;
        if (XW_BF16) v = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(xw_)[(n * H + h) * C + c]);
        else         v = reinterpret_cast<const float*>(xw_)[(n * H + h) * C + c];
        s = fmaf(v, att_src[h * C + c], s);
        d = fmaf(v, att_dst[h * C + c], d);
    }
    s = warp_sum(s);
    d = warp_sum(d);
    if (lane == 0) {
        a_src[n * H + h] = s;
        a_dst[n * H + h] = d;
    }
}

// ---- attention-vector gradients without re-reading xw ------------------------------------------------------
// datt_src[h,c] = sum_n da_src[n,h] * xw[n,h,c] and xw = x W^T, so
//   datt_src[h,c] = sum_k W[hC+c,k] * G_src[h,k],   G_src = da_src^T x   ([H,K], reduction over nodes)
// which needs x (K*4 bytes/node) instead of xw (D*s bytes/node).  Pg[s][2H][K] are slab partials.
template <int H, int F>
__global__ void __launch_bounds__(256)
dax_partial(const float* __restrict__ x, int64_t ldx, const float* __restrict__ da_src, const float* __restrict__ da_dst,
            int64_t N, int K, int64_t rows_per_slice, float* __restrict__ Pg)
{
    // thread = F consecutive feature columns (x rows are read as coalesced segments across the CTA; F = 2 reads
    // float2 pairs and halves the shared/global load instructions per feature), F*2H accumulators.
    // The [da_src | da_dst] rows of RB nodes are staged through shared memory with cp.async, one block ahead, and
    // read back as broadcasts; the x loads of the next block are in flight while the current one is multiplied.
    constexpr int RB = 16, V = 2 * H / 4;                 // V float4 per staged node row
    __shared__ __align__(16) float da_s[2][RB][2 * H];
    const int64_t nb = int64_t(blockIdx.x) * rows_per_slice;
    const int64_t ne = (nb + rows_per_slice < N) ? nb + rows_per_slice : N;
    const int64_t n_blk = (ne > nb) ? (ne - nb + RB - 1) / RB : 0;
    auto stage = [&](int buf, int64_t n0) {
        for (int i = threadIdx.x; i < RB * V; i += blockDim.x) {
            const int r = i / V, part = i % V;
            const int64_t n = n0 + r;
            const float* src = (part < V / 2) ? da_src + n * H + 4 * part : da_dst + n * H + 4 * (part - V / 2);
            const uint32_t dst = uint32_t(__cvta_generic_to_shared(&da_s[buf][r][4 * part]));
            const int sz = (n < ne) ? 16 : 0;             // rows past the slab are zero-filled
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(n < ne ? src : da_src), "r"(sz) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int k0 = 0; k0 < K; k0 += F * blockDim.x) {
        const int k = k0 + F * threadIdx.x;
        const bool act = k < K;                            // F = 2: K is even, so the pair is inside the row
        float acc[F][2 * H];
#pragma unroll
        for (int f = 0; f < F; ++f)
#pragma unroll
            for (int h = 0; h < 2 * H; ++h) acc[f][h] = 0.f;
        float xv[RB][F], xn[RB][F];
        auto load_x = [&](int64_t n0, float (&v)[RB][F]) {
#pragma unroll
            for (int u = 0; u < RB; ++u) {
                const bool ok = act && n0 + u < ne;
                if (F == 2) {
                    const float2 p = ok ? __ldg(reinterpret_cast<const float2*>(x + (n0 + u) * ldx + k)) : make_float2(0.f, 0.f);
                    v[u][0] = p.x;
                    v[u][F - 1] = p.y;
                } else {
                    v[u][0] = ok ? __ldg(x + (n0 + u) * ldx + k) : 0.f;
                }
            }
        };
        auto fma_blk = [&](int buf, const float (&v)[RB][F]) {
#pragma unroll
            for (int u = 0; u < RB; ++u) {
#pragma unroll
                for (int q = 0; q < V; ++q) {
                    const float4 d4 = *reinterpret_cast<const float4*>(&da_s[buf][u][4 * q]);
#pragma unroll
                    for (int f = 0; f < F; ++f) {
                        acc[f][4 * q + 0] = fmaf(d4.x, v[u][f], acc[f][4 * q + 0]); acc[f][4 * q + 1] = fmaf(d4.y, v[u][f], acc[f][4 * q + 1]);
                        acc[f][4 * q + 2] = fmaf(d4.z, v[u][f], acc[f][4 * q + 2]); acc[f][4 * q + 3] = fmaf(d4.w, v[u][f], acc[f][4 * q + 3]);
                    }
                }
            }
        };
        if (n_blk > 0) {
            stage(0, nb);
            load_x(nb, xv);
        }
        for (int64_t b = 0; b < n_blk; b += 2) {
            // even block: data in xv / da_s[0]; odd block: xn / da_s[1]
            stage(1, nb + (b + 1) * RB);
            load_x(nb + (b + 1) * RB, xn);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncthreads();
            fma_blk(0, xv);
            __syncthreads();
            stage(0, nb + (b + 2) * RB);
            load_x(nb + (b + 2) * RB, xv);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncthreads();
            fma_blk(1, xn);                                // past-the-end blocks are all zeros
            __syncthreads();
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if (act) {
#pragma unroll
            for (int f = 0; f < F; ++f)
#pragma unroll
                for (int h = 0; h < 2 * H; ++h) Pg[(int64_t(blockIdx.x) * 2 * H + h) * K + k + f] = acc[f][h];
        }
    }
}
// datt_src[o] = sum_k W[o,k] * G[h(o),k],  datt_dst[o] = sum_k W[o,k] * G[H + h(o),k];  one warp per o
__global__ void datt_from_g(const float* __restrict__ W, const float* __restrict__ G, int D, int K, int H, int C,
                            float* __restrict__ datt_src, float* __restrict__ datt_dst)
{
    const int lane = threadIdx.x & 31;
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (o >= D) return;
    const int h = o / C;
    float s = 0.f, d = 0.f;
    for (int k = lane; k < K; k += 32) {
        const float w = W[int64_t(o) * K + k];
        s = fmaf(w, G[int64_t(h) * K + k], s);
        d = fmaf(w, G[int64_t(H + h) * K + k], d);
    }
    s = warp_sum(s);
    d = warp_sum(d);
    if (lane == 0) {
        datt_src[o] = s;
        datt_dst[o] = d;
    }
}

// finer slabs for the column reductions (one thread per column): up to 16 CTAs per SM
int col_slices(int64_t N)
{
    int64_t s = (N + 255) / 256;
    const int64_t cap = 16 * int64_t(sm_count());
    if (s > cap) s = cap;
    if (s < 1) s = 1;
    return (int)s;
}

int slices_for(int64_t N)
{
    int64_t s = (N + 2047) / 2048;
    const int64_t cap = 4 * int64_t(sm_count());
    if (s > cap) s = cap;
    if (s < 1) s = 1;
    return (int)s;
}

// ---- host entry points for the SIMT path (called from the dispatcher in abi.cu) ----------------------
int project_fwd_simt(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst,
                     int64_t N, int64_t K, int H, int C, int xw_dtype, void* xw, float* a_src, float* a_dst,
                     cudaStream_t st)
{
    const int D = H * C;
    if (N == 0) return GNNFD_OK;
    dim3 grid((unsigned)((N + GB_M - 1) / GB_M), (unsigned)((D + GB_N - 1) / GB_N));
    if (C == GB_N) {
        if (xw_dtype == GNNFD_BF16)
            gemm_simt<true, 1, true><<<grid, 256, 0, st>>>(x, ldx, W, 1, K, N, D, (int)K, nullptr,
                                                           (__nv_bfloat16*)xw, D, att_src, att_dst, a_src, a_dst, H);
        else
            gemm_simt<true, 1, false><<<grid, 256, 0, st>>>(x, ldx, W, 1, K, N, D, (int)K, (float*)xw, nullptr, D,
                                                            att_src, att_dst, a_src, a_dst, H);
        g_launches += 1;
    } else {
        GNNFD_REQUIRE(xw_dtype == GNNFD_F32, GNNFD_ERR_UNSUPPORTED, "project_fwd: bf16 xw needs C == 64");
        gemm_simt<true, 0, false><<<grid, 256, 0, st>>>(x, ldx, W, 1, K, N, D, (int)K, (float*)xw, nullptr, D,
                                                        nullptr, nullptr, nullptr, nullptr, H);
        const int64_t warps = N * H;
        alpha_dots<false><<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(xw, att_src, att_dst, N, H, C,
                                                                                a_src, a_dst);
        g_launches += 2;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

size_t project_bwd_ws_bytes(int64_t N, int64_t K, int H, int C)
{
    const int S = slices_for(N);
    const size_t D = size_t(H) * C;
    return carve_bytes(size_t(S) * D * K, 4) + carve_bytes(size_t(S) * 2 * D, 4) + carve_bytes(size_t(S) * D, 4) +
           carve_bytes(size_t(col_slices(N)) * 2 * H * K, 4) + carve_bytes(size_t(2) * H * K, 4) +
           carve_bytes(size_t(col_slices(N)) * D, 4);
}

// dx[N,K] = dxw[N,D] @ W[D,K]
void project_dx_simt(const float* dxw, const float* W, int64_t N, int64_t K, int D, int H, float* dx, int64_t lddx,
                     cudaStream_t st)
{
    dim3 grid((unsigned)((N + GB_M - 1) / GB_M), (unsigned)((K + GB_N - 1) / GB_N));
    gemm_simt<false, 0, false><<<grid, 256, 0, st>>>(dxw, D, W, K, 1, N, (int)K, D, dx, nullptr, lddx, nullptr,
                                                     nullptr, nullptr, nullptr, H);
    g_launches += 1;
}

int project_bwd_simt(const float* x, int64_t ldx, const float* W, const float* dxw, const void* xw, int xw_dtype,
                     const float* da_src, const float* da_dst, const float* d_out, int64_t N, int64_t K, int H,
                     int C, int Co, float* dW, float* datt_src, float* datt_dst, float* dbias, float* dx,
                     int64_t lddx, void* ws, size_t ws_bytes, cudaStream_t st, bool skip_dw, bool skip_dx)
{
    const int D = H * C;
    GNNFD_REQUIRE(ws_bytes >= project_bwd_ws_bytes(N, K, H, C), GNNFD_ERR_WORKSPACE, "project_bwd: workspace too small");
    char* p = reinterpret_cast<char*>(ws);
    const int S = slices_for(N);
    float* Pw = carve<float>(p, size_t(S) * D * K);
    float* Pa = carve<float>(p, size_t(S) * 2 * D);
    float* Pb = carve<float>(p, size_t(S) * D);
    const int Sg = col_slices(N);
    const int64_t rpg = (N + Sg - 1) / Sg;
    float* Pg = carve<float>(p, size_t(Sg) * 2 * H * K);
    float* Gm = carve<float>(p, size_t(2) * H * K);
    float* Pc = carve<float>(p, size_t(Sg) * D);
    if (N == 0) {
        if (dW) cudaMemsetAsync(dW, 0, sizeof(float) * D * K, st);
        if (datt_src) cudaMemsetAsync(datt_src, 0, sizeof(float) * D, st);
        if (datt_dst) cudaMemsetAsync(datt_dst, 0, sizeof(float) * D, st);
        if (dbias) cudaMemsetAsync(dbias, 0, sizeof(float) * Co, st);
        return GNNFD_OK;
    }
    const int64_t rps = ((N + S - 1) / S + GB_K - 1) / GB_K * GB_K;
    if (dW && !skip_dw) {
        dim3 grid((unsigned)((D + GB_M - 1) / GB_M), (unsigned)((K + GB_N - 1) / GB_N), (unsigned)S);
        dw_partial<<<grid, 256, 0, st>>>(dxw, D, x, ldx, N, (int)K, rps, Pw);
        reduce_slices<<<(unsigned)((int64_t(D) * K + 255) / 256), 256, 0, st>>>(Pw, int64_t(D) * K, S, dW);
        g_launches += 2;
    }
    if (datt_src && datt_dst) {
        if (H == 8 || H == 4) {
            // G = [da_src | da_dst]^T x over node slabs, then datt = W . G  (xw is not re-read)
            const bool pair = (K % 2 == 0) && (ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(x) & 7) == 0;
            const int64_t cols = pair ? K / 2 : K;
            const int bs = int(cols >= 256 ? 256 : ((cols + 31) / 32) * 32);
            if (H == 8) {
                if (pair) dax_partial<8, 2><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
                else      dax_partial<8, 1><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
            } else {
                if (pair) dax_partial<4, 2><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
                else      dax_partial<4, 1><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
            }
            reduce_slices<<<(unsigned)((2 * H * K + 255) / 256), 256, 0, st>>>(Pg, int64_t(2) * H * K, Sg, Gm);
            datt_from_g<<<(unsigned)((D * 32 + 255) / 256), 256, 0, st>>>(W, Gm, D, (int)K, H, C, datt_src, datt_dst);
            g_launches += 3;
        } else {
            if (xw_dtype == GNNFD_BF16)
                datt_partial<true><<<S, 512, 0, st>>>(xw, da_src, da_dst, N, D, H, C, rps, Pa);
            else
                datt_partial<false><<<S, 512, 0, st>>>(xw, da_src, da_dst, N, D, H, C, rps, Pa);
            reduce_slices<<<(unsigned)((2 * D + 255) / 256), 256, 0, st>>>(Pa, 2 * int64_t(D), S, Pb);
            cudaMemcpyAsync(datt_src, Pb, sizeof(float) * D, cudaMemcpyDeviceToDevice, st);
            cudaMemcpyAsync(datt_dst, Pb + D, sizeof(float) * D, cudaMemcpyDeviceToDevice, st);
            g_launches += 2;
        }
    }
    if (dbias) {
        colsum_partial<<<Sg, Co >= 256 ? 256 : 64, 0, st>>>(d_out, N, Co, rpg, Pc);
        reduce_slices<<<(unsigned)((Co + 63) / 64), 64, 0, st>>>(Pc, Co, Sg, dbias);
        g_launches += 2;
    }
    if (dx && !skip_dx) project_dx_simt(dxw, W, N, K, D, H, dx, lddx, st);
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

// ---- input-space path (in_gemm.cu): datt_src / datt_dst / dbias and G = [da_src | da_dst]^T x -----------------------
size_t in_param_ws_bytes(int64_t N, int64_t K)
{
    const int Sg = col_slices(N);
    return carve_bytes(size_t(Sg) * 2 * 8 * K, 4) + carve_bytes(size_t(Sg) * 64, 4) + 512;
}
int in_param_grads_simt(const float* x, int64_t ldx, const float* W, const float* da_src, const float* da_dst,
                        const float* d_out, int64_t N, int64_t K, float* datt_src, float* datt_dst, float* dbias,
                        float* Gm, void* ws, size_t ws_bytes, cudaStream_t st)
{
    constexpr int H = 8, C = 64, D = H * C;
    GNNFD_REQUIRE(ws_bytes >= in_param_ws_bytes(N, K), GNNFD_ERR_WORKSPACE, "in_param_grads: workspace too small");
    if (N == 0) {
        cudaMemsetAsync(datt_src, 0, sizeof(float) * D, st);
        cudaMemsetAsync(datt_dst, 0, sizeof(float) * D, st);
        cudaMemsetAsync(dbias, 0, sizeof(float) * C, st);
        cudaMemsetAsync(Gm, 0, sizeof(float) * 2 * H * K, st);
        return GNNFD_OK;
    }
    char* p = reinterpret_cast<char*>(ws);
    const int Sg = col_slices(N);
    const int64_t rpg = (N + Sg - 1) / Sg;
    float* Pg = carve<float>(p, size_t(Sg) * 2 * H * K);
    float* Pc = carve<float>(p, size_t(Sg) * C);
    const bool pair = (K % 2 == 0) && (ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(x) & 7) == 0;
    const int64_t cols = pair ? K / 2 : K;
    const int bs = int(cols >= 256 ? 256 : ((cols + 31) / 32) * 32);
    if (pair) dax_partial<8, 2><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
    else      dax_partial<8, 1><<<Sg, bs, 0, st>>>(x, ldx, da_src, da_dst, N, (int)K, rpg, Pg);
    reduce_slices<<<(unsigned)((2 * H * K + 255) / 256), 256, 0, st>>>(Pg, int64_t(2) * H * K, Sg, Gm);
    datt_from_g<<<(unsigned)((D * 32 + 255) / 256), 256, 0, st>>>(W, Gm, D, (int)K, H, C, datt_src, datt_dst);
    colsum_partial<<<Sg, 64, 0, st>>>(d_out, N, C, rpg, Pc);
    reduce_slices<<<1, 64, 0, st>>>(Pc, C, Sg, dbias);
    g_launches += 5;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace gnnfd
