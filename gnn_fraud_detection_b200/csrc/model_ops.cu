// Model-level fused operators around the GAT layers (SURVEY.md 8(f) "next" rows), all fp32 on [N, C] activations:
//
//   (f1) train-mode inter-layer tail of the reference's layer loop (src/models/gat.py:82-91 == src/models/tgn.py:96-105):
//        BatchNorm1d with BATCH statistics -> ReLU -> feature dropout -> residual add, as
//          gnnfd_bn_sums (+ all-reduce across GPUs) -> gnnfd_bn_finalize (mean, invstd, running statistics)
//          -> gnnfd_bn_relu_drop_res_fwd (ONE elementwise pass), and the mirror-image backward
//          gnnfd_bn_bwd_sums (+ all-reduce) -> gnnfd_bn_bwd_apply.
//        The dropout keep bits come from the same counter-based generator as the attention dropout (no mask tensor).
//   (f3) the TemporalGNN head (src/models/tgn.py:60,88-89,108-111): GRUCell(h, hidden_state) -> Linear(hidden -> 1), one
//        kernel forward, one backward; with the reference's always-zero state the W_hh product vanishes.
//   (f4) the reference's loss on the device (src/train.py:108-139,360-361): masked BCEWithLogitsLoss(pos_weight) with the
//        mean over labelled nodes, its gradient, and the confusion counters of src/train.py:146-149 -- no host sync.
// Column reductions over nodes use per-block partials in double, summed in block order: deterministic, and accurate enough
// that the batch variance needs no second pass.
#include "in_common.cuh"

#include <atomic>

namespace gnnfd {
extern std::atomic<long long> g_launches;

namespace mo {

constexpr int RED_BLOCKS_MAX = 1024;

// P[block][w] = sum over the block's rows of f(row)[w];  thread = column group, rows strided over the block's slab
// MODE 0: w in [0,2C): (z, z^2)            MODE 1: w in [0,2C): (dy, dy*zhat)
template <int MODE>
__global__ void __launch_bounds__(256)
col_sums_kernel(const float* __restrict__ z, const float* __restrict__ d_out, int64_t N, int C, const float* __restrict__ mean,
                const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                KeepMask km, float keep_scale, int64_t row_base, double* __restrict__ P)
{
    // 256 threads = (256 / C) row lanes x C columns (C <= 256, C | 256 not required: extra threads idle)
    const int rl = threadIdx.x / C, c = threadIdx.x % C, nrl = 256 / C;
    double s0 = 0.0, s1 = 0.0;
    if (rl < nrl) {
        const int64_t rows_per_block = (N + gridDim.x - 1) / gridDim.x;
        const int64_t r0 = int64_t(blockIdx.x) * rows_per_block;
        const int64_t r1 = r0 + rows_per_block < N ? r0 + rows_per_block : N;
        float mu = 0.f, is = 1.f, g = 1.f, b = 0.f;
        if (MODE == 1) { mu = mean[c]; is = invstd[c]; g = gamma ? gamma[c] : 1.f; b = beta ? beta[c] : 0.f; }
        for (int64_t n = r0 + rl; n < r1; n += nrl) {
            const float v = z[n * C + c];
            if (MODE == 0) {
                s0 += double(v);
                s1 += double(v) * double(v);
            } else {
                const float zh = (v - mu) * is;
                const float pre = fmaf(zh, g, b);
                float dy = pre > 0.f ? d_out[n * C + c] : 0.f;
                if (km.thr || km.mask) dy = (km.bits((row_base + n) * C + c, 1) & 1u) ? dy * keep_scale : 0.f;
                s0 += double(dy);
                s1 += double(dy) * double(zh);
            }
        }
    }
    __shared__ double sh[2][256];
    sh[0][threadIdx.x] = s0;
    sh[1][threadIdx.x] = s1;
    __syncthreads();
    if (threadIdx.x < C) {
        double a0 = 0.0, a1 = 0.0;
        for (int r = 0; r < nrl; ++r) { a0 += sh[0][r * C + threadIdx.x]; a1 += sh[1][r * C + threadIdx.x]; }
        P[int64_t(blockIdx.x) * 2 * C + threadIdx.x] = a0;
        P[int64_t(blockIdx.x) * 2 * C + C + threadIdx.x] = a1;
    }
}
__global__ void reduce_partials_kernel(const double* __restrict__ P, int n_blocks, int W, double* __restrict__ out)
{
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += P[int64_t(b) * W + w];
    out[w] = s;
}

// sums = (sum z, sum z^2) over `count` rows -> mean, invstd; running statistics as nn.BatchNorm1d updates them
__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, int C, float eps, float momentum,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ mean, float* __restrict__ invstd)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = sums[c] / count;
    double var = sums[C + c] / count - m * m;
    if (var < 0.0) var = 0.0;
    mean[c] = float(m);
    invstd[c] = float(1.0 / sqrt(var + double(eps)));
    if (running_mean) running_mean[c] = float((1.0 - momentum) * double(running_mean[c]) + momentum * m);
    if (running_var) {
        const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
        running_var[c] = float((1.0 - momentum) * double(running_var[c]) + momentum * unbiased);
    }
}

// out = residual + dropout(relu((z - mean) * invstd * gamma + beta)).  PM (in::PeerRows::mode): 0 = out only (the
// single-GPU kernel); 1 / 2 = each finished 16-byte piece also goes to element (row_off * C + i) of the symmetric buffer
// on every rank (one store per peer / one multimem.st), and out may be NULL.
template <int PM>
__global__ void __launch_bounds__(256)
bn_apply_fwd_kernel(const float* __restrict__ z, int64_t total, int C, const float* __restrict__ mean,
                    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                    KeepMask km, float keep_scale, int64_t elem_base, const float* __restrict__ residual, float* __restrict__ out,
                    in::PeerRows peers)
{
    for (int64_t i = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) * 4; i < total; i += int64_t(gridDim.x) * blockDim.x * 4) {
        const int c = int(i % C);
        const float4 v = *reinterpret_cast<const float4*>(z + i);
        const float vv[4] = {v.x, v.y, v.z, v.w};
        float4 r4 = residual ? *reinterpret_cast<const float4*>(residual + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        float rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float y = fmaf((vv[k] - mean[c + k]) * invstd[c + k], gamma ? gamma[c + k] : 1.f, beta ? beta[c + k] : 0.f);
            y = fmaxf(y, 0.f);
            if (km.thr || km.mask) y = (km.bits(elem_base + i + k, 1) & 1u) ? y * keep_scale : 0.f;
            rr[k] += y;
        }
        const float4 o4 = make_float4(rr[0], rr[1], rr[2], rr[3]);
        if (PM == 0 || out) *reinterpret_cast<float4*>(out + i) = o4;
        if (PM == 1)
            for (int g = 0; g < peers.n; ++g) *reinterpret_cast<float4*>(peers.ptr[g] + peers.row_off * C + i) = o4;
        else if (PM == 2)
            in::multimem_st_v4(peers.mc + peers.row_off * C + i, o4);
    }
}
// dz = gamma * invstd * (dy - s1/count - zhat * s2/count),  dy = d_out * keep * relu'
__global__ void __launch_bounds__(256)
bn_apply_bwd_kernel(const float* __restrict__ z, const float* __restrict__ d_out, int64_t total, int C,
                    const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                    const float* __restrict__ beta, KeepMask km, float keep_scale, int64_t elem_base,
                    const double* __restrict__ sums, double count, float* __restrict__ dz, float* __restrict__ dgamma,
                    float* __restrict__ dbeta)
{
    if (blockIdx.x == 0 && threadIdx.x < C) {
        if (dgamma) dgamma[threadIdx.x] = float(sums[C + threadIdx.x]);
        if (dbeta) dbeta[threadIdx.x] = float(sums[threadIdx.x]);
    }
    for (int64_t i = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) * 4; i < total; i += int64_t(gridDim.x) * blockDim.x * 4) {
        const int c = int(i % C);
        const float4 v = *reinterpret_cast<const float4*>(z + i);
        const float4 d = *reinterpret_cast<const float4*>(d_out + i);
        const float vv[4] = {v.x, v.y, v.z, v.w}, dd[4] = {d.x, d.y, d.z, d.w};
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float g = gamma ? gamma[c + k] : 1.f, b = beta ? beta[c + k] : 0.f, is = invstd[c + k];
            const float zh = (vv[k] - mean[c + k]) * is;
            float dy = fmaf(zh, g, b) > 0.f ? dd[k] : 0.f;
            if (km.thr || km.mask) dy = (km.bits(elem_base + i + k, 1) & 1u) ? dy * keep_scale : 0.f;
            const float m1 = float(sums[c + k] / count), m2 = float(sums[C + c + k] / count);
            o[k] = g * is * (dy - m1 - zh * m2);
        }
        *reinterpret_cast<float4*>(dz + i) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// ---- (f3) GRUCell + Linear(hidden -> 1) head, hidden = 64 -------------------------------------------------------------
// Block = 256 threads = 32 nodes x 8 channel groups (8 channels each).  W_ih^T (and W_hh^T when a state is given) live in
// shared memory as [k][3*64] so that a thread's 8 channels of one gate are two float4s; x rows are staged per tile.
constexpr int HD = 64, G3 = 3 * HD, GRU_NODES = 32;
__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + __expf(-v)); }

struct GruW {
    const float* w_ih; const float* w_hh; const float* b_ih; const float* b_hh; const float* w_out; const float* b_out;
};

// gates of one (node, 8-channel group): r, z, n pre-activations split into the input part (gi) and the state part (gh)
__device__ __forceinline__ void gru_gates(const float* __restrict__ xs /*[64] smem*/, const float* __restrict__ hs /*[64] smem or null*/,
                                          const float* __restrict__ wi /*[64][192] smem*/, const float* __restrict__ wh,
                                          const GruW& W, int c0, float (&gi)[3][8], float (&gh)[3][8])
{
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            gi[g][j] = W.b_ih[g * HD + c0 + j];
            gh[g][j] = W.b_hh[g * HD + c0 + j];
        }
    for (int k = 0; k < HD; ++k) {
        const float xv = xs[k];
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const float4 a = *reinterpret_cast<const float4*>(wi + k * G3 + g * HD + c0);
            const float4 b = *reinterpret_cast<const float4*>(wi + k * G3 + g * HD + c0 + 4);
            gi[g][0] = fmaf(xv, a.x, gi[g][0]); gi[g][1] = fmaf(xv, a.y, gi[g][1]); gi[g][2] = fmaf(xv, a.z, gi[g][2]); gi[g][3] = fmaf(xv, a.w, gi[g][3]);
            gi[g][4] = fmaf(xv, b.x, gi[g][4]); gi[g][5] = fmaf(xv, b.y, gi[g][5]); gi[g][6] = fmaf(xv, b.z, gi[g][6]); gi[g][7] = fmaf(xv, b.w, gi[g][7]);
        }
        if (hs) {
            const float hv = hs[k];
#pragma unroll
            for (int g = 0; g < 3; ++g) {
                const float4 a = *reinterpret_cast<const float4*>(wh + k * G3 + g * HD + c0);
                const float4 b = *reinterpret_cast<const float4*>(wh + k * G3 + g * HD + c0 + 4);
                gh[g][0] = fmaf(hv, a.x, gh[g][0]); gh[g][1] = fmaf(hv, a.y, gh[g][1]); gh[g][2] = fmaf(hv, a.z, gh[g][2]); gh[g][3] = fmaf(hv, a.w, gh[g][3]);
                gh[g][4] = fmaf(hv, b.x, gh[g][4]); gh[g][5] = fmaf(hv, b.y, gh[g][5]); gh[g][6] = fmaf(hv, b.z, gh[g][6]); gh[g][7] = fmaf(hv, b.w, gh[g][7]);
            }
        }
    }
}
__device__ __forceinline__ void load_wT(float* dst /*[64][192]*/, const float* __restrict__ w /*[192][64]*/)
{
    for (int i = threadIdx.x; i < G3 * HD; i += blockDim.x) {
        const int o = i / HD, k = i % HD;
        dst[k * G3 + o] = w[i];
    }
}

template <bool HAS_H>
__global__ void __launch_bounds__(256)
gru_head_fwd_kernel(const float* __restrict__ x, const float* __restrict__ h_prev, int64_t N, GruW W, float* __restrict__ h_new,
                    float* __restrict__ out)
{
    extern __shared__ __align__(16) float gsm[];
    float* wi = gsm;                                  // [64][192]
    float* wh = gsm + HD * G3;                        // [64][192] (HAS_H)
    float* xs = gsm + (HAS_H ? 2 : 1) * HD * G3;      // [32][64]
    float* hs = xs + GRU_NODES * HD;                  // [32][64] (HAS_H)
    load_wT(wi, W.w_ih);
    if (HAS_H) load_wT(wh, W.w_hh);
    const int nl = threadIdx.x >> 3, c0 = (threadIdx.x & 7) * 8;
    for (int64_t t0 = int64_t(blockIdx.x) * GRU_NODES; t0 < N; t0 += int64_t(gridDim.x) * GRU_NODES) {
        __syncthreads();
        for (int i = threadIdx.x; i < GRU_NODES * HD / 4; i += blockDim.x) {
            const int64_t n = t0 + (i * 4) / HD;
            const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
            reinterpret_cast<float4*>(xs)[i] = n < N ? reinterpret_cast<const float4*>(x + t0 * HD)[i] : zero;
            if (HAS_H) reinterpret_cast<float4*>(hs)[i] = n < N ? reinterpret_cast<const float4*>(h_prev + t0 * HD)[i] : zero;
        }
        __syncthreads();
        const int64_t n = t0 + nl;
        float gi[3][8], gh[3][8];
        gru_gates(xs + nl * HD, HAS_H ? hs + nl * HD : nullptr, wi, wh, W, c0, gi, gh);
        float hn[8], po = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float r = sigmoidf_(gi[0][j] + gh[0][j]), zg = sigmoidf_(gi[1][j] + gh[1][j]);
            const float nn = tanhf(gi[2][j] + r * gh[2][j]);
            const float hp = HAS_H ? hs[nl * HD + c0 + j] : 0.f;
            hn[j] = (1.f - zg) * nn + zg * hp;
            po = fmaf(hn[j], W.w_out[c0 + j], po);
        }
        po += __shfl_xor_sync(0xffffffffu, po, 1);
        po += __shfl_xor_sync(0xffffffffu, po, 2);
        po += __shfl_xor_sync(0xffffffffu, po, 4);
        if (n < N) {
            *reinterpret_cast<float4*>(h_new + n * HD + c0) = make_float4(hn[0], hn[1], hn[2], hn[3]);
            *reinterpret_cast<float4*>(h_new + n * HD + c0 + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
            if ((threadIdx.x & 7) == 0) out[n] = po + W.b_out[0];
        }
    }
}

// backward: recomputes the gates; writes d_gi [N,192] (and d_gh when a state is given) for the weight-gradient reductions,
// dx [N,64], dh_prev; w_out / b_out gradients go through per-block partials.
template <bool HAS_H>
__global__ void __launch_bounds__(256)
gru_head_bwd_kernel(const float* __restrict__ x, const float* __restrict__ h_prev, const float* __restrict__ d_out,
                    const float* __restrict__ d_hnew, int64_t N, GruW W, float* __restrict__ d_gi, float* __restrict__ d_gh,
                    float* __restrict__ dh_z /*[N,64]: dh * z, the direct path to the previous state (HAS_H)*/,
                    double* __restrict__ Pout /*[blocks][HD + 1]*/)
{
    extern __shared__ __align__(16) float gsm[];
    float* wi = gsm;
    float* wh = gsm + HD * G3;
    float* xs = gsm + (HAS_H ? 2 : 1) * HD * G3;
    float* hs = xs + GRU_NODES * HD;
    load_wT(wi, W.w_ih);
    if (HAS_H) load_wT(wh, W.w_hh);
    const int nl = threadIdx.x >> 3, c0 = (threadIdx.x & 7) * 8;
    double pw[8], pb = 0.0;
#pragma unroll
    for (int j = 0; j < 8; ++j) pw[j] = 0.0;
    for (int64_t t0 = int64_t(blockIdx.x) * GRU_NODES; t0 < N; t0 += int64_t(gridDim.x) * GRU_NODES) {
        __syncthreads();
        for (int i = threadIdx.x; i < GRU_NODES * HD / 4; i += blockDim.x) {
            const int64_t n = t0 + (i * 4) / HD;
            const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
            reinterpret_cast<float4*>(xs)[i] = n < N ? reinterpret_cast<const float4*>(x + t0 * HD)[i] : zero;
            if (HAS_H) reinterpret_cast<float4*>(hs)[i] = n < N ? reinterpret_cast<const float4*>(h_prev + t0 * HD)[i] : zero;
        }
        __syncthreads();
        const int64_t n = t0 + nl;
        if (n >= N) continue;
        float gi[3][8], gh[3][8];
        gru_gates(xs + nl * HD, HAS_H ? hs + nl * HD : nullptr, wi, wh, W, c0, gi, gh);
        const float dov = d_out ? d_out[n] : 0.f;
        if ((threadIdx.x & 7) == 0) pb += double(dov);
        float o_r[8], o_z[8], o_n[8], o_hn[8], o_dhz[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float r = sigmoidf_(gi[0][j] + gh[0][j]), zg = sigmoidf_(gi[1][j] + gh[1][j]);
            const float nn = tanhf(gi[2][j] + r * gh[2][j]);
            const float hp = HAS_H ? hs[nl * HD + c0 + j] : 0.f;
            const float hn = (1.f - zg) * nn + zg * hp;
            pw[j] += double(dov) * double(hn);
            const float dh = dov * W.w_out[c0 + j] + (d_hnew ? d_hnew[n * HD + c0 + j] : 0.f);
            o_dhz[j] = dh * zg;
            const float dn = dh * (1.f - zg), dzg = dh * (hp - nn);
            const float dpn = dn * (1.f - nn * nn);
            o_n[j] = dpn;                                   // d gi_n
            o_hn[j] = dpn * r;                              // d gh_n
            o_r[j] = dpn * gh[2][j] * r * (1.f - r);        // d pre_r
            o_z[j] = dzg * zg * (1.f - zg);                 // d pre_z
        }
        float* gi_o = d_gi + n * G3;
        *reinterpret_cast<float4*>(gi_o + c0) = make_float4(o_r[0], o_r[1], o_r[2], o_r[3]);
        *reinterpret_cast<float4*>(gi_o + c0 + 4) = make_float4(o_r[4], o_r[5], o_r[6], o_r[7]);
        *reinterpret_cast<float4*>(gi_o + HD + c0) = make_float4(o_z[0], o_z[1], o_z[2], o_z[3]);
        *reinterpret_cast<float4*>(gi_o + HD + c0 + 4) = make_float4(o_z[4], o_z[5], o_z[6], o_z[7]);
        *reinterpret_cast<float4*>(gi_o + 2 * HD + c0) = make_float4(o_n[0], o_n[1], o_n[2], o_n[3]);
        *reinterpret_cast<float4*>(gi_o + 2 * HD + c0 + 4) = make_float4(o_n[4], o_n[5], o_n[6], o_n[7]);
        if (HAS_H) {
            *reinterpret_cast<float4*>(dh_z + n * HD + c0) = make_float4(o_dhz[0], o_dhz[1], o_dhz[2], o_dhz[3]);
            *reinterpret_cast<float4*>(dh_z + n * HD + c0 + 4) = make_float4(o_dhz[4], o_dhz[5], o_dhz[6], o_dhz[7]);
        }
        {   // the state-side gate gradients (also without a state: they carry the bias gradient d b_hh)
            float* gh_o = d_gh + n * G3;
            *reinterpret_cast<float4*>(gh_o + c0) = make_float4(o_r[0], o_r[1], o_r[2], o_r[3]);
            *reinterpret_cast<float4*>(gh_o + c0 + 4) = make_float4(o_r[4], o_r[5], o_r[6], o_r[7]);
            *reinterpret_cast<float4*>(gh_o + HD + c0) = make_float4(o_z[0], o_z[1], o_z[2], o_z[3]);
            *reinterpret_cast<float4*>(gh_o + HD + c0 + 4) = make_float4(o_z[4], o_z[5], o_z[6], o_z[7]);
            *reinterpret_cast<float4*>(gh_o + 2 * HD + c0) = make_float4(o_hn[0], o_hn[1], o_hn[2], o_hn[3]);
            *reinterpret_cast<float4*>(gh_o + 2 * HD + c0 + 4) = make_float4(o_hn[4], o_hn[5], o_hn[6], o_hn[7]);
        }
    }
    // per-block partials of (d w_out [64], d b_out): thread (nl, cg) holds 8 channels; reduce over the 32 node lanes
    __shared__ double red[256][9];
#pragma unroll
    for (int j = 0; j < 8; ++j) red[threadIdx.x][j] = pw[j];
    red[threadIdx.x][8] = pb;
    __syncthreads();
    if (threadIdx.x < HD + 1) {
        double s = 0.0;
        if (threadIdx.x < HD) {
            const int cg = threadIdx.x >> 3, j = threadIdx.x & 7;
            for (int r = 0; r < GRU_NODES; ++r) s += red[r * 8 + cg][j];
        } else {
            for (int r = 0; r < GRU_NODES; ++r) s += red[r * 8][8];
        }
        Pout[int64_t(blockIdx.x) * (HD + 1) + threadIdx.x] = s;
    }
}

// C[N, Kd] = A[N, G3] @ Wm[G3, Kd]   (dx = d_gi @ W_ih ; dh = d_gh @ W_hh): block = 64 nodes, thread = (2 nodes, 8 columns):
// per gate 2 + 2 shared loads feed 16 FMAs
constexpr int GTW_NODES = 64;
__global__ void __launch_bounds__(256)
gates_times_w_kernel(const float* __restrict__ A, const float* __restrict__ Wm /*[192][64]*/, int64_t N, const float* __restrict__ add,
                     float scale_add, float* __restrict__ Cout)
{
    extern __shared__ __align__(16) float gsm[];
    float* ws = gsm;                       // [192][64]
    float* as = gsm + G3 * HD;             // [64][192 + 4]  (padded: the two nodes of a thread and the 8 node pairs of a warp
                                           //                 quarter fall into different banks)
    constexpr int LDA = G3 + 4;
    for (int i = threadIdx.x; i < G3 * HD; i += blockDim.x) ws[i] = Wm[i];
    const int nl = (threadIdx.x >> 3) * 2, c0 = (threadIdx.x & 7) * 8;
    for (int64_t t0 = int64_t(blockIdx.x) * GTW_NODES; t0 < N; t0 += int64_t(gridDim.x) * GTW_NODES) {
        __syncthreads();
        for (int i = threadIdx.x; i < GTW_NODES * G3 / 4; i += blockDim.x) {
            const int r = (i * 4) / G3, c = (i * 4) % G3;
            const int64_t n = t0 + r;
            *reinterpret_cast<float4*>(as + r * LDA + c) =
                n < N ? *reinterpret_cast<const float4*>(A + n * G3 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        float acc[2][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = 0.f;
#pragma unroll 4
        for (int o = 0; o < G3; ++o) {
            const float a0 = as[nl * LDA + o], a1 = as[(nl + 1) * LDA + o];
            const float4 w0 = *reinterpret_cast<const float4*>(ws + o * HD + c0), w1 = *reinterpret_cast<const float4*>(ws + o * HD + c0 + 4);
            acc[0][0] = fmaf(a0, w0.x, acc[0][0]); acc[0][1] = fmaf(a0, w0.y, acc[0][1]); acc[0][2] = fmaf(a0, w0.z, acc[0][2]); acc[0][3] = fmaf(a0, w0.w, acc[0][3]);
            acc[0][4] = fmaf(a0, w1.x, acc[0][4]); acc[0][5] = fmaf(a0, w1.y, acc[0][5]); acc[0][6] = fmaf(a0, w1.z, acc[0][6]); acc[0][7] = fmaf(a0, w1.w, acc[0][7]);
            acc[1][0] = fmaf(a1, w0.x, acc[1][0]); acc[1][1] = fmaf(a1, w0.y, acc[1][1]); acc[1][2] = fmaf(a1, w0.z, acc[1][2]); acc[1][3] = fmaf(a1, w0.w, acc[1][3]);
            acc[1][4] = fmaf(a1, w1.x, acc[1][4]); acc[1][5] = fmaf(a1, w1.y, acc[1][5]); acc[1][6] = fmaf(a1, w1.z, acc[1][6]); acc[1][7] = fmaf(a1, w1.w, acc[1][7]);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int64_t n = t0 + nl + u;
            if (n < N) {
                if (add) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[u][j] = fmaf(scale_add, add[n * HD + c0 + j], acc[u][j]);
                }
                *reinterpret_cast<float4*>(Cout + n * HD + c0) = make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
                *reinterpret_cast<float4*>(Cout + n * HD + c0 + 4) = make_float4(acc[u][4], acc[u][5], acc[u][6], acc[u][7]);
            }
        }
    }
}
// P[block][o][k] partial of  dW[o,k] = sum_n G[n,o] * X[n,k]  and  db[o] = sum_n G[n,o]   (o < 192, k < 64).
// block = 192 threads: thread (og = t % 48, kq = t / 48) owns the 4 gate columns 4 og .. and the 16 inputs 16 kq ..:
// 64 accumulators fed per node by ONE 128-bit load of G and four broadcast 128-bit shared loads of x.
// X == NULL (the reference's zero state: dW_hh = 0): only the column sums are computed.
constexpr int GO_THREADS = 192;
__global__ void __launch_bounds__(GO_THREADS)
gates_outer_kernel(const float* __restrict__ G, const float* __restrict__ X, int64_t N, double* __restrict__ P /*[blocks][192][65]*/)
{
    __shared__ __align__(16) float xs[GRU_NODES][HD];
    const int og = threadIdx.x % 48, kq = threadIdx.x / 48;
    const int64_t rows_per_block = ((N + gridDim.x - 1) / gridDim.x + GRU_NODES - 1) / GRU_NODES * GRU_NODES;
    const int64_t r0 = int64_t(blockIdx.x) * rows_per_block;
    const int64_t r1 = r0 + rows_per_block < N ? r0 + rows_per_block : N;
    float acc[4][16];
    float accb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[u][k] = 0.f;
    if (X == nullptr) {
        if (kq == 0)
            for (int64_t r = r0; r < r1; ++r) {
                const float4 g = *reinterpret_cast<const float4*>(G + r * G3 + 4 * og);
                accb[0] += g.x; accb[1] += g.y; accb[2] += g.z; accb[3] += g.w;
            }
    } else {
        for (int64_t t0 = r0; t0 < r1; t0 += GRU_NODES) {
            __syncthreads();
            for (int i = threadIdx.x; i < GRU_NODES * HD / 4; i += blockDim.x) {
                const int64_t n = t0 + (i * 4) / HD;
                reinterpret_cast<float4*>(&xs[0][0])[i] = n < r1 ? reinterpret_cast<const float4*>(X + t0 * HD)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __syncthreads();
            const int cnt = int(r1 - t0 < GRU_NODES ? r1 - t0 : GRU_NODES);
            for (int r = 0; r < cnt; ++r) {
                const float4 g4 = *reinterpret_cast<const float4*>(G + (t0 + r) * G3 + 4 * og);
                const float g[4] = {g4.x, g4.y, g4.z, g4.w};
                if (kq == 0) { accb[0] += g[0]; accb[1] += g[1]; accb[2] += g[2]; accb[3] += g[3]; }
#pragma unroll
                for (int k = 0; k < 16; k += 4) {
                    const float4 xv = *reinterpret_cast<const float4*>(&xs[r][16 * kq + k]);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        acc[u][k] = fmaf(g[u], xv.x, acc[u][k]); acc[u][k + 1] = fmaf(g[u], xv.y, acc[u][k + 1]);
                        acc[u][k + 2] = fmaf(g[u], xv.z, acc[u][k + 2]); acc[u][k + 3] = fmaf(g[u], xv.w, acc[u][k + 3]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        double* p = P + (int64_t(blockIdx.x) * G3 + 4 * og + u) * (HD + 1);
#pragma unroll
        for (int k = 0; k < 16; ++k) p[16 * kq + k] = double(acc[u][k]);
        if (kq == 0) p[HD] = double(accb[u]);
    }
}
// dW[o,k] / db[o] from the block partials (fixed order)
__global__ void gates_outer_reduce_kernel(const double* __restrict__ P, int n_blocks, float* __restrict__ dW, float* __restrict__ db)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G3 * (HD + 1)) return;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += P[int64_t(b) * G3 * (HD + 1) + i];
    const int o = i / (HD + 1), k = i % (HD + 1);
    if (k < HD) { if (dW) dW[o * HD + k] = float(s); }
    else if (db) db[o] = float(s);
}
__global__ void head_out_reduce_kernel(const double* __restrict__ P, int n_blocks, float* __restrict__ dw_out, float* __restrict__ db_out)
{
    const int i = threadIdx.x;
    if (i > HD) return;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += P[int64_t(b) * (HD + 1) + i];
    if (i < HD) dw_out[i] = float(s);
    else db_out[0] = float(s);
}

// ---- (f4) masked BCE-with-logits(pos_weight), mean over labelled nodes --------------------------------------------------
// stats (double[8]): [0] sum of losses, [1] labelled count, [2] TP, [3] FP, [4] TN, [5] FN (threshold: sigmoid >= 0.5)
__global__ void __launch_bounds__(256)
bce_partial_kernel(const float* __restrict__ logits, const int64_t* __restrict__ y, int64_t N, float pos_weight,
                   float* __restrict__ g_unnorm, double* __restrict__ P /*[blocks][6]*/)
{
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < N; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t yi = y[i];
        float g = 0.f;
        if (yi != -1) {
            const float xv = logits[i], yf = float(yi);
            // softplus(v) = max(v,0) + log1p(exp(-|v|)); the accurate expf: a well-classified node's loss IS the log1p term,
            // and __expf's error grows with |v| (about 25 ulp at |v| = 20) and flushes results below 2^-126 to zero
            const float l1p = log1pf(expf(-fabsf(xv)));
            const float sp_pos = fmaxf(xv, 0.f) + l1p, sp_neg = fmaxf(-xv, 0.f) + l1p;
            s[0] += double(pos_weight * yf * sp_neg + (1.f - yf) * sp_pos);
            s[1] += 1.0;
            const float sg = 1.f / (1.f + __expf(-xv));
            g = sg * (pos_weight * yf + 1.f - yf) - pos_weight * yf;
            // the reference's predicate is torch.sigmoid(logit) >= 0.5 in fp32, which torch on CUDA evaluates as
            // 1 / (1 + expf(-x)) with IEEE add and divide: it holds for small negative logits too (down to -1.6525915e-7
            // with CUDA's expf; CPU torch's differs, -1.7881391e-7), so `xv >= 0` would miscount those.  Same arithmetic,
            // same answer, bit for bit.
            const bool pred = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-xv))) >= 0.5f, pos = yi == 1;
            s[2] += (pred && pos); s[3] += (pred && !pos); s[4] += (!pred && !pos); s[5] += (!pred && pos);
        }
        g_unnorm[i] = g;
    }
    __shared__ double sh[6][256];
#pragma unroll
    for (int k = 0; k < 6; ++k) sh[k][threadIdx.x] = s[k];
    __syncthreads();
    if (threadIdx.x < 6) {
        double a = 0.0;
        for (int t = 0; t < 256; ++t) a += sh[threadIdx.x][t];
        P[int64_t(blockIdx.x) * 6 + threadIdx.x] = a;
    }
}
__global__ void bce_finalize_kernel(const double* __restrict__ P, int n_blocks, double* __restrict__ stats, float* __restrict__ loss)
{
    const int k = threadIdx.x;
    if (k < 6) {
        double a = 0.0;
        for (int b = 0; b < n_blocks; ++b) a += P[int64_t(b) * 6 + k];
        stats[k] = a;
    }
    __syncthreads();
    if (k == 0) loss[0] = stats[1] > 0.0 ? float(stats[0] / stats[1]) : 0.f;
}
__global__ void bce_scale_kernel(float* __restrict__ g, int64_t N, const double* __restrict__ stats, float upstream)
{
    const float inv = stats[1] > 0.0 ? float(double(upstream) / stats[1]) : 0.f;
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < N; i += int64_t(gridDim.x) * blockDim.x) g[i] *= inv;
}

static int red_blocks(int64_t N, int64_t rows_per)
{
    int64_t b = (N + rows_per - 1) / rows_per;
    if (b > RED_BLOCKS_MAX) b = RED_BLOCKS_MAX;
    if (b < 1) b = 1;
    return int(b);
}

}  // namespace mo
}  // namespace gnnfd

using namespace gnnfd;
using namespace gnnfd::mo;

extern "C" {

/* workspace for every call in this section (bytes) */
int gnnfd_model_ops_workspace_bytes(int64_t N, size_t* bytes)
{
    GNNFD_REQUIRE(bytes && N >= 0, GNNFD_ERR_ARG, "model_ops_workspace_bytes: bad argument");
    *bytes = size_t(RED_BLOCKS_MAX) * 2 * 256 * sizeof(double) + size_t(296) * G3 * (HD + 1) * sizeof(double) +
             size_t(RED_BLOCKS_MAX) * (HD + 1) * sizeof(double) + 4096;
    return GNNFD_OK;
}

/* sums [2C] (double) = column sums of z and z*z over the N rows (one rank's share of the batch). */
int gnnfd_bn_sums(const float* z, int64_t N, int C, double* sums, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(C >= 1 && C <= 256 && C % 4 == 0 && N >= 0 && sums, GNNFD_ERR_ARG, "bn_sums: C must be a multiple of 4, <= 256");
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) { GNNFD_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * C, st)); return GNNFD_OK; }
    const int nb = red_blocks(N, 256);
    GNNFD_REQUIRE(z && ws && ws_bytes >= size_t(nb) * 2 * C * sizeof(double), GNNFD_ERR_WORKSPACE, "bn_sums: workspace too small");
    double* P = reinterpret_cast<double*>(ws);
    col_sums_kernel<0><<<nb, 256, 0, st>>>(z, nullptr, N, C, nullptr, nullptr, nullptr, nullptr, KeepMask(), 1.f, 0, P);
    reduce_partials_kernel<<<(2 * C + 127) / 128, 128, 0, st>>>(P, nb, 2 * C, sums);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* mean / invstd [C] from the (all-reduced) sums over `count` rows; updates running_mean / running_var (may be NULL) exactly
 * as nn.BatchNorm1d does in training (momentum, unbiased variance). */
int gnnfd_bn_finalize(const double* sums, double count, int C, float eps, float momentum, float* running_mean,
                      float* running_var, float* mean, float* invstd, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(sums && mean && invstd && C >= 1 && count >= 1.0, GNNFD_ERR_ARG, "bn_finalize: bad argument");
    bn_finalize_kernel<<<(C + 63) / 64, 64, 0, (cudaStream_t)stream>>>(sums, count, C, eps, momentum, running_mean, running_var, mean, invstd);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* out = residual + dropout_p(relu((z - mean) * invstd * gamma + beta))   (src/models/gat.py:82-91).  Feature dropout:
 * p_drop = 0 => none; otherwise the counter-based generator keyed on (dropout_seed, (row_base + n) * C + c). */
int gnnfd_bn_relu_drop_res_fwd(const float* z, int64_t N, int C, const float* mean, const float* invstd, const float* gamma,
                               const float* beta, float p_drop, uint64_t dropout_seed, int64_t row_base,
                               const float* residual, float* out, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(C >= 4 && C % 4 == 0 && N >= 0 && p_drop >= 0.f && p_drop < 1.f, GNNFD_ERR_ARG, "bn_relu_drop_res_fwd: bad argument");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(z && mean && invstd && out, GNNFD_ERR_ARG, "bn_relu_drop_res_fwd: NULL tensor");
    float ks = 1.f;
    const KeepMask km = make_keep(nullptr, p_drop, dropout_seed, &ks);
    const int64_t total = N * C;
    int64_t blocks = (total / 4 + 255) / 256;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    bn_apply_fwd_kernel<0><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(z, total, C, mean, invstd, gamma, beta, km, ks,
                                                                            row_base * C, residual, out, in::PeerRows{});
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* gnnfd_bn_relu_drop_res_fwd fused with the all-gather of its rows: every finished 16-byte piece of row r also goes to row
 * (row_offset + r) of h_all [n_pos, C] on every rank (one multimem.st, or one store per peer).  out (own rows) may be NULL. */
int gnnfd_bn_relu_drop_res_fwd_bcast(const float* z, int64_t N, int C, const float* mean, const float* invstd,
                                     const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed,
                                     int64_t row_base, const float* residual, const gnnfd_peers_t* h_all,
                                     int64_t row_offset, int use_multicast, float* out, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(C >= 4 && C % 4 == 0 && N >= 0 && p_drop >= 0.f && p_drop < 1.f, GNNFD_ERR_ARG,
                  "bn_relu_drop_res_fwd_bcast: bad argument");
    in::PeerRows peers;
    const int rc = in::peer_rows_from(h_all, row_offset, use_multicast, "bn_relu_drop_res_fwd_bcast", peers);
    if (rc) return rc;
    GNNFD_REQUIRE(!use_multicast || (reinterpret_cast<uintptr_t>(h_all->multicast) & 15) == 0, GNNFD_ERR_ARG,
                  "bn_relu_drop_res_fwd_bcast: the multicast address must be 16-byte aligned");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(z && mean && invstd, GNNFD_ERR_ARG, "bn_relu_drop_res_fwd_bcast: NULL tensor");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(z) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(residual) & 15) == 0, GNNFD_ERR_ARG,
                  "bn_relu_drop_res_fwd_bcast: z, residual and out must be 16-byte aligned");
    float ks = 1.f;
    const KeepMask km = make_keep(nullptr, p_drop, dropout_seed, &ks);
    const int64_t total = N * C;
    int64_t blocks = (total / 4 + 255) / 256;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    cudaStream_t st = (cudaStream_t)stream;
    if (use_multicast)
        bn_apply_fwd_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(z, total, C, mean, invstd, gamma, beta, km, ks, row_base * C,
                                                                residual, out, peers);
    else
        bn_apply_fwd_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(z, total, C, mean, invstd, gamma, beta, km, ks, row_base * C,
                                                                residual, out, peers);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* backward, step 1: sums [2C] (double) = column sums of dy and dy*zhat over this rank's rows (dy = d_out through dropout and
 * ReLU). */
int gnnfd_bn_bwd_sums(const float* z, const float* d_out, int64_t N, int C, const float* mean, const float* invstd,
                      const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed, int64_t row_base,
                      double* sums, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(C >= 1 && C <= 256 && C % 4 == 0 && N >= 0 && sums, GNNFD_ERR_ARG, "bn_bwd_sums: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) { GNNFD_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * C, st)); return GNNFD_OK; }
    const int nb = red_blocks(N, 256);
    GNNFD_REQUIRE(z && d_out && mean && invstd && ws && ws_bytes >= size_t(nb) * 2 * C * sizeof(double), GNNFD_ERR_WORKSPACE,
                  "bn_bwd_sums: NULL tensor or workspace too small");
    float ks = 1.f;
    const KeepMask km = make_keep(nullptr, p_drop, dropout_seed, &ks);
    double* P = reinterpret_cast<double*>(ws);
    col_sums_kernel<1><<<nb, 256, 0, st>>>(z, d_out, N, C, mean, invstd, gamma, beta, km, ks, row_base, P);
    reduce_partials_kernel<<<(2 * C + 127) / 128, 128, 0, st>>>(P, nb, 2 * C, sums);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}
/* backward, step 2: dz [N,C], dgamma / dbeta [C] (may be NULL) from the (all-reduced) sums over `count` rows. */
int gnnfd_bn_bwd_apply(const float* z, const float* d_out, int64_t N, int C, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed, int64_t row_base,
                       const double* sums, double count, float* dz, float* dgamma, float* dbeta, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(C >= 4 && C <= 256 && C % 4 == 0 && N >= 0 && count >= 1.0 && sums, GNNFD_ERR_ARG, "bn_bwd_apply: bad argument");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(z && d_out && mean && invstd && dz, GNNFD_ERR_ARG, "bn_bwd_apply: NULL tensor");
    float ks = 1.f;
    const KeepMask km = make_keep(nullptr, p_drop, dropout_seed, &ks);
    const int64_t total = N * C;
    int64_t blocks = (total / 4 + 255) / 256;
    if (blocks > int64_t(sm_count()) * 16) blocks = int64_t(sm_count()) * 16;
    bn_apply_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(z, d_out, total, C, mean, invstd, gamma, beta, km, ks,
                                                                         row_base * C, sums, count, dz, dgamma, dbeta);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* TemporalGNN head (hidden = 64): h_new [N,64] = GRUCell(x, h_prev) (h_prev NULL = the reference's zero state), out [N] =
 * h_new . w_out + b_out.  Weights in nn.GRUCell / nn.Linear layout: w_ih, w_hh [192,64], b_ih, b_hh [192], w_out [64]. */
int gnnfd_gru_head_fwd(const float* x, const float* h_prev, int64_t N, const float* w_ih, const float* w_hh,
                       const float* b_ih, const float* b_hh, const float* w_out, const float* b_out, float* h_new,
                       float* out, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && w_ih && w_hh && b_ih && b_hh && w_out && b_out, GNNFD_ERR_ARG, "gru_head_fwd: NULL parameter");
    if (N == 0) return GNNFD_OK;
    GNNFD_REQUIRE(x && h_new && out, GNNFD_ERR_ARG, "gru_head_fwd: NULL tensor");
    cudaStream_t st = (cudaStream_t)stream;
    const GruW W{w_ih, w_hh, b_ih, b_hh, w_out, b_out};
    int64_t blocks = (N + GRU_NODES - 1) / GRU_NODES;
    if (blocks > int64_t(sm_count()) * 2) blocks = int64_t(sm_count()) * 2;
    if (h_prev) {
        const int smem = (2 * HD * G3 + 2 * GRU_NODES * HD) * 4;
        GNNFD_CUDA(cudaFuncSetAttribute(gru_head_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        gru_head_fwd_kernel<true><<<(unsigned)blocks, 256, smem, st>>>(x, h_prev, N, W, h_new, out);
    } else {
        const int smem = (HD * G3 + 2 * GRU_NODES * HD) * 4;
        GNNFD_CUDA(cudaFuncSetAttribute(gru_head_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        gru_head_fwd_kernel<false><<<(unsigned)blocks, 256, smem, st>>>(x, nullptr, N, W, h_new, out);
    }
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* backward of the head: d_out [N] and / or d_hnew [N,64] (either may be NULL) -> dx [N,64], dh_prev [N,64] (NULL when no
 * state), dw_ih / dw_hh [192,64], db_ih / db_hh [192], dw_out [64], db_out [1].  scratch: d_gi (and d_gh) [N,192] from the
 * caller (gates_ws, 2*N*192 floats). */
int gnnfd_gru_head_bwd(const float* x, const float* h_prev, const float* d_out, const float* d_hnew, int64_t N,
                       const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, const float* w_out,
                       const float* b_out, float* dx, float* dh_prev, float* dw_ih, float* dw_hh, float* db_ih,
                       float* db_hh, float* dw_out, float* db_out, float* gates_ws, void* ws, size_t ws_bytes,
                       gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && w_ih && w_hh && b_ih && b_hh && w_out && b_out && dw_ih && dw_hh && db_ih && db_hh && dw_out && db_out,
                  GNNFD_ERR_ARG, "gru_head_bwd: NULL parameter");
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) {
        cudaMemsetAsync(dw_ih, 0, sizeof(float) * G3 * HD, st); cudaMemsetAsync(dw_hh, 0, sizeof(float) * G3 * HD, st);
        cudaMemsetAsync(db_ih, 0, sizeof(float) * G3, st); cudaMemsetAsync(db_hh, 0, sizeof(float) * G3, st);
        cudaMemsetAsync(dw_out, 0, sizeof(float) * HD, st); cudaMemsetAsync(db_out, 0, sizeof(float), st);
        return GNNFD_OK;
    }
    size_t need = 0;
    gnnfd_model_ops_workspace_bytes(N, &need);
    GNNFD_REQUIRE(x && dx && gates_ws && ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "gru_head_bwd: NULL tensor or workspace too small");
    const GruW W{w_ih, w_hh, b_ih, b_hh, w_out, b_out};
    float* d_gi = gates_ws;
    float* d_gh = gates_ws + N * G3;
    char* p = reinterpret_cast<char*>(ws);
    double* Pout = carve<double>(p, size_t(RED_BLOCKS_MAX) * (HD + 1));
    double* Pg = carve<double>(p, size_t(296) * G3 * (HD + 1));
    int64_t blocks = (N + GRU_NODES - 1) / GRU_NODES;
    if (blocks > int64_t(sm_count()) * 2) blocks = int64_t(sm_count()) * 2;
    if (h_prev) {
        GNNFD_REQUIRE(dh_prev, GNNFD_ERR_ARG, "gru_head_bwd: dh_prev is NULL");
        const int smem = (2 * HD * G3 + 2 * GRU_NODES * HD) * 4;
        GNNFD_CUDA(cudaFuncSetAttribute(gru_head_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        gru_head_bwd_kernel<true><<<(unsigned)blocks, 256, smem, st>>>(x, h_prev, d_out, d_hnew, N, W, d_gi, d_gh, dh_prev, Pout);
    } else {
        const int smem = (HD * G3 + 2 * GRU_NODES * HD) * 4;
        GNNFD_CUDA(cudaFuncSetAttribute(gru_head_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        gru_head_bwd_kernel<false><<<(unsigned)blocks, 256, smem, st>>>(x, nullptr, d_out, d_hnew, N, W, d_gi, d_gh, nullptr, Pout);
    }
    head_out_reduce_kernel<<<1, 128, 0, st>>>(Pout, (int)blocks, dw_out, db_out);
    const int smem_w = (G3 * HD + GTW_NODES * (G3 + 4)) * 4;
    int64_t wblocks = (N + GTW_NODES - 1) / GTW_NODES;
    if (wblocks > int64_t(sm_count()) * 2) wblocks = int64_t(sm_count()) * 2;
    GNNFD_CUDA(cudaFuncSetAttribute(gates_times_w_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_w));
    gates_times_w_kernel<<<(unsigned)wblocks, 256, smem_w, st>>>(d_gi, w_ih, N, nullptr, 0.f, dx);
    int ob = int((N + 511) / 512);
    if (ob > 296) ob = 296;
    if (ob < 1) ob = 1;
    gates_outer_kernel<<<ob, GO_THREADS, 0, st>>>(d_gi, x, N, Pg);
    gates_outer_reduce_kernel<<<(G3 * (HD + 1) + 255) / 256, 256, 0, st>>>(Pg, ob, dw_ih, db_ih);
    // state side: dW_hh = d_gh^T h_prev (zero without a state), d b_hh = column sums of d_gh, dh_prev = dh*z + d_gh W_hh
    gates_outer_kernel<<<ob, GO_THREADS, 0, st>>>(d_gh, h_prev, N, Pg);
    gates_outer_reduce_kernel<<<(G3 * (HD + 1) + 255) / 256, 256, 0, st>>>(Pg, ob, dw_hh, db_hh);
    g_launches += 7;
    if (h_prev) {
        gates_times_w_kernel<<<(unsigned)wblocks, 256, smem_w, st>>>(d_gh, w_hh, N, dh_prev, 1.f, dh_prev);
        g_launches += 1;
    }
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

/* loss [1] = mean over {n : y[n] != -1} of BCEWithLogits(logits[n], y[n]; pos_weight); d_logits [N] = upstream * dloss/dlogits
 * (0 at unlabelled nodes); stats (double[8], device): sum of losses, labelled count, TP, FP, TN, FN at sigmoid >= 0.5. */
int gnnfd_bce_masked(const float* logits, const int64_t* y, int64_t N, float pos_weight, float upstream, float* loss,
                     float* d_logits, double* stats, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && loss && stats, GNNFD_ERR_ARG, "bce_masked: NULL output");
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) {
        GNNFD_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 8, st));
        GNNFD_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), st));
        return GNNFD_OK;
    }
    const int nb = red_blocks(N, 2048);
    GNNFD_REQUIRE(logits && y && d_logits && ws && ws_bytes >= size_t(nb) * 6 * sizeof(double), GNNFD_ERR_WORKSPACE,
                  "bce_masked: NULL tensor or workspace too small");
    double* P = reinterpret_cast<double*>(ws);
    bce_partial_kernel<<<nb, 256, 0, st>>>(logits, y, N, pos_weight, d_logits, P);
    bce_finalize_kernel<<<1, 32, 0, st>>>(P, nb, stats, loss);
    bce_scale_kernel<<<nb, 256, 0, st>>>(d_logits, N, stats, upstream);
    g_launches += 3;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // extern "C"
