// Three-phase exclusive scan over a functor, shared by the CSR builder / snapshot builder (csr_radix.cu) and the
// neighbour sampler (sample.cu).  exclusive_scan(f, g, n, ...) computes v[i] = f(i), calls g(i, v[i], exclusive prefix)
// for every i < n in one pass over the input after the block sums, and writes the grand total to *total_dev.  f is
// evaluated twice per element (block sums, then apply), so it must return the same value both times.
#pragma once
#include "common.cuh"

#include <atomic>

namespace gnnfd {

extern std::atomic<long long> g_launches;

constexpr int SC_THREADS = 256;
constexpr int SC_ITEMS = 16;
constexpr int SC_TILE = SC_THREADS * SC_ITEMS;

template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* total, T* smem /* [9] */)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T n = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) smem[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        T w = lane < (SC_THREADS / 32) ? smem[lane] : T(0);
        T wi = w;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            T n = __shfl_up_sync(FULL, wi, o);
            if (lane >= o) wi += n;
        }
        if (lane < 8) smem[lane] = wi - w;
        if (lane == 7) smem[8] = wi;
    }
    __syncthreads();
    T r = smem[warp] + incl - v;
    *total = smem[8];
    __syncthreads();
    return r;
}

template <typename T, class F>
__global__ void __launch_bounds__(SC_THREADS) scan_block_sums(F f, int64_t n, T* block_sums)
{
    __shared__ T sm[9];
    const int64_t base = int64_t(blockIdx.x) * SC_TILE + int64_t(threadIdx.x) * SC_ITEMS;
    T s = 0;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i)
        if (base + i < n) s += f(base + i);
    T total;
    block_exclusive_scan<T>(s, &total, sm);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: in-place exclusive scan of block_sums[nb], grand total to *total_out
template <typename T>
__global__ void __launch_bounds__(SC_THREADS) scan_block_offsets(T* block_sums, int64_t nb, T* total_out)
{
    __shared__ T sm[9];
    T carry = 0;
    for (int64_t base = 0; base < nb; base += SC_THREADS) {
        int64_t i = base + threadIdx.x;
        T v = i < nb ? block_sums[i] : T(0);
        T total;
        T ex = block_exclusive_scan<T>(v, &total, sm);
        if (i < nb) block_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

template <typename T, class F, class G>
__global__ void __launch_bounds__(SC_THREADS) scan_apply(F f, G g, int64_t n, const T* block_off)
{
    __shared__ T sm[9];
    const int64_t base = int64_t(blockIdx.x) * SC_TILE + int64_t(threadIdx.x) * SC_ITEMS;
    T v[SC_ITEMS];
    T s = 0;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        v[i] = (base + i < n) ? f(base + i) : T(0);
        s += v[i];
    }
    T total;
    T run = block_exclusive_scan<T>(s, &total, sm) + block_off[blockIdx.x];
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        if (base + i < n) g(base + i, v[i], run);
        run += v[i];
    }
}

// block_sums needs (n + SC_TILE - 1) / SC_TILE entries
template <typename T, class F, class G>
static int exclusive_scan(F f, G g, int64_t n, T* block_sums, T* total_dev, cudaStream_t st)
{
    if (n <= 0) {
        cudaMemsetAsync(total_dev, 0, sizeof(T), st);
        return GNNFD_OK;
    }
    const int64_t nb = (n + SC_TILE - 1) / SC_TILE;
    scan_block_sums<T, F><<<(unsigned)nb, SC_THREADS, 0, st>>>(f, n, block_sums);
    scan_block_offsets<T><<<1, SC_THREADS, 0, st>>>(block_sums, nb, total_dev);
    scan_apply<T, F, G><<<(unsigned)nb, SC_THREADS, 0, st>>>(f, g, n, block_sums);
    g_launches += 3;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // namespace gnnfd
