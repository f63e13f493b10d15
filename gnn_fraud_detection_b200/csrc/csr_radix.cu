// (1) edge_index -> destination-sorted CSR (+ source-sorted CSC twin) and hub plans.
//
// Replaces, bit-exactly, what PyG's GATConv.forward does to edge_index on every call at the reference's
// call sites (src/models/gat.py:80, src/models/tgn.py:94): remove_self_loops (order-preserving mask),
// add_self_loops (arange(N) appended), and the destination ordering that torch.sort(dst', stable=True)
// gives.  Built from: an order-preserving stream compaction (three-phase scan), a stable LSD radix sort
// (8 bits per pass, warp match_any ranking so equal keys keep their input order), and boundary fills
// for the row pointers.  All index work is int32 inside; the caller-facing edge_index stays int64.
#include "common.cuh"
#include "scan.cuh"

#include <atomic>
#include <cstdarg>

namespace gnnfd {

// ---- error + launch counter -------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
std::atomic<long long> g_launches{0};
const uint64_t* g_dropout_seed_src = nullptr;

// ---- self-loop rewrite ----------------------------------------------------------------------------
struct KeepFlag {
    const int64_t* src;
    const int64_t* dst;
    int64_t N;
    int drop_loops;
    int* err;
    __device__ uint32_t operator()(int64_t e) const
    {
        int64_t s = src[e], d = dst[e];
        if (s < 0 || s >= N || d < 0 || d >= N) {
            *err = 1;
            return 0;
        }
        return (drop_loops && s == d) ? 0u : 1u;
    }
};
struct CompactEdge {
    const int64_t* src;
    const int64_t* dst;
    uint32_t* key;   // dst'
    int32_t* srcc;   // src'
    __device__ void operator()(int64_t e, uint32_t keep, uint32_t pos) const
    {
        if (keep) {
            key[pos] = (uint32_t)dst[e];
            srcc[pos] = (int32_t)src[e];
        }
    }
};
__global__ void append_loops(uint32_t* key, int32_t* srcc, const uint32_t* Ef_dev, int64_t N)
{
    const uint32_t Ef = *Ef_dev;
    for (int64_t n = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; n < N; n += int64_t(gridDim.x) * blockDim.x) {
        key[Ef + n] = (uint32_t)n;
        srcc[Ef + n] = (int32_t)n;
    }
}

// ---- stable LSD radix sort, 8 bits per pass -------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ROUNDS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ROUNDS;  // 4096 keys per block, 512 consecutive keys per warp
constexpr int RADIX = 256;

__global__ void __launch_bounds__(RS_THREADS)
radix_hist(const uint32_t* __restrict__ keys, int64_t n, int shift, uint32_t* __restrict__ counts, int nblocks)
{
    __shared__ uint32_t hist[RADIX];
    hist[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = int64_t(blockIdx.x) * RS_TILE;
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
        int64_t i = base + r * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&hist[(keys[i] >> shift) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    counts[int64_t(threadIdx.x) * nblocks + blockIdx.x] = hist[threadIdx.x];  // digit-major for the scan
}

struct LoadU32 {
    const uint32_t* p;
    __device__ uint32_t operator()(int64_t i) const { return p[i]; }
};
struct StoreExcl {
    uint32_t* p;
    __device__ void operator()(int64_t i, uint32_t, uint32_t ex) const { p[i] = ex; }
};

// Scatter pass.  A thread knows the final slot of each of its keys (global base of (digit, block) + rank inside the tile), but
// writing it directly means 4-byte stores to ~256 open streams per block: every store dirties a 32-byte sector on its own.
// So the tile is first reordered in shared memory by tile-local rank (the same stable order), then written out in that
// order: consecutive threads then hold consecutive slots of one digit run, and a run (16 keys on average) leaves as full
// sectors.  The slots are identical to the direct scatter, bit for bit.
__global__ void __launch_bounds__(RS_THREADS)
radix_scatter(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
              uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n, int shift,
              const uint32_t* __restrict__ offsets, int nblocks)
{
    __shared__ uint32_t warp_cnt[RS_WARPS][RADIX];
    __shared__ uint32_t base_off[RADIX];      // global slot of the tile's first key with digit d
    __shared__ uint32_t dig_start[RADIX];     // tile-local slot of the tile's first key with digit d
    __shared__ uint32_t scan_w[RS_WARPS];
    __shared__ uint32_t sk[RS_TILE], sv[RS_TILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * RADIX; i += RS_THREADS) (&warp_cnt[0][0])[i] = 0;
    __syncthreads();

    // warp w owns the 512 consecutive keys [w*512, (w+1)*512) of the tile; round r = 32 consecutive keys
    const int64_t tile0 = int64_t(blockIdx.x) * RS_TILE;
    const int64_t wbase = tile0 + warp * (RS_ROUNDS * 32);
    uint32_t key[RS_ROUNDS], rank[RS_ROUNDS];
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        const bool valid = i < n;
        key[r] = valid ? keys_in[i] : 0u;
        const uint32_t d = valid ? ((key[r] >> shift) & (RADIX - 1)) : 0xFFFFu;
        const uint32_t peers = __match_any_sync(FULL, d);
        const int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (valid && lane == leader) {
            old = warp_cnt[warp][d];
            warp_cnt[warp][d] = old + __popc(peers);
        }
        old = __shfl_sync(FULL, old, leader);
        rank[r] = old + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    {   // exclusive prefix of each digit over the warps of this block, the block's global base, and the exclusive prefix
        // over the digits of the tile histogram (thread d owns digit d)
        const int d = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) {
            uint32_t c = warp_cnt[w][d];
            warp_cnt[w][d] = run;
            run += c;
        }
        base_off[d] = offsets[int64_t(d) * nblocks + blockIdx.x];
        uint32_t inc = run;                              // inclusive scan of the 256 digit counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) scan_w[warp] = inc;
        __syncthreads();
        uint32_t before = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) before += (w < warp) ? scan_w[w] : 0u;
        dig_start[d] = before + inc - run;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        if (i < n) {
            const uint32_t d = (key[r] >> shift) & (RADIX - 1);
            const uint32_t lp = dig_start[d] + warp_cnt[warp][d] + rank[r];
            sk[lp] = key[r];
            sv[lp] = vals_in ? vals_in[i] : (uint32_t)i;
        }
    }
    __syncthreads();
    const int tile_n = int(n - tile0 < RS_TILE ? n - tile0 : RS_TILE);
    for (int i = threadIdx.x; i < tile_n; i += RS_THREADS) {
        const uint32_t k = sk[i];
        const uint32_t d = (k >> shift) & (RADIX - 1);
        const uint32_t pos = base_off[d] + (uint32_t(i) - dig_start[d]);
        keys_out[pos] = k;
        vals_out[pos] = sv[i];
    }
}

// sorts n (key,val) pairs; vals_in==nullptr means identity.  Result lands in (kA,vA) or (kB,vB);
// returns which through *res_k / *res_v.
static int radix_sort_pairs(const uint32_t* keys_in, int64_t n, int key_bits, uint32_t* kA, uint32_t* vA,
                            uint32_t* kB, uint32_t* vB, uint32_t* counts, uint32_t* block_sums,
                            uint32_t* total_dev, const uint32_t** res_k, const uint32_t** res_v,
                            cudaStream_t st, const uint32_t* vals_in = nullptr)
{
    const int nblocks = (int)((n + RS_TILE - 1) / RS_TILE);
    int passes = (key_bits + 7) / 8;
    if (passes < 1) passes = 1;
    const uint32_t* kin = keys_in;
    const uint32_t* vin = vals_in;
    uint32_t* kout = kA;
    uint32_t* vout = vA;
    for (int p = 0; p < passes; ++p) {
        const int shift = 8 * p;
        radix_hist<<<nblocks, RS_THREADS, 0, st>>>(kin, n, shift, counts, nblocks);
        g_launches += 1;
        int rc = exclusive_scan<uint32_t>(LoadU32{counts}, StoreExcl{counts}, int64_t(RADIX) * nblocks,
                                          block_sums, total_dev, st);
        if (rc) return rc;
        radix_scatter<<<nblocks, RS_THREADS, 0, st>>>(kin, vin, kout, vout, n, shift, counts, nblocks);
        g_launches += 1;
        GNNFD_LAUNCH_CHECK();
        kin = kout;
        vin = vout;
        if (kout == kA) { kout = kB; vout = vB; } else { kout = kA; vout = vA; }
    }
    *res_k = kin;
    *res_v = vin;
    return GNNFD_OK;
}

// ---- finalisation -----------------------------------------------------------------------------------
// ptr[r] = first position e with key[e] >= r  (keys sorted ascending); handles empty rows.
__global__ void fill_ptr(const uint32_t* __restrict__ key, int64_t n, int64_t n_rows, int32_t* __restrict__ ptr)
{
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < n; e += int64_t(gridDim.x) * blockDim.x) {
        const int64_t k = key[e];
        const int64_t kp = e > 0 ? int64_t(key[e - 1]) : -1;
        for (int64_t r = kp + 1; r <= k; ++r) ptr[r] = (int32_t)e;
        if (e == n - 1)
            for (int64_t r = k + 1; r <= n_rows; ++r) ptr[r] = (int32_t)n;
    }
}
__global__ void finalize_csr(const uint32_t* __restrict__ key, const uint32_t* __restrict__ val,
                             const int32_t* __restrict__ srcc, int64_t n, int32_t* __restrict__ col,
                             int32_t* __restrict__ perm, int32_t* __restrict__ dst_sorted)
{
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < n; e += int64_t(gridDim.x) * blockDim.x) {
        const uint32_t p = val[e];
        perm[e] = (int32_t)p;
        col[e] = srcc[p];
        if (dst_sorted) dst_sorted[e] = (int32_t)key[e];
    }
}
// ORDER_DST_SRC, between the two sorts: the destination of every source-sorted edge becomes the key of the second sort
__global__ void gather_keys(const uint32_t* __restrict__ key_of, const uint32_t* __restrict__ idx, int64_t n,
                            uint32_t* __restrict__ out)
{
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < n; e += int64_t(gridDim.x) * blockDim.x)
        out[e] = key_of[idx[e]];
}
__global__ void finalize_csc(const uint32_t* __restrict__ val, const int32_t* __restrict__ dst_sorted, int64_t n,
                             int32_t* __restrict__ csc_row, int32_t* __restrict__ csc_eid)
{
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < n; e += int64_t(gridDim.x) * blockDim.x) {
        const uint32_t p = val[e];
        csc_eid[e] = (int32_t)p;
        csc_row[e] = dst_sorted[p];
    }
}

static int bits_for(int64_t n)
{
    int b = 1;
    while ((int64_t(1) << b) < n) ++b;
    return b;
}
static unsigned grid_for(int64_t n, int threads)
{
    int64_t g = (n + threads - 1) / threads;
    int64_t cap = int64_t(sm_count()) * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

struct CsrWs {
    int32_t* srcc;
    uint32_t *kA, *vA, *kB, *vB;
    int32_t* dst_sorted;
    uint32_t* counts;
    uint32_t* block_sums;
    uint32_t* scalars;  // [0]=Ef, [1]=err, [2]=scan total scratch
    size_t bytes;
};
static CsrWs carve_csr(void* ws, int64_t N, int64_t E, int flags)
{
    const int64_t cap = E + ((flags & GNNFD_ADD_SELF_LOOPS) ? N : 0);
    const int64_t nblocks = (cap + RS_TILE - 1) / RS_TILE + 1;
    const int64_t n_counts = nblocks * RADIX;
    const int64_t n_bs = (((E > n_counts ? E : n_counts) + SC_TILE - 1) / SC_TILE) + 1;
    CsrWs w{};
    char* p = reinterpret_cast<char*>(ws);
    char* p0 = p;
    w.srcc = carve<int32_t>(p, cap + 1);
    w.kA = carve<uint32_t>(p, cap + 1);
    w.vA = carve<uint32_t>(p, cap + 1);
    w.kB = carve<uint32_t>(p, cap + 1);
    w.vB = carve<uint32_t>(p, cap + 1);
    w.dst_sorted = carve<int32_t>(p, cap + 1);
    w.counts = carve<uint32_t>(p, n_counts);
    w.block_sums = carve<uint32_t>(p, n_bs);
    w.scalars = carve<uint32_t>(p, 8);
    w.bytes = size_t(p - p0) + 256;
    return w;
}

// ---- hub plan -----------------------------------------------------------------------------------------
struct HubValue {
    const int32_t* ptr;
    int32_t threshold, chunk;
    __device__ unsigned long long operator()(int64_t r) const
    {
        const int32_t deg = ptr[r + 1] - ptr[r];
        if (deg <= threshold) return 0ull;
        return (1ull << 32) | (unsigned long long)((deg + chunk - 1) / chunk);
    }
};
struct HubEmit {
    int32_t* hub_row;
    int32_t* hub_chunk_ptr;
    int32_t* chunk_hub;
    int64_t cap_hub, cap_chunk;
    __device__ void operator()(int64_t r, unsigned long long v, unsigned long long ex) const
    {
        if (!v) return;
        const int64_t slot = (int64_t)(ex >> 32);
        const int64_t c0 = (int64_t)(ex & 0xffffffffull);
        const int64_t nc = (int64_t)(v & 0xffffffffull);
        if (slot < cap_hub) {
            hub_row[slot] = (int32_t)r;
            hub_chunk_ptr[slot] = (int32_t)c0;
        }
        for (int64_t c = 0; c < nc; ++c)
            if (c0 + c < cap_chunk) chunk_hub[c0 + c] = (int32_t)slot;
    }
};

// ---- work-item plan ---------------------------------------------------------------------------------------
// cost(i) = ptr[i] + i*w;  item_start[t] = first row i with cost(i) >= t*target  (t = 0..n_items-1),
// item_start[n_items] = n_rows
__global__ void item_plan_kernel(const int32_t* __restrict__ ptr, int64_t n_rows, int32_t target, int32_t w,
                                 int32_t n_items, int32_t* __restrict__ item_start)
{
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i <= n_rows; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t cur = int64_t(ptr[i]) + i * w;
        const int64_t t0 = (i == 0) ? 0 : (int64_t(ptr[i - 1]) + (i - 1) * w) / target + 1;
        const int64_t t1 = cur / target;
        for (int64_t t = t0; t <= t1 && t < n_items; ++t) item_start[t] = (int32_t)i;
        if (i == n_rows) item_start[n_items] = (int32_t)n_rows;
    }
}

__global__ void invert_perm_kernel(const int32_t* __restrict__ perm, int64_t n, int32_t* __restrict__ inv)
{
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
        inv[perm[i]] = (int32_t)i;
}

}  // namespace gnnfd

using namespace gnnfd;

extern "C" {

const char* gnnfd_last_error(void) { return g_err; }
int gnnfd_abi_version(void) { return GNNFD_ABI_VERSION; }
void gnnfd_set_dropout_seed_source(const uint64_t* device_word) { gnnfd::g_dropout_seed_src = device_word; }
size_t gnnfd_sizeof_graph(void) { return sizeof(gnnfd_graph_t); }
size_t gnnfd_sizeof_hub_plan(void) { return sizeof(gnnfd_hub_plan_t); }
size_t gnnfd_sizeof_item_plan(void) { return sizeof(gnnfd_item_plan_t); }

int gnnfd_invert_perm(const int32_t* perm, int64_t n, int32_t* inv, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(n >= 0 && (n == 0 || (perm && inv)), GNNFD_ERR_ARG, "invert_perm: bad arguments");
    if (n == 0) return GNNFD_OK;
    invert_perm_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(perm, n, inv);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

int gnnfd_item_plan(const int32_t* ptr, int64_t n_rows, int64_t n_edges, int32_t target, int32_t row_weight,
                    int32_t* item_start, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(ptr && item_start, GNNFD_ERR_ARG, "item_plan: NULL array");
    GNNFD_REQUIRE(n_rows >= 0 && n_edges >= 0 && target >= 1 && row_weight >= 0, GNNFD_ERR_ARG, "item_plan: bad sizes");
    const int32_t n_items = (int32_t)((n_edges + n_rows * row_weight) / target + 1);
    item_plan_kernel<<<grid_for(n_rows + 1, 256), 256, 0, (cudaStream_t)stream>>>(ptr, n_rows, target, row_weight, n_items,
                                                                                  item_start);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}
int64_t gnnfd_launch_count(void) { return (int64_t)g_launches.load(); }
void gnnfd_launch_count_reset(void) { g_launches.store(0); }
int gnnfd_shutdown(void)
{
    g_dropout_seed_src = nullptr;
    g_launches.store(0);
    return GNNFD_OK;
}

int gnnfd_csr_workspace_bytes(int64_t N, int64_t E, int flags, size_t* bytes)
{
    GNNFD_REQUIRE(bytes != nullptr, GNNFD_ERR_ARG, "csr_workspace_bytes: bytes is NULL");
    GNNFD_REQUIRE(N >= 0 && E >= 0, GNNFD_ERR_ARG, "csr_workspace_bytes: negative N/E");
    GNNFD_REQUIRE(E + N < (int64_t(1) << 31) - RS_TILE, GNNFD_ERR_RANGE, "E + N = %lld does not fit int32 indices",
                  (long long)(E + N));
    *bytes = carve_csr(nullptr, N, E, flags).bytes;
    return GNNFD_OK;
}

int gnnfd_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int flags, int32_t* rowptr, int32_t* col,
                    int32_t* perm, int32_t* colptr, int32_t* csc_row, int32_t* csc_eid, int64_t* E_out_host,
                    void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    GNNFD_REQUIRE(N >= 0 && E >= 0, GNNFD_ERR_ARG, "csr_build: negative N/E");
    GNNFD_REQUIRE(E == 0 || edge_index, GNNFD_ERR_ARG, "csr_build: edge_index is NULL");
    GNNFD_REQUIRE(rowptr && E_out_host, GNNFD_ERR_ARG, "csr_build: rowptr/E_out_host is NULL");
    GNNFD_REQUIRE(E + N < (int64_t(1) << 31) - RS_TILE, GNNFD_ERR_RANGE, "E + N = %lld does not fit int32 indices",
                  (long long)(E + N));
    const bool loops = (flags & GNNFD_ADD_SELF_LOOPS) != 0;
    const bool want_csc = (flags & GNNFD_BUILD_CSC) != 0;
    GNNFD_REQUIRE(!want_csc || (colptr && (csc_row && csc_eid || E + (loops ? N : 0) == 0)), GNNFD_ERR_ARG,
                  "csr_build: BUILD_CSC needs colptr/csc_row/csc_eid");
    size_t need = 0;
    int rc = gnnfd_csr_workspace_bytes(N, E, flags, &need);
    if (rc) return rc;
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "csr_build: workspace %zu < %zu", ws_bytes, need);
    CsrWs w = carve_csr(ws, N, E, flags);

    GNNFD_CUDA(cudaMemsetAsync(w.scalars, 0, 8 * sizeof(uint32_t), st));
    // 1. order-preserving removal of self-loops (or plain narrowing copy), range check
    KeepFlag kf{edge_index, edge_index + E, N, loops ? 1 : 0, reinterpret_cast<int*>(w.scalars + 1)};
    CompactEdge ce{edge_index, edge_index + E, w.kA, w.srcc};
    rc = exclusive_scan<uint32_t>(kf, ce, E, w.block_sums, w.scalars + 0, st);
    if (rc) return rc;
    // 2. append one self-loop per node
    if (loops && N > 0) {
        append_loops<<<grid_for(N, 256), 256, 0, st>>>(w.kA, w.srcc, w.scalars + 0, N);
        g_launches += 1;
        GNNFD_LAUNCH_CHECK();
    }
    uint32_t host_sc[2] = {0, 0};
    GNNFD_CUDA(cudaMemcpyAsync(host_sc, w.scalars, sizeof(host_sc), cudaMemcpyDeviceToHost, st));
    GNNFD_CUDA(cudaStreamSynchronize(st));
    GNNFD_REQUIRE(host_sc[1] == 0, GNNFD_ERR_RANGE, "csr_build: edge_index has an entry outside [0, %lld)", (long long)N);
    const int64_t Ep = int64_t(host_sc[0]) + (loops ? N : 0);
    *E_out_host = Ep;

    GNNFD_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * size_t(N + 1), st));
    if (want_csc) GNNFD_CUDA(cudaMemsetAsync(colptr, 0, sizeof(int32_t) * size_t(N + 1), st));
    if (Ep == 0) return GNNFD_OK;
    GNNFD_REQUIRE(col && perm, GNNFD_ERR_ARG, "csr_build: col/perm is NULL");

    // 3. stable sort by destination; values = positions in edge_index'
    const int bits = bits_for(N);
    const uint32_t *rk = nullptr, *rv = nullptr;
    int32_t* dst_sorted_out = w.dst_sorted;
    if (flags & GNNFD_ORDER_DST_SRC) {
        // PyG sort_edge_index(sort_by_row=False): stable sort on (dst', src') = LSD over the two fields: first a stable sort
        // by source (values = positions in edge_index'), then a stable sort of THAT sequence by destination.  kA (the
        // destinations) must survive the first sort, so it ping-pongs between (kB, vB) and (dst_sorted, vA).
        uint32_t* dk = reinterpret_cast<uint32_t*>(w.dst_sorted);
        rc = radix_sort_pairs(reinterpret_cast<const uint32_t*>(w.srcc), Ep, bits, w.kB, w.vB, dk, w.vA, w.counts, w.block_sums,
                              w.scalars + 2, &rk, &rv, st);
        if (rc) return rc;
        uint32_t* k1 = const_cast<uint32_t*>(rk);      // the sorted sources are no longer needed: their buffer takes the new keys
        uint32_t* v1 = const_cast<uint32_t*>(rv);
        uint32_t* k2 = (k1 == w.kB) ? dk : w.kB;
        uint32_t* v2 = (v1 == w.vB) ? w.vA : w.vB;
        gather_keys<<<grid_for(Ep, 256), 256, 0, st>>>(w.kA, v1, Ep, k1);
        g_launches += 1;
        rc = radix_sort_pairs(k1, Ep, bits, k2, v2, k1, v1, w.counts, w.block_sums, w.scalars + 2, &rk, &rv, st, v1);
        if (rc) return rc;
        if (rk == dk) dst_sorted_out = nullptr;        // the sorted keys already sit in dst_sorted
    } else {
        // first pass reads kA and must not write it: run A -> B -> A ...
        rc = radix_sort_pairs(w.kA, Ep, bits, w.kB, w.vB, w.kA, w.vA, w.counts, w.block_sums, w.scalars + 2, &rk, &rv, st);
        if (rc) return rc;
    }
    finalize_csr<<<grid_for(Ep, 256), 256, 0, st>>>(rk, rv, w.srcc, Ep, col, perm, dst_sorted_out);
    fill_ptr<<<grid_for(Ep, 256), 256, 0, st>>>(rk, Ep, N, rowptr);
    g_launches += 2;
    GNNFD_LAUNCH_CHECK();

    // 4. source-major twin: stable sort of the CSR-ordered col array, values = CSR positions
    if (want_csc) {
        rc = radix_sort_pairs(reinterpret_cast<const uint32_t*>(col), Ep, bits, w.kA, w.vA, w.kB, w.vB, w.counts,
                              w.block_sums, w.scalars + 2, &rk, &rv, st);
        if (rc) return rc;
        finalize_csc<<<grid_for(Ep, 256), 256, 0, st>>>(rv, w.dst_sorted, Ep, csc_row, csc_eid);
        fill_ptr<<<grid_for(Ep, 256), 256, 0, st>>>(rk, Ep, N, colptr);
        g_launches += 2;
        GNNFD_LAUNCH_CHECK();
    }
    return GNNFD_OK;
}

// ---- snapshot / induced-subgraph builder (vectorised create_temporal_subgraph, src/data/dataset.py:198-240) -----
// Two order-preserving compactions on the scan machinery above: nodes whose time step is selected (ascending id,
// relabelled by the exclusive prefix sum of the selection flag), then edges with both endpoints selected (original
// order, endpoints relabelled).  HBM-bound integer work: reads time_steps (8 B/node) and edge_index (16 B/edge) once
// for the flags and once for the scatter.
struct NodeSel {
    const int64_t* ts;
    const uint8_t* table;
    int64_t n_table;
    int* err;
    __device__ uint32_t operator()(int64_t i) const
    {
        const int64_t t = ts[i];
        if (t < 0) {
            *err = 1;
            return 0;
        }
        return (t < n_table && table[t]) ? 1u : 0u;       // steps beyond the table are simply not selected
    }
};
struct NodeScatter {
    int64_t* node_ids;
    int64_t* relabel;      // optional int64 copy for the caller
    int32_t* relabel32;    // workspace: 4 B/node keeps the table the edge passes gather from inside L2
    uint8_t* sel;          // workspace: 1 B/node selection flag for the edge flag pass
    __device__ void operator()(int64_t i, uint32_t keep, uint32_t pos) const
    {
        const int32_t r = keep ? int32_t(pos) : -1;
        relabel32[i] = r;
        sel[i] = uint8_t(keep);
        if (relabel) relabel[i] = r;
        if (keep) node_ids[pos] = i;
    }
};
struct EdgeSel {
    const int64_t* src;
    const int64_t* dst;
    const uint8_t* sel;
    int64_t N;
    int* err;
    __device__ uint32_t operator()(int64_t e) const
    {
        const int64_t s = src[e], d = dst[e];
        if (s < 0 || s >= N || d < 0 || d >= N) {
            *err = 2;
            return 0;
        }
        return (sel[s] & sel[d]) ? 1u : 0u;
    }
};
struct EdgeScatter {
    const int64_t* src;
    const int64_t* dst;
    const int32_t* relabel32;
    int64_t* out_src;
    int64_t* out_dst;
    __device__ void operator()(int64_t e, uint32_t keep, uint32_t pos) const
    {
        if (keep) {
            out_src[pos] = relabel32[src[e]];
            out_dst[pos] = relabel32[dst[e]];
        }
    }
};

int gnnfd_subgraph_workspace_bytes(int64_t N, int64_t E, size_t* bytes)
{
    GNNFD_REQUIRE(bytes != nullptr && N >= 0 && E >= 0, GNNFD_ERR_ARG, "subgraph_workspace_bytes: bad args");
    const int64_t m = N > E ? N : E;
    *bytes = carve_bytes(8, 4) + carve_bytes(size_t((m + SC_TILE - 1) / SC_TILE + 2), 4) + carve_bytes(size_t(N), 4) +
             carve_bytes(size_t(N), 1) + 512;
    return GNNFD_OK;
}

int gnnfd_subgraph_build(const int64_t* time_steps, int64_t N, const uint8_t* step_selected, int64_t n_step_table,
                         const int64_t* edge_index, int64_t E, int64_t* node_ids, int64_t* relabel,
                         int64_t* sub_edge_index, int64_t ld_sub, int64_t* counts_host, void* ws, size_t ws_bytes,
                         gnnfd_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    GNNFD_REQUIRE(N >= 0 && E >= 0 && n_step_table >= 0, GNNFD_ERR_ARG, "subgraph_build: negative size");
    GNNFD_REQUIRE(N < (int64_t(1) << 31) && E < (int64_t(1) << 31), GNNFD_ERR_RANGE, "subgraph_build: N/E do not fit 31 bits");
    GNNFD_REQUIRE(counts_host != nullptr, GNNFD_ERR_ARG, "subgraph_build: counts_host is NULL");
    GNNFD_REQUIRE(N == 0 || (time_steps && step_selected && node_ids), GNNFD_ERR_ARG, "subgraph_build: NULL node argument");
    GNNFD_REQUIRE(E == 0 || (edge_index && sub_edge_index && ld_sub >= E), GNNFD_ERR_ARG,
                  "subgraph_build: NULL edge argument or ld_sub < E");
    size_t need = 0;
    int rc = gnnfd_subgraph_workspace_bytes(N, E, &need);
    if (rc) return rc;
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "subgraph_build: workspace %zu < %zu", ws_bytes, need);
    char* p = reinterpret_cast<char*>(ws);
    uint32_t* scalars = carve<uint32_t>(p, 8);              // [0] n_sel, [1] m, [2] error flag
    const int64_t mx = N > E ? N : E;
    uint32_t* block_sums = carve<uint32_t>(p, size_t((mx + SC_TILE - 1) / SC_TILE + 2));
    int32_t* relabel32 = carve<int32_t>(p, size_t(N));
    uint8_t* sel = carve<uint8_t>(p, size_t(N));
    GNNFD_CUDA(cudaMemsetAsync(scalars, 0, 8 * sizeof(uint32_t), st));
    int* err = reinterpret_cast<int*>(scalars + 2);
    NodeSel ns{time_steps, step_selected, n_step_table, err};
    NodeScatter nsc{node_ids, relabel, relabel32, sel};
    rc = exclusive_scan<uint32_t>(ns, nsc, N, block_sums, scalars + 0, st);
    if (rc) return rc;
    EdgeSel es{edge_index, edge_index + E, sel, N, err};
    EdgeScatter esc{edge_index, edge_index + E, relabel32, sub_edge_index, sub_edge_index + ld_sub};
    rc = exclusive_scan<uint32_t>(es, esc, E, block_sums, scalars + 1, st);
    if (rc) return rc;
    uint32_t host_sc[3] = {0, 0, 0};
    GNNFD_CUDA(cudaMemcpyAsync(host_sc, scalars, sizeof(host_sc), cudaMemcpyDeviceToHost, st));
    GNNFD_CUDA(cudaStreamSynchronize(st));
    GNNFD_REQUIRE(host_sc[2] != 1, GNNFD_ERR_RANGE, "subgraph_build: negative time step");
    GNNFD_REQUIRE(host_sc[2] != 2, GNNFD_ERR_RANGE, "subgraph_build: edge_index has an entry outside [0, %lld)", (long long)N);
    counts_host[0] = host_sc[0];
    counts_host[1] = host_sc[1];
    return GNNFD_OK;
}

int gnnfd_hub_plan_workspace_bytes(int64_t n_rows, size_t* bytes)
{
    GNNFD_REQUIRE(bytes != nullptr && n_rows >= 0, GNNFD_ERR_ARG, "hub_plan_workspace_bytes: bad args");
    *bytes = carve_bytes(size_t((n_rows + SC_TILE - 1) / SC_TILE + 2), 8) + 512;
    return GNNFD_OK;
}

int gnnfd_hub_plan(const int32_t* ptr, int64_t n_rows, int32_t threshold, int32_t chunk, int32_t* hub_row,
                   int32_t* hub_chunk_ptr, int32_t* chunk_hub, int64_t cap_hub, int64_t cap_chunk,
                   int64_t* counts_host, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    GNNFD_REQUIRE(counts_host, GNNFD_ERR_ARG, "hub_plan: counts_host is NULL");
    GNNFD_REQUIRE(threshold >= 32 && chunk >= 32 && chunk % 32 == 0, GNNFD_ERR_ARG,
                  "hub_plan: threshold/chunk must be >= 32 and chunk a multiple of 32");
    counts_host[0] = counts_host[1] = 0;
    if (n_rows == 0) return GNNFD_OK;
    GNNFD_REQUIRE(ptr && hub_row && hub_chunk_ptr && chunk_hub, GNNFD_ERR_ARG, "hub_plan: NULL array");
    size_t need = 0;
    gnnfd_hub_plan_workspace_bytes(n_rows, &need);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "hub_plan: workspace %zu < %zu", ws_bytes, need);
    char* p = reinterpret_cast<char*>(ws);
    unsigned long long* total = carve<unsigned long long>(p, 1);
    unsigned long long* bs = carve<unsigned long long>(p, size_t((n_rows + SC_TILE - 1) / SC_TILE + 1));
    int rc = exclusive_scan<unsigned long long>(HubValue{ptr, threshold, chunk},
                                                HubEmit{hub_row, hub_chunk_ptr, chunk_hub, cap_hub, cap_chunk},
                                                n_rows, bs, total, st);
    if (rc) return rc;
    unsigned long long h = 0;
    GNNFD_CUDA(cudaMemcpyAsync(&h, total, sizeof(h), cudaMemcpyDeviceToHost, st));
    GNNFD_CUDA(cudaStreamSynchronize(st));
    const int64_t n_hub = (int64_t)(h >> 32), n_chunk = (int64_t)(h & 0xffffffffull);
    GNNFD_REQUIRE(n_hub <= cap_hub && n_chunk <= cap_chunk, GNNFD_ERR_WORKSPACE,
                  "hub_plan: %lld hubs / %lld chunks exceed capacity %lld / %lld", (long long)n_hub,
                  (long long)n_chunk, (long long)cap_hub, (long long)cap_chunk);
    const int32_t last = (int32_t)n_chunk;
    GNNFD_CUDA(cudaMemcpyAsync(hub_chunk_ptr + n_hub, &last, sizeof(int32_t), cudaMemcpyHostToDevice, st));
    GNNFD_CUDA(cudaStreamSynchronize(st));
    counts_host[0] = n_hub;
    counts_host[1] = n_chunk;
    return GNNFD_OK;
}

}  // extern "C"
