// (8) Neighbour sampling: the GPU form of PyG's NeighborLoader(num_neighbors=[k_1..k_L]) with replace=False,
// directed=True, over the raw destination-sorted CSR (gnnfd_csr_build, flags = 0).  Contract: include/gnnfd_b200.h (8).
//
// One call samples one batch.  The frontier of every hop is a contiguous range of local ids (the nodes new in the previous
// hop), so nothing but a few device scalars travels between hops; kernels are launched over host-side bounds and read the
// actual sizes from those scalars.  Per hop:
//   1. exclusive scan of min(d, k) over the frontier -> the edge offset of every frontier node (and the hop's edge count);
//   2. one warp per frontier node emits its edges: all positions (k == -1 or d <= k), else Floyd's algorithm -- in
//      registers, one chosen position per lane, for k <= 32; through the node's own output slots for larger k -- then the
//      chosen positions in ascending order; the global source goes to edge_index[0] for the moment;
//   3. deduplication of the new sources in first-appearance order: every edge whose source has no local id yet does
//      atomicMin(node_map[s], INT_MIN + edge position), so node_map[s] ends up holding the claim of the FIRST edge of s;
//      a flag scan over the edges (flag = this edge holds the claim) then gives the new id n_prev + rank.  The ids depend
//      only on the edge order, not on the scheduling;
//   4. edge_index[0] = node_map[global source].
// The reset at the end writes -1 to node_map[n_id[i]] for the sampled nodes only.
#include "common.cuh"
#include "gat_common.cuh"
#include "scan.cuh"

#include <climits>

namespace gnnfd {

namespace {

constexpr uint64_t GOLDEN = 0x9E3779B97F4A7C15ull;
constexpr int REG_K = 32;                 // Floyd in registers (one chosen position per lane) up to this fanout
constexpr int EMIT_WARPS = 8;
constexpr int MAX_HOPS = 64;

enum : uint32_t { ERR_RANGE = 1, ERR_DUP = 2, ERR_EDGE_CAP = 4, ERR_NODE_CAP = 8 };

// device scalars shared by the kernels of one call
struct Meta {
    uint32_t err;
    uint32_t front_begin, front_size;   // frontier of the current hop: local ids [front_begin, front_begin + front_size)
    uint32_t new_begin;                 // first local id of the nodes new in the current hop
    uint32_t ebase;                     // first output edge of the current hop
    uint32_t m_cur, n_cur;              // edges / new nodes of the current hop (scan totals)
    uint32_t pad_;
    // followed by hist[0..2L]: num_sampled_nodes [B, n_1..n_L], then num_sampled_edges [m_1..m_L]
};
__device__ __forceinline__ uint32_t* hist_of(Meta* m) { return reinterpret_cast<uint32_t*>(m + 1); }

// the draw of step i of Floyd's algorithm for node v: U_i(j) = mulhi64(w, j+1), uniform on [0, j]
__device__ __forceinline__ uint32_t floyd_draw(uint64_t seed, uint32_t v, uint32_t i, uint32_t j)
{
    const uint64_t w = KeepMask::mix(seed + GOLDEN * (2ull * ((uint64_t(v) << 32) | i) + 1ull));
    return uint32_t(__umul64hi(w, uint64_t(j) + 1ull));
}

__global__ void register_seeds(const int64_t* __restrict__ seeds, int64_t B, int64_t N, int32_t* __restrict__ node_map,
                               int64_t* __restrict__ n_id, Meta* meta)
{
    const int64_t t0 = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
    if (t0 == 0) {
        meta->front_begin = 0;
        meta->front_size = uint32_t(B);
        meta->new_begin = uint32_t(B);
        hist_of(meta)[0] = uint32_t(B);
    }
    for (int64_t i = t0; i < B; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t v = seeds[i];
        n_id[i] = v;
        if (v < 0 || v >= N) {
            atomicOr(&meta->err, ERR_RANGE);
            continue;
        }
        if (atomicCAS(&node_map[v], -1, int32_t(i)) != -1) atomicOr(&meta->err, ERR_DUP);
    }
}

// hop step 1: number of edges each frontier node contributes; 0 for everything once an error is flagged (the frontier
// may then hold ids outside [0, N))
struct HopCount {
    const int32_t* rowptr;
    const int64_t* n_id;
    const Meta* meta;
    int32_t k;
    __device__ uint32_t operator()(int64_t i) const
    {
        if (meta->err != 0 || i >= meta->front_size) return 0u;
        const int64_t v = n_id[meta->front_begin + i];
        const uint32_t d = uint32_t(rowptr[v + 1] - rowptr[v]);
        return (k < 0 || d <= uint32_t(k)) ? d : uint32_t(k);
    }
};
struct StoreOffset {
    uint32_t* edge_start;
    __device__ void operator()(int64_t i, uint32_t, uint32_t ex) const { edge_start[i] = ex; }
};

// single thread, after the count scan: the hop's edge count, checked against the capacity (all or nothing)
__global__ void hop_begin(Meta* meta, int64_t edge_cap)
{
    uint32_t m = meta->m_cur;
    if (meta->err != 0) {
        m = 0;
    } else if (uint64_t(meta->ebase) + m > uint64_t(edge_cap)) {
        meta->err |= ERR_EDGE_CAP;
        m = 0;
    }
    meta->m_cur = m;
}

struct EdgeOut {
    const int32_t* col;
    const int32_t* eid;
    int64_t* src;       // edge_index[0]: the global source until step 4
    int64_t* dst;       // edge_index[1]
    int64_t* e_id;
    __device__ __forceinline__ void put(int64_t slot, int32_t e, int64_t dst_local) const
    {
        src[slot] = col[e];
        e_id[slot] = eid[e];
        dst[slot] = dst_local;
    }
};

// hop step 2: one warp per frontier node
__global__ void __launch_bounds__(EMIT_WARPS * 32)
emit_edges(const int32_t* __restrict__ rowptr, const int64_t* __restrict__ n_id, const uint32_t* __restrict__ edge_start,
           int64_t n_front_bound, const Meta* meta, int32_t k, uint64_t seed, EdgeOut out)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
    if (w >= n_front_bound || meta->m_cur == 0 || w >= meta->front_size) return;
    const int64_t dst_local = int64_t(meta->front_begin) + w;
    const int64_t vv = n_id[dst_local];
    const uint32_t v = uint32_t(vv);
    const int32_t row0 = rowptr[vv];
    const uint32_t d = uint32_t(rowptr[vv + 1] - row0);
    const int64_t base = int64_t(meta->ebase) + edge_start[w];

    if (k < 0 || d <= uint32_t(k)) {
        for (uint32_t p = lane; p < d; p += 32) out.put(base + p, row0 + int32_t(p), dst_local);
        return;
    }
    const uint32_t kk = uint32_t(k);
    if (kk <= REG_K) {
        // lane i draws t_i; the steps then resolve in order: chosen_i = (t_i among chosen_0..i-1) ? j_i : t_i
        const uint32_t t = lane < kk ? floyd_draw(seed, v, lane, d - kk + lane) : 0u;
        uint32_t chosen = 0xffffffffu;
        for (uint32_t i = 0; i < kk; ++i) {
            const uint32_t ti = __shfl_sync(FULL, t, i);
            const unsigned hit = __ballot_sync(FULL, lane < int(i) && chosen == ti);
            if (lane == int(i)) chosen = hit ? d - kk + i : ti;
        }
        // the positions are distinct: the rank of a lane's position among the k is its output slot
        uint32_t rank = 0;
        for (int l = 0; l < REG_K; ++l) {
            const uint32_t c = __shfl_sync(FULL, chosen, l);
            rank += (uint32_t(l) < kk && c < chosen) ? 1u : 0u;
        }
        if (uint32_t(lane) < kk) out.put(base + rank, row0 + int32_t(chosen), dst_local);
        return;
    }
    // large k: the chosen positions are staged in the node's own e_id slots, their sorted order in its src slots.  Each Floyd
    // step is committed by lane 0 through global memory and the ranking reads all k entries per position: O(k^2 / 32) per
    // node and serial per warp -- correct for any k, fast only for the small fanouts above
    int64_t* chosen = out.e_id + base;
    for (uint32_t i = 0; i < kk; ++i) {
        const uint32_t j = d - kk + i;
        const uint32_t ti = floyd_draw(seed, v, i, j);
        bool found = false;
        for (uint32_t q = lane; q < i; q += 32) found |= chosen[q] == int64_t(ti);
        found = __any_sync(FULL, found);
        if (lane == 0) chosen[i] = found ? j : ti;
        __syncwarp();
    }
    for (uint32_t q = lane; q < kk; q += 32) {
        const int64_t c = chosen[q];
        uint32_t rank = 0;
        for (uint32_t r = 0; r < kk; ++r) rank += chosen[r] < c ? 1u : 0u;
        out.src[base + rank] = c;
    }
    __syncwarp();
    for (uint32_t r = lane; r < kk; r += 32) out.put(base + r, row0 + int32_t(out.src[base + r]), dst_local);
}

// hop step 3a: the first edge of every source without a local id claims it (smallest edge position wins)
__global__ void claim_sources(const int64_t* __restrict__ src, int64_t m_bound, const Meta* meta, int32_t* node_map)
{
    const uint32_t m = meta->m_cur, eb = meta->ebase;
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < m_bound && e < m; e += int64_t(gridDim.x) * blockDim.x) {
        const int64_t s = src[eb + e];
        if (node_map[s] < 0) atomicMin(&node_map[s], INT_MIN + int32_t(e));
    }
}

// hop step 3b: flag = this edge holds its source's claim; the claimer assigns the new local id
struct ClaimFlag {
    const int64_t* src;
    const int32_t* node_map;
    const Meta* meta;
    __device__ uint32_t operator()(int64_t e) const
    {
        if (e >= meta->m_cur) return 0u;
        const int64_t s = src[meta->ebase + e];
        return *(volatile const int32_t*)&node_map[s] == INT_MIN + int32_t(e) ? 1u : 0u;
    }
};
struct AssignId {
    const int64_t* src;
    int32_t* node_map;
    int64_t* n_id;
    Meta* meta;
    int64_t node_cap;
    __device__ void operator()(int64_t e, uint32_t flag, uint32_t ex) const
    {
        if (!flag) return;
        const int64_t s = src[meta->ebase + e];
        const int64_t pos = int64_t(meta->new_begin) + ex;
        if (pos < node_cap) {
            node_map[s] = int32_t(pos);
            n_id[pos] = s;
        } else {                               // no slot: release the claim so that node_map stays restorable
            node_map[s] = -1;
            atomicOr(&meta->err, ERR_NODE_CAP);
        }
    }
};

// hop step 4: local source ids
__global__ void localize_sources(int64_t* __restrict__ src, int64_t m_bound, const Meta* meta,
                                 const int32_t* __restrict__ node_map)
{
    const uint32_t m = meta->m_cur, eb = meta->ebase;
    for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < m_bound && e < m; e += int64_t(gridDim.x) * blockDim.x)
        src[eb + e] = node_map[src[eb + e]];
}

// single thread: the new nodes of this hop become the next frontier
__global__ void hop_end(Meta* meta, int hop, int n_hops)
{
    uint32_t* hist = hist_of(meta);
    hist[hop] = meta->n_cur;
    hist[n_hops + hop] = meta->m_cur;
    meta->front_begin = meta->new_begin;
    meta->front_size = meta->n_cur;
    meta->new_begin += meta->n_cur;
    meta->ebase += meta->m_cur;
}

__global__ void reset_node_map(const int64_t* __restrict__ n_id, int64_t node_cap, int64_t N, const Meta* meta,
                               int32_t* __restrict__ node_map)
{
    const int64_t n = meta->new_begin < node_cap ? int64_t(meta->new_begin) : node_cap;
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t v = n_id[i];
        if (v >= 0 && v < N) node_map[v] = -1;
    }
}

unsigned grid_for(int64_t n, int threads)
{
    int64_t g = (n + threads - 1) / threads;
    const int64_t cap = int64_t(sm_count()) * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

struct SampleWs {
    Meta* meta;
    uint32_t* edge_start;
    uint32_t* block_sums;
    size_t bytes;
};
SampleWs carve_sample(void* ws, int64_t node_cap, int64_t edge_cap, int32_t n_hops)
{
    const int64_t mx = node_cap > edge_cap ? node_cap : edge_cap;
    SampleWs w{};
    char* p = reinterpret_cast<char*>(ws);
    char* p0 = p;
    w.meta = reinterpret_cast<Meta*>(carve<uint32_t>(p, sizeof(Meta) / 4 + 2 * size_t(n_hops) + 1));
    w.edge_start = carve<uint32_t>(p, size_t(node_cap) + 1);
    w.block_sums = carve<uint32_t>(p, size_t((mx + SC_TILE - 1) / SC_TILE) + 1);
    w.bytes = size_t(p - p0) + 256;
    return w;
}

}  // namespace

}  // namespace gnnfd

using namespace gnnfd;

extern "C" {

int gnnfd_sample_workspace_bytes(int64_t node_cap, int64_t edge_cap, int32_t n_hops, size_t* bytes)
{
    GNNFD_REQUIRE(bytes != nullptr, GNNFD_ERR_ARG, "sample_workspace_bytes: bytes is NULL");
    GNNFD_REQUIRE(node_cap >= 0 && edge_cap >= 0 && n_hops >= 0, GNNFD_ERR_ARG, "sample_workspace_bytes: negative size");
    GNNFD_REQUIRE(node_cap < (int64_t(1) << 31) && edge_cap < (int64_t(1) << 31), GNNFD_ERR_RANGE,
                  "sample_workspace_bytes: caps must fit int32");
    *bytes = carve_sample(nullptr, node_cap, edge_cap, n_hops).bytes;
    return GNNFD_OK;
}

int gnnfd_neighbor_sample(const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t N, const int64_t* seeds,
                          int64_t n_seeds, const int32_t* fanouts_host, int32_t n_hops, uint64_t seed, int32_t* node_map,
                          int64_t* n_id, int64_t node_cap, int64_t* edge_index, int64_t ld_edge, int64_t* e_id,
                          int64_t edge_cap, int64_t* counts_host, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    GNNFD_REQUIRE(N >= 0 && N < (int64_t(1) << 31) && n_seeds >= 0 && n_hops >= 0 && n_hops <= MAX_HOPS, GNNFD_ERR_ARG,
                  "neighbor_sample: bad sizes (at most %d hops)", MAX_HOPS);
    GNNFD_REQUIRE(counts_host && (n_hops == 0 || fanouts_host), GNNFD_ERR_ARG, "neighbor_sample: NULL host argument");
    for (int32_t l = 0; l < n_hops; ++l)
        GNNFD_REQUIRE(fanouts_host[l] >= -1, GNNFD_ERR_ARG, "neighbor_sample: fanout %d of hop %d is < -1",
                      fanouts_host[l], l + 1);
    GNNFD_REQUIRE(node_cap >= n_seeds, GNNFD_ERR_WORKSPACE, "neighbor_sample: node_cap %lld < %lld seeds",
                  (long long)node_cap, (long long)n_seeds);
    GNNFD_REQUIRE(ld_edge >= edge_cap, GNNFD_ERR_ARG, "neighbor_sample: ld_edge < edge_cap");
    GNNFD_REQUIRE(rowptr && (n_seeds == 0 || (seeds && n_id && node_map)) && (edge_cap == 0 || (col && eid && edge_index && e_id)),
                  GNNFD_ERR_ARG, "neighbor_sample: NULL device argument");
    size_t need = 0;
    int rc = gnnfd_sample_workspace_bytes(node_cap, edge_cap, n_hops, &need);
    if (rc) return rc;
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "neighbor_sample: workspace %zu < %zu", ws_bytes, need);
    SampleWs w = carve_sample(ws, node_cap, edge_cap, n_hops);
    const size_t meta_bytes = sizeof(Meta) + sizeof(uint32_t) * size_t(2 * n_hops + 1);

    GNNFD_CUDA(cudaMemsetAsync(w.meta, 0, meta_bytes, st));
    register_seeds<<<grid_for(n_seeds > 0 ? n_seeds : 1, 256), 256, 0, st>>>(seeds, n_seeds, N, node_map, n_id, w.meta);
    g_launches += 1;
    GNNFD_LAUNCH_CHECK();

    EdgeOut out{col, eid, edge_index, edge_index + ld_edge, e_id};
    int64_t front_bound = n_seeds;            // host bounds of the frontier and of the hop's edges (launch sizes)
    for (int32_t l = 0; l < n_hops; ++l) {
        const int32_t k = fanouts_host[l];
        int64_t m_bound = k < 0 ? edge_cap : front_bound * int64_t(k);
        if (m_bound > edge_cap) m_bound = edge_cap;
        if (front_bound == 0) m_bound = 0;
        rc = exclusive_scan<uint32_t>(HopCount{rowptr, n_id, w.meta, k}, StoreOffset{w.edge_start}, front_bound,
                                      w.block_sums, &w.meta->m_cur, st);
        if (rc) return rc;
        hop_begin<<<1, 1, 0, st>>>(w.meta, edge_cap);
        g_launches += 1;
        if (front_bound > 0 && m_bound > 0) {
            const int64_t blocks = (front_bound + EMIT_WARPS - 1) / EMIT_WARPS;
            emit_edges<<<(unsigned)blocks, EMIT_WARPS * 32, 0, st>>>(rowptr, n_id, w.edge_start, front_bound, w.meta, k,
                                                                     seed, out);
            claim_sources<<<grid_for(m_bound, 256), 256, 0, st>>>(edge_index, m_bound, w.meta, node_map);
            g_launches += 2;
            GNNFD_LAUNCH_CHECK();
        }
        rc = exclusive_scan<uint32_t>(ClaimFlag{edge_index, node_map, w.meta},
                                      AssignId{edge_index, node_map, n_id, w.meta, node_cap}, m_bound, w.block_sums,
                                      &w.meta->n_cur, st);
        if (rc) return rc;
        if (m_bound > 0) {
            localize_sources<<<grid_for(m_bound, 256), 256, 0, st>>>(edge_index, m_bound, w.meta, node_map);
            g_launches += 1;
        }
        hop_end<<<1, 1, 0, st>>>(w.meta, l + 1, n_hops);
        g_launches += 1;
        GNNFD_LAUNCH_CHECK();
        front_bound = m_bound < node_cap ? m_bound : node_cap;
    }
    if (node_cap > 0) {
        reset_node_map<<<grid_for(node_cap, 256), 256, 0, st>>>(n_id, node_cap, N, w.meta, node_map);
        g_launches += 1;
        GNNFD_LAUNCH_CHECK();
    }

    uint32_t host[sizeof(Meta) / 4 + 2 * MAX_HOPS + 1];
    GNNFD_CUDA(cudaMemcpyAsync(host, w.meta, meta_bytes, cudaMemcpyDeviceToHost, st));
    GNNFD_CUDA(cudaStreamSynchronize(st));
    const Meta* hm = reinterpret_cast<const Meta*>(host);
    const uint32_t* hist = host + sizeof(Meta) / 4;
    GNNFD_REQUIRE(!(hm->err & ERR_RANGE), GNNFD_ERR_RANGE, "neighbor_sample: a seed is outside [0, %lld)", (long long)N);
    GNNFD_REQUIRE(!(hm->err & ERR_DUP), GNNFD_ERR_ARG, "neighbor_sample: duplicate seeds");
    GNNFD_REQUIRE(!(hm->err & (ERR_EDGE_CAP | ERR_NODE_CAP)), GNNFD_ERR_WORKSPACE,
                  "neighbor_sample: the sample exceeds node_cap %lld / edge_cap %lld", (long long)node_cap,
                  (long long)edge_cap);
    int64_t n_tot = 0, m_tot = 0;
    for (int32_t l = 0; l <= n_hops; ++l) {
        counts_host[2 + l] = hist[l];
        n_tot += hist[l];
    }
    for (int32_t l = 1; l <= n_hops; ++l) {
        counts_host[2 + n_hops + l] = hist[n_hops + l];
        m_tot += hist[n_hops + l];
    }
    counts_host[0] = n_tot;
    counts_host[1] = m_tot;
    return GNNFD_OK;
}

}  // extern "C"
