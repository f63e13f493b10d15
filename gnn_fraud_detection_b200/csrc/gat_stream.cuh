// Warp-stream machinery shared by the forward and the dst-major backward kernels.
//
// One warp owns one edge-balanced work item (a run of whole destination rows, ~target edges) and walks it
// as a stream of chunks (<= 32 edges of one row).  The 2 KB (fp32) / 1 KB (bf16) source-feature rows are
// NOT loaded through registers: lane 0 hands each row to the bulk async-copy engine
// (cp.async.bulk global->shared, completion on an mbarrier), into a per-warp ring of R row slots, and the
// warp consumes the slots in order with conflict-free 128-bit shared loads.  Bytes in flight therefore
// live in shared memory (R x 2 KB per warp) instead of registers, and phase A of the NEXT chunk (index
// and logit gathers, softmax statistics) runs while the CURRENT chunk's rows are still landing.
#pragma once
#include "gat_common.cuh"

namespace gnnfd {

constexpr int ST_WARPS = 4;                 // warps (items) per CTA
constexpr int ST_THREADS = ST_WARPS * 32;

__device__ __forceinline__ uint32_t st_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void st_mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void st_mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t addr = st_smem_u32(bar);
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
        if (++spins > (1u << 26)) __trap();   // a protocol bug must not hang the GPU
    }
}
__device__ __forceinline__ void st_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     st_smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(st_smem_u32(bar))
                 : "memory");
}

template <class GE, int EXTRA = 0>
struct StreamGeo {
    static constexpr int ROW_BYTES = GE::D * int(sizeof(typename GE::XT));
    static constexpr int R = ROW_BYTES >= 2048 ? 5 : (ROW_BYTES >= 1024 ? 8 : 12);   // ring slots per warp
    static constexpr int RING_BYTES = R * ROW_BYTES;
    static constexpr int P_BYTES = 2 * 32 * GE::H * 4;        // two staging buffers of per-edge per-head floats
    static constexpr int J_BYTES = 2 * 32 * 4;
    static constexpr int BAR_BYTES = ((R * 8 + 15) / 16) * 16;
    static constexpr int EXTRA_BYTES = EXTRA;                 // kernel-specific per-warp scratch
    static constexpr int WARP_BYTES = ((RING_BYTES + P_BYTES + J_BYTES + BAR_BYTES + EXTRA + 127) / 128) * 128;
    static constexpr int CTA_BYTES = ST_WARPS * WARP_BYTES;
};

// CTAs per SM the stream kernels are compiled for (their __launch_bounds__).  Up to 2 KB rows four 4-warp CTAs share
// an SM; a 4 KB row (8 heads x 128 fp32) makes the ring alone 20 KB per warp, so at most two CTAs fit and each thread
// may use twice the registers -- which its 32 accumulators per lane need.
template <class GE>
constexpr int st_min_ctas()
{
    return GE::D * int(sizeof(typename GE::XT)) > 2048 ? 2 : 4;
}

// per-warp view of the dynamic shared memory
template <class GE, int EXTRA = 0>
struct WarpRing {
    using SG = StreamGeo<GE, EXTRA>;
    uint8_t* ring;
    uint8_t* extra;  // [EXTRA] bytes
    float* p_s;      // [2][32*H]
    int* j_s;        // [2][32]
    uint64_t* full;  // [R]
    int issued = 0, consumed = 0;

    __device__ __forceinline__ void init(uint8_t* base, int lane)
    {
        ring = base;
        p_s = reinterpret_cast<float*>(base + SG::RING_BYTES);
        j_s = reinterpret_cast<int*>(base + SG::RING_BYTES + SG::P_BYTES);
        full = reinterpret_cast<uint64_t*>(base + SG::RING_BYTES + SG::P_BYTES + SG::J_BYTES);
        extra = base + SG::RING_BYTES + SG::P_BYTES + SG::J_BYTES + SG::BAR_BYTES;
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < SG::R; ++i) st_mbar_init(&full[i], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }
    __device__ __forceinline__ bool has_room() const { return issued - consumed < SG::R; }
    // hand source row j to the copy engine (lane 0), all lanes track the counter
    __device__ __forceinline__ void issue(const typename GE::XT* __restrict__ xw, int j, int lane)
    {
        if (lane == 0) {
            const int slot = issued % SG::R;
            st_mbar_expect_tx(&full[slot], SG::ROW_BYTES);
            st_bulk_g2s(ring + slot * SG::ROW_BYTES, xw + int64_t(j) * GE::D, SG::ROW_BYTES, &full[slot]);
        }
        ++issued;
    }
    // wait for the oldest in-flight row; returns its slot base
    __device__ __forceinline__ const uint8_t* front()
    {
        const int slot = consumed % SG::R;
        st_mbar_wait(&full[slot], (consumed / SG::R) & 1);
        return ring + slot * SG::ROW_BYTES;
    }
    __device__ __forceinline__ void pop()
    {
        __syncwarp();     // every lane has read the slot before it can be refilled
        ++consumed;
    }
};

// one slot (VW elements) of a staged row
__device__ __forceinline__ void lds_slot(const uint8_t* row, int q, int lane, float (&v)[4])
{
    const float4 t = *reinterpret_cast<const float4*>(row + (lane + 32 * q) * 16);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void lds_slot(const uint8_t* row, int q, int lane, float (&v)[8])
{
    const uint4 t = *reinterpret_cast<const uint4*>(row + (lane + 32 * q) * 16);
    v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
    v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
    v[4] = __uint_as_float(t.z << 16); v[5] = __uint_as_float(t.z & 0xffff0000u);
    v[6] = __uint_as_float(t.w << 16); v[7] = __uint_as_float(t.w & 0xffff0000u);
}

// Walks the rows of one work item as chunks of <= 32 edges.  Hub rows (split elsewhere) are skipped;
// empty rows are reported through on_empty.
struct ChunkCursor {
    int row, row_end;      // current row, one past the last row of the item
    int beg, end;          // remaining edge range of the current row
    int hub_threshold;
    bool fresh;            // the next chunk handed out is the first of its row / segment
    __device__ __forceinline__ void start_rows(int r0, int r1, int thr)
    {
        row = r0 - 1; row_end = r1; beg = end = 0; hub_threshold = thr; fresh = false;
    }
    __device__ __forceinline__ void start_segment(int r, int b, int e)   // a single explicit (row, range)
    {
        row = r; row_end = r + 1; beg = b; end = e; hub_threshold = 0x7fffffff; fresh = true;
    }
    // next chunk: returns false when the item is exhausted.  first/last mark row boundaries.
    template <class OnEmpty>
    __device__ __forceinline__ bool next(const int32_t* __restrict__ rowptr, int& out_row, int& out_beg, int& out_n,
                                         bool& first, bool& last, OnEmpty on_empty)
    {
        while (beg >= end) {
            ++row;
            if (row >= row_end) return false;
            beg = rowptr[row];
            end = rowptr[row + 1];
            if (end - beg > hub_threshold) { beg = end; continue; }
            if (end == beg) { on_empty(row); continue; }
            fresh = true;
        }
        first = fresh;
        fresh = false;
        out_row = row;
        out_beg = beg;
        out_n = min(32, end - beg);
        beg += out_n;
        last = beg >= end;
        return true;
    }
    // Low-degree graphs: at a row boundary, try to hand out a PACK of k >= 2 whole consecutive rows (each with
    // 1..32 edges, at most 32 edges in total) as one chunk, so that one phase A serves many rows.  Returns 2 for a
    // pack (out_row = first row, out_beg = first edge, out_n = edges, pack_rows = k; every lane l < k keeps its row's
    // edge range in lane_a/lane_b), 1 for an ordinary single-row chunk, 0 when the item is exhausted.
    template <class OnEmpty>
    __device__ __forceinline__ int next_any(const int32_t* __restrict__ rowptr, int lane, int& out_row, int& out_beg,
                                            int& out_n, bool& first, bool& last, int& pack_rows, int& lane_a,
                                            int& lane_b, OnEmpty on_empty)
    {
        if (beg >= end && row + 1 < row_end) {
            const int r = row + 1;
            const int ri = min(r + lane, row_end - 1);
            const int a = rowptr[ri], b = rowptr[ri + 1];
            const int a0 = __shfl_sync(0xffffffffu, a, 0);
            const bool ok = (r + lane < row_end) && (b > a) && (b - a0 <= 32);
            const unsigned bal = __ballot_sync(0xffffffffu, ok);
            const int k = (bal == 0xffffffffu) ? 32 : __ffs(~bal) - 1;
            if (k >= 2) {
                out_row = r;
                out_beg = a0;
                out_n = __shfl_sync(0xffffffffu, b, k - 1) - a0;
                pack_rows = k;
                lane_a = a;
                lane_b = b;
                first = last = true;
                row = r + k - 1;            // the cursor now sits at the end of the last packed row
                beg = end = a0 + out_n;
                fresh = false;
                return 2;
            }
        }
        return next(rowptr, out_row, out_beg, out_n, first, last, on_empty) ? 1 : 0;
    }
};

}  // namespace gnnfd
