/*
 * libgnnfd_b200 -- C ABI of the B200-native GAT message-passing hot path.
 *
 * This is the drop-in boundary for ONE path of aum2606/GNN-Fraud-Detection: the GATConv layer that
 * src/models/gat.py:39,45,51,80 and src/models/tgn.py:43,49,55,94 construct and call
 * (`gat(h, edge_index) -> [N, out_channels]`), forward and backward.  The reference has no FFI of its
 * own (the arithmetic sits in third-party torch_geometric.nn.GATConv); the entry points below are what
 * a binding for that layer would bind, one per stage of GATConv.forward / its autograd mirror:
 *
 *   reference stage (PyG GATConv.forward, SURVEY.md 8(a2))          entry point
 *   ---------------------------------------------------------------  --------------------------------
 *   remove_self_loops + add_self_loops, edge ordering (every call)   gnnfd_csr_build  (+ gnnfd_hub_plan)
 *   x @ W^T, alpha_src/alpha_dst = (xw * att).sum(-1)                gnnfd_project_fwd
 *   edge_update (leaky_relu, softmax, dropout) + message + aggregate
 *     + head mean/concat + bias                                      gnnfd_gat_fwd   (gnnfd_gat_alpha)
 *   loss.backward() through the layer (src/train.py:142)             gnnfd_gat_bwd_dst, gnnfd_gat_bwd_src,
 *                                                                    gnnfd_project_bwd
 *
 * Conventions
 *   - every pointer is DEVICE memory owned by the caller unless the parameter name ends in `_host`;
 *   - all work is enqueued on `stream` (a cudaStream_t); no implicit synchronisation except where a
 *     `_host` output is written (gnnfd_csr_build, gnnfd_hub_plan);
 *   - return value 0 = ok, <0 = error code below; text via gnnfd_last_error() (thread-local);
 *   - the library never allocates device memory: scratch comes in through (ws, ws_bytes), sized by the
 *     matching *_workspace_bytes call;
 *   - indices inside the library are int32 (E' < 2^31); the caller-facing edge_index is int64 [2,E]
 *     exactly as the reference passes it;
 *   - features/gradients are fp32; the projected features xw may be stored fp32 or bf16 (xw_dtype).
 */
#ifndef GNNFD_B200_H_
#define GNNFD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNNFD_ABI_VERSION 22

typedef void* gnnfd_stream_t; /* cudaStream_t */

enum {
    GNNFD_OK = 0,
    GNNFD_ERR_ARG = -1,         /* null pointer, bad shape, misalignment */
    GNNFD_ERR_CUDA = -2,        /* a CUDA runtime call or launch failed */
    GNNFD_ERR_WORKSPACE = -3,   /* ws_bytes too small */
    GNNFD_ERR_RANGE = -4,       /* edge_index entry outside [0,N) or E' >= 2^31 */
    GNNFD_ERR_UNSUPPORTED = -5  /* (H,C), dtype or option not built */
};

/* gnnfd_csr_build flags.  Default edge order inside a row = order of appearance in edge_index' (stable sort on dst', what
 * PyG's scatter sees); GNNFD_ORDER_DST_SRC = PyG sort_edge_index(sort_by_row=False): stable sort on (dst', src'). */
enum { GNNFD_ADD_SELF_LOOPS = 1, GNNFD_BUILD_CSC = 2, GNNFD_ORDER_DST_SRC = 4 };
enum { GNNFD_F32 = 0, GNNFD_BF16 = 1 };                           /* xw_dtype */
enum { GNNFD_ACT_NONE = 0, GNNFD_ACT_RELU = 1, GNNFD_ACT_ELU = 2 };/* fused epilogue activation */
enum { GNNFD_GEMM_AUTO = 0, GNNFD_GEMM_SIMT = 1, GNNFD_GEMM_TC = 2 }; /* projection algorithm */

/* Rows with more than GNNFD_HUB_THRESHOLD edges are split into chunks of GNNFD_HUB_CHUNK edges
 * (edge-balanced hub splitting); both are what gnnfd_hub_plan is normally called with. */
#define GNNFD_HUB_THRESHOLD 512
#define GNNFD_HUB_CHUNK 512

/* A segment plan for one orientation (dst-major CSR or src-major CSC): the hub rows and their chunks. */
typedef struct gnnfd_hub_plan {
    int32_t n_hub;                 /* rows with degree > threshold */
    int32_t n_chunk;               /* sum over hub rows of ceil(degree / chunk) */
    int32_t threshold;
    int32_t chunk;
    const int32_t* hub_row;        /* [n_hub]   row id, ascending */
    const int32_t* hub_chunk_ptr;  /* [n_hub+1] first chunk of each hub row */
    const int32_t* chunk_hub;      /* [n_chunk] hub slot of each chunk */
} gnnfd_hub_plan_t;

/* Cost-balanced work items over a row-pointer array.  The cost of the rows before row i is
 * ptr[i] + i*row_weight (edges plus a per-row charge for the row epilogue, so that long runs of empty or
 * tiny rows are bounded too); item t owns the rows whose cost offset lies in [t*target, (t+1)*target), i.e.
 * rows [item_start[t], item_start[t+1]).  One warp streams one item, so every warp moves about the same
 * number of bytes whatever the degree distribution. */
typedef struct gnnfd_item_plan {
    int32_t n_items;
    int32_t target;                /* cost units (edges + rows*row_weight) per item */
    const int32_t* item_start;     /* [n_items+1] */
} gnnfd_item_plan_t;

/* Destination-sorted CSR (+ optional source-sorted CSC twin) of the rewritten edge list.
 * Rows are destinations [0,n_dst); col[] holds source ids in [0,n_src). */
typedef struct gnnfd_graph {
    int64_t n_dst;
    int64_t n_src;
    int64_t n_edges;               /* E' */
    const int32_t* rowptr;         /* [n_dst+1] */
    const int32_t* col;            /* [E'] source of each dst-sorted edge */
    const int32_t* perm;           /* [E'] position of each dst-sorted edge in edge_index' (PyG order) */
    const int32_t* colptr;         /* [n_src+1]  (NULL when no CSC was built) */
    const int32_t* csc_row;        /* [E'] destination of each src-sorted edge */
    const int32_t* csc_eid;        /* [E'] CSR position of each src-sorted edge */
    const int32_t* csr2csc;        /* [E'] inverse of csc_eid: source-major position of each dst-sorted edge */
    gnnfd_hub_plan_t hub_dst;      /* plan over rowptr  (n_hub = 0 => none) */
    gnnfd_hub_plan_t hub_src;      /* plan over colptr */
    gnnfd_item_plan_t items_dst;   /* work items over rowptr (required by gat_fwd / gat_bwd_dst) */
    gnnfd_item_plan_t items_src;   /* work items over colptr (required by gat_bwd_src) */
    /* gat_bwd_src only: 0 = alpha_used/dz rows are already in source-major order (what gat_bwd_dst writes);
     * 1 = the row of src-sorted entry p is csc_eid[p] (edge gradients received from other GPUs, in arrival order) */
    int32_t edge_grads_indirect;
    int32_t reserved_;
} gnnfd_graph_t;

/* ---- introspection ------------------------------------------------------------------------- */
const char* gnnfd_last_error(void);
int gnnfd_abi_version(void);
size_t gnnfd_sizeof_graph(void);      /* sizeof(gnnfd_graph_t), for binding sanity checks */
size_t gnnfd_sizeof_hub_plan(void);
size_t gnnfd_sizeof_item_plan(void);
/* Number of kernel launches issued by this library since the last reset (bench.py "gpu_launches"). */
int64_t gnnfd_launch_count(void);
void gnnfd_launch_count_reset(void);
/* End of use.  The library owns no device memory (every buffer and workspace is the caller's), so this only detaches the
 * process-wide state it does keep: the dropout seed source and the launch counter.  Safe to call more than once. */
int gnnfd_shutdown(void);

/* ---- (1) edge_index -> destination-sorted CSR ------------------------------------------------
 * Replaces: remove_self_loops/add_self_loops + the per-call scatter ordering inside GATConv.forward
 * (reference call site src/models/gat.py:80).  Bit-exact contract: perm == torch.sort(dst',
 * stable=True).indices, col == src'[perm], rowptr == row offsets; CSC twin == stable sort of col.
 * Output capacity of col/perm/csc_* must be >= E + N (ADD_SELF_LOOPS) or E.  E_out_host receives E'. */
int gnnfd_csr_workspace_bytes(int64_t N, int64_t E, int flags, size_t* bytes);
int gnnfd_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int flags,
                    int32_t* rowptr, int32_t* col, int32_t* perm,
                    int32_t* colptr, int32_t* csc_row, int32_t* csc_eid,
                    int64_t* E_out_host, void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* Hub plan over a row-pointer array (rowptr or colptr).  cap_hub / cap_chunk are the capacities of the
 * output arrays (hub_chunk_ptr needs cap_hub+1).  counts_host[0]=n_hub, counts_host[1]=n_chunk. */
int gnnfd_hub_plan_workspace_bytes(int64_t n_rows, size_t* bytes);
int gnnfd_hub_plan(const int32_t* ptr, int64_t n_rows, int32_t threshold, int32_t chunk,
                   int32_t* hub_row, int32_t* hub_chunk_ptr, int32_t* chunk_hub,
                   int64_t cap_hub, int64_t cap_chunk, int64_t* counts_host,
                   void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* Snapshot / induced-subgraph builder: the vectorised form of create_temporal_subgraph
 * (src/data/dataset.py:198-240: nodes of one time step, edges with both endpoints inside, original orders kept,
 * endpoints relabelled 0..n_sel-1) generalised to a SET of time steps (block-diagonal batch of snapshots).
 * A node i is selected iff time_steps[i] < n_step_table and step_selected[time_steps[i]] != 0; negative time steps
 * and edge endpoints outside [0, N) are GNNFD_ERR_RANGE.  Outputs (device): node_ids[n_sel] ascending original ids,
 * relabel[N] = new id or -1 (optional, may be NULL), sub_edge_index rows at [0, m) and [ld_sub, ld_sub + m) (ld_sub >= E).
 * counts_host[0] = n_sel, counts_host[1] = m.  Synchronises `stream` once to return the counts. */
int gnnfd_subgraph_workspace_bytes(int64_t N, int64_t E, size_t* bytes);
int gnnfd_subgraph_build(const int64_t* time_steps, int64_t N, const uint8_t* step_selected, int64_t n_step_table,
                         const int64_t* edge_index, int64_t E, int64_t* node_ids, int64_t* relabel,
                         int64_t* sub_edge_index, int64_t ld_sub, int64_t* counts_host,
                         void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* inv[perm[i]] = i for a permutation of [0,n) (used for csr2csc = inverse of csc_eid). */
int gnnfd_invert_perm(const int32_t* perm, int64_t n, int32_t* inv, gnnfd_stream_t stream);

/* Work-item plan over a row-pointer array.  n_items = (n_edges + n_rows*row_weight)/target + 1 and
 * item_start needs n_items + 1 entries.  Fully asynchronous on `stream`. */
int gnnfd_item_plan(const int32_t* ptr, int64_t n_rows, int64_t n_edges, int32_t target, int32_t row_weight,
                    int32_t* item_start, gnnfd_stream_t stream);

/* ---- (2) projection  xw = x @ W^T, a_src/a_dst in the epilogue --------------------------------
 * Replaces: lin_src(x).view(-1,H,C); (x_src*att_src).sum(-1); (x_dst*att_dst).sum(-1).
 * x [N,K] fp32 row-major with leading dimension ldx (elements); W [H*C,K] fp32 row-major;
 * att_src/att_dst [H*C]; xw [N,H*C] (xw_dtype); a_src/a_dst [N,H] fp32. */
int gnnfd_project_workspace_bytes(int64_t N, int64_t K, int H, int C, int algo, size_t* bytes);
int gnnfd_project_fwd(const float* x, int64_t ldx, const float* W, const float* att_src,
                      const float* att_dst, int64_t N, int64_t K, int H, int C, int xw_dtype, int algo,
                      void* xw, float* a_src, float* a_dst, void* ws, size_t ws_bytes,
                      gnnfd_stream_t stream);

/* Cached-image projection for a STATIC layer input (the first layer's x does not change between training steps): x is split
 * once into the fp16-pair tensor-core image (power-of-two scale per row; csrc/in_common.cuh layout) and gnnfd_project_fwd_image
 * then computes exactly what gnnfd_project_fwd computes (xw fp32 + per-head logits), with both operands delivered by the bulk
 * copy engine instead of staging warps.  H = 8, C = 64, K <= 192.  ximg 1024-byte aligned; ws 1024-byte aligned. */
int gnnfd_project_image_bytes(int64_t N, int64_t K, size_t* ximg_bytes, size_t* ws_bytes);
int gnnfd_project_image_build(const float* x, int64_t ldx, int64_t N, int64_t K, void* ximg, float* row_scale,
                              gnnfd_stream_t stream);
int gnnfd_project_fwd_image(const void* ximg, const float* row_scale, int64_t N, int64_t K, const float* W,
                            const float* att_src, const float* att_dst, float* xw, float* a_src, float* a_dst,
                            void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* ---- (3) fused LeakyReLU + online segment softmax + weighted neighbour gather-sum ------------
 * Replaces: edge_update + message + aggregate + head mean/concat + bias of GATConv.forward.
 * out [n_dst, concat ? H*C : C]; rowmax/rowsum [n_dst,H] are saved for the backward (rowsum already
 * includes PyG's +1e-16).  a_dst is indexed by LOCAL destination row, a_src/xw by source id.
 * Attention dropout (GATConv(..., dropout=p) in training, src/models/gat.py:39): p_drop = 0 => none.  With p_drop > 0
 * either keep_mask is an explicit [E',H] uint8 keep mask in edge_index' (PyG) order, applied as alpha*keep/(1-p) (parity
 * tests inject one), or keep_mask is NULL and the kernels draw the bits from a counter-based RNG keyed on (dropout_seed,
 * position in edge_index', head) -- no [E',H] tensor exists; forward and backward must be given the same seed.
 * gnnfd_dropout_mask writes those bits out (test hook) and returns the survivor scale.
 * Built geometries (heads, out_channels, xw dtype): (8,32,f32), (8,64,f32), (8,64,bf16), (8,128,f32), (4,32,f32); any other
 * returns GNNFD_ERR_UNSUPPORTED ("... is not built; available: ...").  The same set holds for (4). */
int gnnfd_dropout_mask(uint64_t dropout_seed, float p_drop, int64_t n_edges, int H, uint8_t* keep_mask,
                       float* scale_host, gnnfd_stream_t stream);
/* Process-wide: when device_word is not NULL every kernel that draws dropout bits adds *device_word to its seed.  A training
 * step replayed from a CUDA graph (seeds are baked into the captured launches) increments that word inside the graph and so
 * draws a fresh mask on every replay; forward and backward of one step read the same value.  NULL (default) turns it off. */
void gnnfd_set_dropout_seed_source(const uint64_t* device_word);
int gnnfd_gat_fwd_workspace_bytes(const gnnfd_graph_t* g, int H, int C, size_t* bytes);
int gnnfd_gat_fwd(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src,
                  const float* a_dst, const float* bias, int H, int C, float negative_slope, int concat,
                  int act, const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed, float* out,
                  float* rowmax, float* rowsum, void* ws, size_t ws_bytes, gnnfd_stream_t stream);
/* Same with the layer loop's eval-mode tail fused into the row epilogue (src/models/gat.py:80-91, tgn.py:94-105):
 *   v = mean/concat + bias;  v = v*post_scale[c] + post_shift[c] (BatchNorm1d with running statistics, folded);
 *   v = act(v);  v += residual[row,c].   post_scale/post_shift [Co] come together or both NULL; residual
 *   [n_dst,Co] or NULL. */
int gnnfd_gat_fwd_fused(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src,
                        const float* a_dst, const float* bias, int H, int C, float negative_slope, int concat,
                        int act, const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed,
                        const float* post_scale, const float* post_shift, const float* residual, float* out,
                        float* rowmax, float* rowsum, void* ws, size_t ws_bytes, gnnfd_stream_t stream);
/* alpha [E',H] in dst-sorted (CSR) order, recomputed from the saved row statistics
 * (return_attention_weights=True; un-permute through perm to get PyG order). */
int gnnfd_gat_alpha(const gnnfd_graph_t* g, const float* a_src, const float* a_dst, const float* rowmax,
                    const float* rowsum, int H, float negative_slope, float* alpha,
                    gnnfd_stream_t stream);

/* ---- (4) backward ----------------------------------------------------------------------------
 * dst-major pass: recomputes alpha, forms d_alpha = <dO_h[i], xw[j]>, softmax + LeakyReLU backward.
 *   writes alpha_used [E',H] (alpha after dropout scaling) and dz [E',H] -- both in SOURCE-MAJOR (CSC)
 *   order, i.e. the value of dst-sorted edge e lands at row csr2csc[e], so that the src-major pass (and,
 *   across GPUs, the exchange to the source owners) reads them contiguously -- and da_dst [n_dst,H].
 *   alpha_used and dz are either two dense [E',H] arrays or the two halves of ONE interleaved [E',2H]
 *   buffer (dz == alpha_used + H: 64 contiguous bytes per edge) -- the library recognises the latter from
 *   the pointers.  Needs the CSC twin and csr2csc.  For the head mean (concat = 0) on a graph with the whole CSC twin
 *   (colptr, csc_row, csc_eid), a source work-item plan, direct edge-gradient slots and n_src == n_dst, d_alpha is
 *   computed source-major into an [E',H] fp32 buffer carved from ws (gnnfd_gat_bwd_workspace_bytes includes it; a smaller
 *   ws returns GNNFD_ERR_WORKSPACE).
 * src-major pass (needs the CSC twin): dxw[j] = sum_e alpha_used*dO_h[i] + da_src[j]*att_src
 *   + da_dst_full[j]*att_dst, da_src[j] = sum_e dz.  da_dst_full is indexed by SOURCE id (for a single
 *   GPU it is the da_dst the dst pass produced; NULL => the att_dst term is skipped).
 * d_out [n_dst, concat ? H*C : C].  Geometries as in (3); gnnfd_gat_bwd_src takes fp32 only. */
int gnnfd_gat_bwd_workspace_bytes(const gnnfd_graph_t* g, int H, int C, size_t* bytes);
int gnnfd_gat_bwd_dst(const gnnfd_graph_t* g, const void* xw, int xw_dtype, const float* a_src,
                      const float* a_dst, const float* rowmax, const float* rowsum, const float* d_out,
                      int H, int C, float negative_slope, int concat, const uint8_t* keep_mask,
                      float p_drop, uint64_t dropout_seed, float* alpha_used, float* dz, float* da_dst,
                      void* ws, size_t ws_bytes, gnnfd_stream_t stream);
int gnnfd_gat_bwd_src(const gnnfd_graph_t* g, const float* alpha_used, const float* dz,
                      const float* d_out, const float* att_src, const float* att_dst,
                      const float* da_dst_full, int H, int C, int concat, float* dxw, float* da_src,
                      void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* Projection backward: dW [H*C,K] = dxw^T x ; dx [N,K] = dxw W (NULL => skipped, layer 1);
 * datt_src/datt_dst [H*C] = sum_n da_*[n,h] * xw[n,h,:] ; dbias [Co] = sum_n d_out[n,:]. */
int gnnfd_project_bwd_workspace_bytes(int64_t N, int64_t K, int H, int C, int algo, size_t* bytes);
int gnnfd_project_bwd(const float* x, int64_t ldx, const float* W, const float* dxw, const void* xw,
                      int xw_dtype, const float* da_src, const float* da_dst, const float* d_out,
                      int64_t N, int64_t K, int H, int C, int Co, int algo, float* dW, float* datt_src,
                      float* datt_dst, float* dbias, float* dx, int64_t lddx, void* ws, size_t ws_bytes,
                      gnnfd_stream_t stream);
/* dx [N,K] (leading dimension lddx) = dxw [N,H*C] W alone: the dx GEMM of gnnfd_project_bwd (GNNFD_GEMM_AUTO's choice of
 * kernel), for callers that have dxw but no xw -- the input-space formulation of a hidden layer (5). */
int gnnfd_project_dx_workspace_bytes(int64_t N, int64_t K, int H, int C, size_t* bytes);
int gnnfd_project_dx(const float* dxw, const float* W, int64_t N, int64_t K, int H, int C, float* dx, int64_t lddx,
                     void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* ---- (5) input-space formulation (concat = 0, H = 8, C = 64, K <= 192; gradient w.r.t. x at K = 64 only) -----------------
 * Same reference stages as (2)-(4) (GATConv.forward / backward at src/models/gat.py:39,80, src/train.py:142) evaluated
 * without projected features:  Z[i,h,:] = sum_e alpha[e,h] x[j,:] ;  out = Z W_r / H + bias ;  logits from x . (W_h^T att);
 * backward d_alpha[e,h] = Gd[i,h,:] . x[j,:] with Gd = dO W_r^T / H, dW from the saved Z.  The per-edge gather is K*4
 * bytes instead of H*C*4, and across GPUs (destination ranges, x replicated) only [N,H] logits / logit gradients travel.
 * A first layer needs no dx.  A hidden layer (K = 64) gets it as the projected path does: gnnfd_in_bwd_edges also writes the
 * alpha_used / dz records, gnnfd_gat_bwd_src turns them into dxw and da_src, and gnnfd_project_dx computes dx = dxw W.
 * Z lives in HBM as the fp16-pair tensor-core image described in csrc/in_common.cuh (opaque to the caller).
 *   prep  : per-call constants + weight images, gnnfd_in_sizes().prep_bytes, 1024-byte aligned, built by
 *           gnnfd_in_logits (u) + gnnfd_in_prepare (scales, images); valid until W / att / max|x| change
 *   zimg  : gnnfd_in_sizes().zimg_bytes for n_dst rows, 1024-byte aligned; written by gnnfd_in_fwd, read by gnnfd_in_out
 *           and gnnfd_in_bwd_params
 *   gd    : [rows, gd_ld] fp32, gd_ld = gnnfd_in_sizes().gd_ld
 *   x     : in every call below the PADDED layout (see gnnfd_in_pad_x) */
int gnnfd_in_supported(int64_t K, int H, int C, int concat);
int gnnfd_in_sizes(int64_t n_dst, int64_t K, size_t* prep_bytes, size_t* zimg_bytes, int64_t* gd_ld, int64_t* x_ld);
/* The edge kernels hand whole x rows to the bulk-copy engine, so x must have 16-byte aligned rows of x_ld = round_up(K, 8)
 * floats, zero beyond K (leading dimension % 4 == 0 and >= x_ld).  gnnfd_in_pad_x builds such a copy x16 [N, x_ld] of an
 * arbitrary x (the reference's K = 166 / 165 rows are only 8- / 4-byte aligned); for a static first-layer input it is
 * built once, like the CSR. */
int gnnfd_in_pad_x(const float* x, int64_t ldx, int64_t N, int64_t K, float* x16, gnnfd_stream_t stream);
/* a_src / a_dst [N,H] of rows [0,N) of x; xmax[0] = max(xmax[0], max|x|) (zero it before the first call; across GPUs
 * max-reduce it before gnnfd_in_prepare). */
int gnnfd_in_logits(const float* x, int64_t ldx, int64_t N, int64_t K, const float* W, const float* att_src,
                    const float* att_dst, float* a_src, float* a_dst, float* xmax, void* prep,
                    gnnfd_stream_t stream);
int gnnfd_in_prepare(const float* W, int64_t K, const float* xmax, void* prep, gnnfd_stream_t stream);
int gnnfd_in_fwd_workspace_bytes(const gnnfd_graph_t* g, size_t* bytes);
/* edge_update + message + aggregate in input space -> zimg, rowmax / rowsum [n_dst,H] (as gnnfd_gat_fwd saves them).
 * Two passes: the attention pass writes alpha [E',H] (fp32, CSR order, normalised, BEFORE dropout; the sign bit marks logits
 * in LeakyReLU's negative region) and jflag [E'] (int32: source id | row-end flag << 31); the feature pass streams the edges
 * with those.  alpha and jflag are outputs the caller keeps for gnnfd_in_bwd_edges. */
int gnnfd_in_fwd(const gnnfd_graph_t* g, const float* x, int64_t ldx, int64_t K, const float* a_src,
                 const float* a_dst, float negative_slope, const uint8_t* keep_mask, float p_drop,
                 uint64_t dropout_seed, const void* prep, void* zimg, float* rowmax, float* rowsum, float* alpha,
                 int32_t* jflag, void* ws, size_t ws_bytes, gnnfd_stream_t stream);
/* out [n,C] = act((Z W_r / H + bias) * post_scale + post_shift) + residual  (epilogue as gnnfd_gat_fwd_fused). */
int gnnfd_in_out(const void* zimg, int64_t n, int64_t K, const void* prep, const float* bias, int act,
                 const float* post_scale, const float* post_shift, const float* residual, float* out,
                 gnnfd_stream_t stream);
/* gd [n, gd_ld] = d_out [n,C] W_r^T / H; row-range agnostic (call per block of rows to bound gd).  ws (1024-byte aligned,
 * gnnfd_in_bwd_gd_workspace_bytes) holds the fp16-pair image of the d_out rows that feeds the tensor cores. */
int gnnfd_in_bwd_gd_workspace_bytes(int64_t n, size_t* bytes);
int gnnfd_in_bwd_gd(const float* d_out, int64_t n, int64_t K, const void* prep, float* gd, void* ws, size_t ws_bytes,
                    gnnfd_stream_t stream);
int gnnfd_in_bwd_edges_workspace_bytes(const gnnfd_graph_t* g, size_t* bytes);
/* dz [E',H] (source-major order, row csr2csc[e]) and da_dst [n_dst,H] for the destination rows covered by the work items
 * [item_lo, item_hi) = rows [row_lo, row_hi) (0, n_items, 0, n_dst for everything); gd holds the Gd rows from gd_row0 on.
 * phase bit 0: process the block; bit 1: finish the hub rows (after the last block, same ws).  Needs the CSC twin.
 * alpha / jflag: what gnnfd_in_fwd saved (the backward gathers no logits and recomputes no softmax).
 * alpha_used: NULL, or (K <= 64, padded to 64) the first half of ONE 32-byte aligned interleaved [E',2H] buffer with
 * dz == alpha_used + H, which then receives the (alpha_used, dz) records gnnfd_gat_bwd_src reads, as gnnfd_gat_bwd_dst
 * writes them; dz and da_dst are the same either way. */
int gnnfd_in_bwd_edges(const gnnfd_graph_t* g, const float* x, int64_t ldx, int64_t K, const float* alpha,
                       const int32_t* jflag, const float* gd,
                       int64_t gd_row0, int64_t item_lo, int64_t item_hi, int64_t row_lo, int64_t row_hi,
                       float negative_slope, const uint8_t* keep_mask, float p_drop, uint64_t dropout_seed,
                       float* alpha_used, float* dz, float* da_dst, void* ws, size_t ws_bytes, int phase,
                       gnnfd_stream_t stream);
/* da_src [n_src,H] = per-source sums of dz (over g's CSC). */
int gnnfd_in_bwd_dasrc(const gnnfd_graph_t* g, const float* dz, float* da_src, gnnfd_stream_t stream);
int gnnfd_in_bwd_params_workspace_bytes(int64_t n, int64_t K, size_t* bytes);
/* dW [H*C,K], datt_src / datt_dst [H*C], dbias [C] from the saved image and the logit gradients of rows [0,n).
 * phase bit 0: tensor-core reduction dO^T Z into ws (no logit gradients needed: overlaps their exchange across GPUs);
 * bit 1: node reductions with da_src / da_dst + final dW (same ws); 3 = both. */
int gnnfd_in_bwd_params(const void* zimg, const float* d_out, const float* x, int64_t ldx, int64_t n, int64_t K,
                        const float* W, const float* att_src, const float* att_dst, const float* da_src,
                        const float* da_dst, const void* prep, float* dW, float* datt_src, float* datt_dst,
                        float* dbias, void* ws, size_t ws_bytes, int phase, gnnfd_stream_t stream);

/* ---- (6) model-level fused operators around the layers (SURVEY.md 8(f)) ---------------------------------------------------
 * Train-mode tail of the reference's layer loop (src/models/gat.py:82-91 == src/models/tgn.py:96-105): BatchNorm1d with batch
 * statistics -> ReLU -> feature dropout -> residual add.  Forward: gnnfd_bn_sums (per-rank partial sums, all-reduced by the
 * caller across GPUs) -> gnnfd_bn_finalize -> gnnfd_bn_relu_drop_res_fwd; backward: gnnfd_bn_bwd_sums (+ all-reduce) ->
 * gnnfd_bn_bwd_apply.  Feature dropout uses the counter-based generator of the attention dropout, keyed on
 * (dropout_seed, (row_base + n) * C + c); p_drop = 0 => none.  ws: gnnfd_model_ops_workspace_bytes. */
int gnnfd_model_ops_workspace_bytes(int64_t N, size_t* bytes);
int gnnfd_bn_sums(const float* z, int64_t N, int C, double* sums, void* ws, size_t ws_bytes, gnnfd_stream_t stream);
int gnnfd_bn_finalize(const double* sums, double count, int C, float eps, float momentum, float* running_mean,
                      float* running_var, float* mean, float* invstd, gnnfd_stream_t stream);
int gnnfd_bn_relu_drop_res_fwd(const float* z, int64_t N, int C, const float* mean, const float* invstd,
                               const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed,
                               int64_t row_base, const float* residual, float* out, gnnfd_stream_t stream);
int gnnfd_bn_bwd_sums(const float* z, const float* d_out, int64_t N, int C, const float* mean, const float* invstd,
                      const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed, int64_t row_base,
                      double* sums, void* ws, size_t ws_bytes, gnnfd_stream_t stream);
int gnnfd_bn_bwd_apply(const float* z, const float* d_out, int64_t N, int C, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed, int64_t row_base,
                       const double* sums, double count, float* dz, float* dgamma, float* dbeta,
                       gnnfd_stream_t stream);
/* TemporalGNN head (src/models/tgn.py:60,88-89,108-111), hidden = 64: h_new [N,64] = GRUCell(x, h_prev) with h_prev NULL =
 * the reference's zero state, out [N] = Linear(64 -> 1)(h_new).  Parameters in nn.GRUCell / nn.Linear layout. */
int gnnfd_gru_head_fwd(const float* x, const float* h_prev, int64_t N, const float* w_ih, const float* w_hh,
                       const float* b_ih, const float* b_hh, const float* w_out, const float* b_out, float* h_new,
                       float* out, gnnfd_stream_t stream);
int gnnfd_gru_head_bwd(const float* x, const float* h_prev, const float* d_out, const float* d_hnew, int64_t N,
                       const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, const float* w_out,
                       const float* b_out, float* dx, float* dh_prev, float* dw_ih, float* dw_hh, float* db_ih,
                       float* db_hh, float* dw_out, float* db_out, float* gates_ws, void* ws, size_t ws_bytes,
                       gnnfd_stream_t stream);
/* The reference's loss on the device (src/train.py:108-139,360-361): masked BCEWithLogitsLoss(pos_weight), mean over the
 * labelled nodes (y != -1); d_logits = upstream * dloss/dlogits; stats (double[8], device): sum of losses, labelled count,
 * TP, FP, TN, FN at sigmoid >= 0.5 (src/train.py:146-149) -- no host synchronisation. */
int gnnfd_bce_masked(const float* logits, const int64_t* y, int64_t N, float pos_weight, float upstream, float* loss,
                     float* d_logits, double* stats, void* ws, size_t ws_bytes, gnnfd_stream_t stream);

/* ---- (7) multi-GPU exchange over peer memory (SURVEY.md 8(e); the reference itself is single-process) -------------------
 * One process per GPU; every rank allocates the same buffer in peer-accessible ("symmetric") memory and passes the G device
 * addresses (its own included, ptr[rank]) plus, where the allocation has one, the NVSwitch multicast address.  The kernels
 * store / load straight through NVLink -- no staging buffer, no collective call; the caller separates a producing kernel
 * from the consuming one with a cross-GPU barrier (any: a signal-pad barrier of the symmetric allocation, a 1-element
 * all-reduce).  Host side: partition.PeerExchange (torch symmetric memory).  Scoring a whole model across GPUs
 * (partition.InputSpaceModelPartition) uses gnnfd_in_logits_bcast, gnnfd_in_out_bcast and gnnfd_peer_reduce; training it
 * (partition.InputSpaceModelTrainStep) uses gnnfd_in_logits_bcast, gnnfd_bn_relu_drop_res_fwd_bcast (the hidden rows, finished
 * after the batch statistics) and gnnfd_peer_reduce (da_src and the dx partials, reduced by their owners). */
#define GNNFD_MAX_PEERS 16
typedef struct gnnfd_peers {
    int32_t n_peers;               /* G */
    int32_t rank;                  /* this process */
    void* ptr[GNNFD_MAX_PEERS];    /* the buffer's address on every rank, as mapped in THIS process */
    void* multicast;               /* multicast mapping of the same buffer (NULL: none) */
} gnnfd_peers_t;
/* gnnfd_in_logits fused with the all-gather of a_src: the logit rows of the N own rows are stored into rows
 * [row_offset, row_offset + N) of a_src_all [n_pos,H] ON EVERY RANK (use_multicast: one multimem.st per 16 bytes, replicated
 * by the switch; else one store per peer).  a_dst, xmax stay local (pull-reduce xmax with gnnfd_peer_reduce). */
int gnnfd_in_logits_bcast(const float* x, int64_t ldx, int64_t N, int64_t K, const float* W, const float* att_src,
                          const float* att_dst, const gnnfd_peers_t* a_src_all, int64_t row_offset, int use_multicast,
                          float* a_dst, float* xmax, void* prep, gnnfd_stream_t stream);
/* gnnfd_in_out fused with the all-gather of the layer output: every finished 16-byte piece of output row r (r in [0,n)) is
 * also stored into row row_offset + r of h_all [n_pos,C] ON EVERY RANK (use_multicast: one multimem.st, replicated by the
 * switch; else one store per peer).  Same arithmetic as gnnfd_in_out, bit for bit; out (the own rows) may be NULL.  Checked
 * before anything is launched: 1..GNNFD_MAX_PEERS peers, non-NULL 16-byte aligned peer addresses, a multicast address when
 * use_multicast; n = 0 launches nothing.  With gnnfd_in_logits_bcast this runs a hidden GAT layer across GPUs exchanging
 * only h [N,64] (256 B per node) and a_src [N,H] (32 B per node); partition.InputSpaceModelPartition drives it. */
int gnnfd_in_out_bcast(const void* zimg, int64_t n, int64_t K, const void* prep, const float* bias, int act,
                       const float* post_scale, const float* post_shift, const float* residual,
                       const gnnfd_peers_t* h_all, int64_t row_offset, int use_multicast, float* out,
                       gnnfd_stream_t stream);
/* gnnfd_bn_relu_drop_res_fwd (section 6) fused with the all-gather of its rows: same arithmetic and dropout key
 * (dropout_seed, (row_base + n) * C + c), bit for bit; every finished 16-byte piece of row r (r in [0,N)) is also stored into
 * row row_offset + r of h_all [n_pos,C] ON EVERY RANK (use_multicast: one multimem.st; else one store per peer).  out (the own
 * rows) may be NULL.  Same refusals as gnnfd_in_out_bcast, before anything is launched.  In training the batch statistics
 * exist only after the output GEMM, so this -- not gnnfd_in_out_bcast -- is where a hidden row is finished and broadcast;
 * partition.InputSpaceModelTrainStep drives it. */
int gnnfd_bn_relu_drop_res_fwd_bcast(const float* z, int64_t N, int C, const float* mean, const float* invstd,
                                     const float* gamma, const float* beta, float p_drop, uint64_t dropout_seed,
                                     int64_t row_base, const float* residual, const gnnfd_peers_t* h_all,
                                     int64_t row_offset, int use_multicast, float* out, gnnfd_stream_t stream);
/* out[i] = reduce over ranks of buf_r[offset + i], i in [0,n)  (op 0: sum, 1: max).  use_multicast (sum only, offset and n
 * multiples of 4): multimem.ld_reduce -- the addition happens inside the NVSwitch; else peer loads summed in rank order
 * (deterministic).  The reduce-scatter of the partial da_src [n_pos,H]: every rank reduces ITS OWN row range. */
int gnnfd_peer_reduce(const gnnfd_peers_t* buf, int64_t offset, int64_t n, int op, int use_multicast, float* out,
                      gnnfd_stream_t stream);

/* ---- (8) neighbour sampling (src/data/dataloader.py:42-66, NeighborLoader(num_neighbors=[10,10,10]) with PyG's defaults
 * replace=False, directed=True) ----------------------------------------------------------------------------------------
 * Graph: the RAW destination-sorted CSR of edge_index [2,E] (gnnfd_csr_build with flags = 0): rowptr [N+1], col [E] the
 * source of each sorted edge, eid [E] its column in edge_index (the csr_build `perm`).  The neighbours of v are its in-edges
 * j -> v, duplicates and self-loops included; position p is the p-th in-edge of v in edge_index order.
 * Hop 1 expands the seeds; hop l expands exactly the nodes first discovered in hop l-1 (no node is expanded twice).
 * Selection for a node v of in-degree d expanded with fanout k: every position 0..d-1 when k == -1 or d <= k; otherwise
 * Floyd's algorithm -- for i = 0..k-1: j = d-k+i, t = U_i(j), add j if t is already chosen, else t -- and the chosen
 * positions in ascending order (fanouts up to 32 resolve Floyd in registers; larger ones cost O(k^2/32) per node, serial per
 * warp).  U_i(j) = mulhi64(w, j+1), w = splitmix64(seed + 0x9E3779B97F4A7C15 * (2*(v*2^32 + i) + 1))
 * (mod 2^64), so a node's sample depends only on (seed, v): not on the batch, the hop or the scheduling.
 * Outputs: n_id [node_cap] int64 global ids -- the seeds (local ids 0..B-1, input order), then the nodes new in hop 1 in
 * order of first appearance in hop 1's edge list, then hop 2, ...; edges ordered by hop, then by local destination id, then
 * by position: edge_index rows at [0, m) (local source) and [ld_edge, ld_edge + m) (local destination, non-decreasing),
 * e_id [m] = column in the input edge_index.
 * counts_host [3 + 2*n_hops]: total nodes, total edges, then num_sampled_nodes = [B, n_1..n_L], then
 * num_sampled_edges = [m_1..m_L].  Synchronises `stream` once to return them.
 * node_map [N] int32 must be all -1 on entry and is all -1 on return, also when the call fails after launching (the reset
 * touches only the sampled entries: a call costs work proportional to the sample, never O(N)).
 * Errors: seed outside [0,N) -> GNNFD_ERR_RANGE; duplicate seeds (found on the device), a fanout < -1 or more than 64 hops
 * -> GNNFD_ERR_ARG;
 * more nodes than node_cap or edges than edge_cap -> GNNFD_ERR_WORKSPACE (nothing is written beyond the caps).  Caps that
 * always suffice: nodes min(N, B * prod(1 + k_l)), edges min(E, sum_l F_l * k_l) with F_1 = B, F_{l+1} = min(N, F_l * k_l),
 * reading k = -1 as the maximum in-degree. */
int gnnfd_sample_workspace_bytes(int64_t node_cap, int64_t edge_cap, int32_t n_hops, size_t* bytes);
int gnnfd_neighbor_sample(const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t N,
                          const int64_t* seeds, int64_t n_seeds, const int32_t* fanouts_host, int32_t n_hops,
                          uint64_t seed, int32_t* node_map, int64_t* n_id, int64_t node_cap, int64_t* edge_index,
                          int64_t ld_edge, int64_t* e_id, int64_t edge_cap, int64_t* counts_host,
                          void* ws, size_t ws_bytes, gnnfd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNNFD_B200_H_ */
