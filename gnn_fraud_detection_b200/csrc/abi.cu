// extern "C" dispatch for the projection stage (forward + backward): argument checks, algorithm choice.
#include "common.cuh"

namespace gnnfd {
int project_fwd_simt(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst,
                     int64_t N, int64_t K, int H, int C, int xw_dtype, void* xw, float* a_src, float* a_dst,
                     cudaStream_t st);
size_t project_bwd_ws_bytes(int64_t N, int64_t K, int H, int C);
int project_bwd_simt(const float* x, int64_t ldx, const float* W, const float* dxw, const void* xw, int xw_dtype,
                     const float* da_src, const float* da_dst, const float* d_out, int64_t N, int64_t K, int H,
                     int C, int Co, float* dW, float* datt_src, float* datt_dst, float* dbias, float* dx,
                     int64_t lddx, void* ws, size_t ws_bytes, cudaStream_t st, bool skip_dw, bool skip_dx);
void project_dx_simt(const float* dxw, const float* W, int64_t N, int64_t K, int D, int H, float* dx, int64_t lddx,
                     cudaStream_t st);
// tensor-core path (project_tc.cu)
bool tc_supported(int64_t N, int64_t K, int H, int C);
size_t tc_ws_bytes(int64_t N, int64_t K, int H, int C);
int project_fwd_tc(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst,
                   int64_t N, int64_t K, int H, int C, int xw_dtype, void* xw, float* a_src, float* a_dst, void* ws,
                   size_t ws_bytes, cudaStream_t st);
int project_bwd_dx_tc(const float* dxw, const float* W, int64_t N, int64_t K, int D, float* dx, int64_t lddx, void* ws,
                      size_t ws_bytes, cudaStream_t st);
size_t dx_tc_ws_bytes(int64_t K, int D);
int project_bwd_dw_tc(const float* dxw, const float* x, int64_t ldx, int64_t N, int64_t K, int D, float* dW, void* ws,
                      size_t ws_bytes, cudaStream_t st);
bool dw_tc_supported(int64_t K, int D);
size_t dw_tc_ws_bytes(int64_t N, int64_t K, int D);
}  // namespace gnnfd

using namespace gnnfd;

static int pick_algo(int algo, int64_t N, int64_t K, int H, int C)
{
    if (algo == GNNFD_GEMM_SIMT) return GNNFD_GEMM_SIMT;
    if (algo == GNNFD_GEMM_TC) return tc_supported(N, K, H, C) ? GNNFD_GEMM_TC : -1;
    return tc_supported(N, K, H, C) ? GNNFD_GEMM_TC : GNNFD_GEMM_SIMT;
}

extern "C" {

int gnnfd_project_workspace_bytes(int64_t N, int64_t K, int H, int C, int algo, size_t* bytes)
{
    GNNFD_REQUIRE(bytes, GNNFD_ERR_ARG, "project_workspace_bytes: bytes is NULL");
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0, GNNFD_ERR_ARG, "project_workspace_bytes: bad shape");
    (void)algo;
    *bytes = tc_ws_bytes(N, K, H, C) + 256;
    return GNNFD_OK;
}

int gnnfd_project_fwd(const float* x, int64_t ldx, const float* W, const float* att_src, const float* att_dst,
                      int64_t N, int64_t K, int H, int C, int xw_dtype, int algo, void* xw, float* a_src,
                      float* a_dst, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0 && ldx >= K, GNNFD_ERR_ARG, "project_fwd: bad shape");
    GNNFD_REQUIRE(W && att_src && att_dst, GNNFD_ERR_ARG, "project_fwd: NULL parameter tensor");
    GNNFD_REQUIRE(N == 0 || (x && xw && a_src && a_dst), GNNFD_ERR_ARG, "project_fwd: NULL tensor");
    GNNFD_REQUIRE(xw_dtype == GNNFD_F32 || xw_dtype == GNNFD_BF16, GNNFD_ERR_ARG, "project_fwd: bad xw_dtype");
    GNNFD_REQUIRE((reinterpret_cast<uintptr_t>(xw) & 15) == 0 && (H * C) % 4 == 0, GNNFD_ERR_ARG,
                  "project_fwd: xw must be 16-byte aligned and H*C a multiple of 4");
    const int a = pick_algo(algo, N, K, H, C);
    GNNFD_REQUIRE(a > 0, GNNFD_ERR_UNSUPPORTED, "project_fwd: tensor-core path does not support N=%lld K=%lld H=%d C=%d",
                  (long long)N, (long long)K, H, C);
    cudaStream_t st = (cudaStream_t)stream;
    if (a == GNNFD_GEMM_TC)
        return project_fwd_tc(x, ldx, W, att_src, att_dst, N, K, H, C, xw_dtype, xw, a_src, a_dst, ws, ws_bytes, st);
    return project_fwd_simt(x, ldx, W, att_src, att_dst, N, K, H, C, xw_dtype, xw, a_src, a_dst, st);
}

int gnnfd_project_bwd_workspace_bytes(int64_t N, int64_t K, int H, int C, int algo, size_t* bytes)
{
    GNNFD_REQUIRE(bytes, GNNFD_ERR_ARG, "project_bwd_workspace_bytes: bytes is NULL");
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0, GNNFD_ERR_ARG, "project_bwd_workspace_bytes: bad shape");
    (void)algo;
    *bytes = project_bwd_ws_bytes(N, K, H, C) + tc_ws_bytes(N, K, H, C) + 512;
    return GNNFD_OK;
}

int gnnfd_project_bwd(const float* x, int64_t ldx, const float* W, const float* dxw, const void* xw, int xw_dtype,
                      const float* da_src, const float* da_dst, const float* d_out, int64_t N, int64_t K, int H,
                      int C, int Co, int algo, float* dW, float* datt_src, float* datt_dst, float* dbias, float* dx,
                      int64_t lddx, void* ws, size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0 && ldx >= K, GNNFD_ERR_ARG, "project_bwd: bad shape");
    GNNFD_REQUIRE(Co == C || Co == H * C, GNNFD_ERR_ARG, "project_bwd: Co must be C (mean) or H*C (concat)");
    GNNFD_REQUIRE(N == 0 || (x && W && dxw && xw && da_src && da_dst), GNNFD_ERR_ARG, "project_bwd: NULL tensor");
    GNNFD_REQUIRE(!dbias || d_out || N == 0, GNNFD_ERR_ARG, "project_bwd: dbias needs d_out");
    GNNFD_REQUIRE(!dx || lddx >= K, GNNFD_ERR_ARG, "project_bwd: bad lddx");
    size_t need = 0;
    gnnfd_project_bwd_workspace_bytes(N, K, H, C, algo, &need);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "project_bwd: workspace %zu < %zu", ws_bytes, need);
    const int a = pick_algo(algo, N, K, H, C);
    GNNFD_REQUIRE(a > 0, GNNFD_ERR_UNSUPPORTED, "project_bwd: tensor-core path does not support this shape");
    cudaStream_t st = (cudaStream_t)stream;
    const bool tc = a == GNNFD_GEMM_TC && N > 0;
    const size_t simt_bytes = project_bwd_ws_bytes(N, K, H, C);
    const bool tc_dw = tc && dW && dw_tc_supported(K, H * C);
    int rc = project_bwd_simt(x, ldx, W, dxw, xw, xw_dtype, da_src, da_dst, d_out, N, K, H, C, Co, dW, datt_src,
                              datt_dst, dbias, dx, lddx, ws, simt_bytes, st, /*skip_dw=*/tc_dw, /*skip_dx=*/tc);
    if (rc || !tc) return rc;
    char* tws = reinterpret_cast<char*>(ws) + ((simt_bytes + 255) & ~size_t(255));
    const size_t tws_bytes = ws_bytes - ((simt_bytes + 255) & ~size_t(255));
    if (tc_dw) {
        rc = project_bwd_dw_tc(dxw, x, ldx, N, K, H * C, dW, tws, tws_bytes, st);
        if (rc) return rc;
    }
    if (dx) rc = project_bwd_dx_tc(dxw, W, N, K, H * C, dx, lddx, tws, tws_bytes, st);
    return rc;
}

int gnnfd_project_dx_workspace_bytes(int64_t N, int64_t K, int H, int C, size_t* bytes)
{
    GNNFD_REQUIRE(bytes, GNNFD_ERR_ARG, "project_dx_workspace_bytes: bytes is NULL");
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0, GNNFD_ERR_ARG, "project_dx_workspace_bytes: bad shape");
    *bytes = dx_tc_ws_bytes(K, H * C) + 256;
    return GNNFD_OK;
}

int gnnfd_project_dx(const float* dxw, const float* W, int64_t N, int64_t K, int H, int C, float* dx, int64_t lddx, void* ws,
                     size_t ws_bytes, gnnfd_stream_t stream)
{
    GNNFD_REQUIRE(N >= 0 && K > 0 && H > 0 && C > 0 && lddx >= K, GNNFD_ERR_ARG, "project_dx: bad shape");
    GNNFD_REQUIRE(N == 0 || (dxw && W && dx), GNNFD_ERR_ARG, "project_dx: NULL tensor");
    size_t need = 0;
    gnnfd_project_dx_workspace_bytes(N, K, H, C, &need);
    GNNFD_REQUIRE(ws && ws_bytes >= need, GNNFD_ERR_WORKSPACE, "project_dx: workspace %zu < %zu", ws_bytes, need);
    if (N == 0) return GNNFD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (pick_algo(GNNFD_GEMM_AUTO, N, K, H, C) == GNNFD_GEMM_TC)
        return project_bwd_dx_tc(dxw, W, N, K, H * C, dx, lddx, ws, ws_bytes, st);
    project_dx_simt(dxw, W, N, K, H * C, H, dx, lddx, st);
    GNNFD_LAUNCH_CHECK();
    return GNNFD_OK;
}

}  // extern "C"
