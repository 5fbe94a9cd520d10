// cf_fusion.cu -- C-ABI dispatcher of K-4 (cf_fusion_fwd): picks the tcgen05 kernel (cf_mlp_tc.cu) or the
// CUDA-core cross-check kernel (cf_mlp_simt.cu) from `mode`.
#include "cf_common.cuh"

namespace cf {
size_t fusion_simt_workspace_bytes(int32_t C);
int fusion_simt(const float *d_bev, const float *d_T, const int32_t *d_knn, int32_t B, int32_t N, int32_t C,
                int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy, const float *d_W1,
                int32_t Ci, const float *d_W2, const float *d_b2, const float *d_W3, const float *d_b3,
                float *d_out, bool io16, bool nhwc, void *d_workspace, cudaStream_t st);
size_t fusion_tc_workspace_bytes(int32_t C, int32_t mode, int32_t B, int32_t H, int32_t W);
int fusion_tc(const float *d_bev, const float *d_T, const int32_t *d_knn, int32_t B, int32_t N, int32_t C,
              int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy, const float *d_W1,
              int32_t Ci, const float *d_W2, const float *d_b2, const float *d_W3, const float *d_b3,
              float *d_out, int32_t mode, const void *d_packed, void *d_workspace, cudaStream_t st);
size_t fusion_tc_packed_bytes(int32_t C, int32_t mode);
int fusion_tc_pack(const float *d_W2, const float *d_W3, int32_t C, int32_t mode, void *d_packed, cudaStream_t st);
}  // namespace cf

extern "C" size_t cf_fusion_packed_bytes(int32_t C, int32_t mode)
{
    mode = cf::mode_base(mode);
    if (C <= 0 || mode == CF_MODE_FP32_SIMT) return 0;
    return cf::fusion_tc_packed_bytes(C, mode);
}

extern "C" int cf_fusion_pack_weights(const float *d_W2, const float *d_W3, int32_t C, int32_t mode, void *d_packed,
                                      void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    mode = mode_base(mode);
    CF_REQUIRE(d_W2 && d_W3 && d_packed, CF_ERR_ARG, "cf_fusion_pack_weights: null pointer");
    CF_REQUIRE(mode == CF_MODE_FP32 || mode == CF_MODE_BF16 || mode == CF_MODE_BF16_TABLES, CF_ERR_ARG,
               "cf_fusion_pack_weights: mode %d has no packed form", mode);
    CF_REQUIRE(aligned16(d_packed), CF_ERR_ALIGN, "cf_fusion_pack_weights: buffer must be 16-byte aligned");
    return fusion_tc_pack(d_W2, d_W3, C, mode, d_packed, (cudaStream_t)stream);
}

extern "C" size_t cf_fusion_workspace_bytes(int32_t C, int32_t mode, int32_t B, int32_t H, int32_t W)
{
    if (C <= 0 || B <= 0 || H <= 0 || W <= 0) return 0;
    mode = cf::mode_base(mode);
    if (mode == CF_MODE_FP32_SIMT) return cf::fusion_simt_workspace_bytes(C);
    return cf::fusion_tc_workspace_bytes(C, mode, B, H, W);
}

extern "C" int cf_fusion_fwd(const float *d_bev, const float *d_T, const int32_t *d_knn_idx, int32_t B, int32_t N,
                             int32_t C, int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy,
                             const float *d_W1, int32_t Ci, const float *d_W2, const float *d_b2,
                             const float *d_W3, const float *d_b3, float *d_out, int32_t mode, const void *d_packed,
                             void *d_workspace, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_bev && d_T && d_knn_idx && d_W1 && d_W2 && d_b2 && d_W3 && d_b3 && d_out && d_workspace, CF_ERR_ARG,
               "cf_fusion_fwd: null pointer");
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && H > 0 && W > 0 && Ci >= 0, CF_ERR_ARG, "cf_fusion_fwd: bad extents");
    CF_REQUIRE(C >= 16 && C <= 256 && C % 16 == 0, CF_ERR_ARG, "cf_fusion_fwd: C=%d must be a multiple of 16 in [16,256]", C);
    CF_REQUIRE(K >= 1 && K <= CF_MAX_K, CF_ERR_ARG, "cf_fusion_fwd: K=%d outside [1,%d]", K, CF_MAX_K);
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_T) & 31u) == 0 && aligned16(d_workspace), CF_ERR_ALIGN,
               "cf_fusion_fwd: T must be 32-byte aligned, the workspace 16-byte aligned");
    const bool io16 = (mode & CF_IO_BF16) != 0;   // bev / out are bf16 maps
    const bool nhwc = (mode & CF_IO_NHWC) != 0;   // bev / out are (B,H,W,C) maps
    cudaStream_t st = (cudaStream_t)stream;
    switch (mode_base(mode)) {
        case CF_MODE_FP32_SIMT:
            return fusion_simt(d_bev, d_T, d_knn_idx, B, N, C, H, W, K, x0, y0, dx, dy, d_W1, Ci, d_W2, d_b2, d_W3,
                               d_b3, d_out, io16, nhwc, d_workspace, st);
        case CF_MODE_FP32:
        case CF_MODE_BF16:
        case CF_MODE_BF16_TABLES:   // d_T holds bf16 rows
            CF_REQUIRE(d_packed == nullptr || aligned16(d_packed), CF_ERR_ALIGN, "cf_fusion_fwd: packed weights must be 16-byte aligned");
            return fusion_tc(d_bev, d_T, d_knn_idx, B, N, C, H, W, K, x0, y0, dx, dy, d_W1, Ci, d_W2, d_b2, d_W3,
                             d_b3, d_out, mode, d_packed, d_workspace, st);   // fusion_tc reads CF_IO_BF16 / CF_IO_NHWC itself
        default:
            set_error("cf_fusion_fwd: unknown mode %d", mode);
            return CF_ERR_ARG;
    }
}
