// cf_mlp_simt.cu -- K-4a (per-point half of MLP layer 1) and the CUDA-core (FFMA) version of K-4.
//
// The MLP of SURVEY Appendix A9 is evaluated in an exactly equivalent factorised form:
//   layer 1 is affine in its input [f_p, p - c], so   W1 [f_p, p-c] + b1 = T_p - e_c   with
//     T_p = W1[:, :Ci] f_p + W1[:, Ci:] p + b1      (per POINT, this file: k_point_mlp1, an SGEMM)
//     e_c = W1[:, Ci] cx + W1[:, Ci+1] cy           (per CELL, two FMAs per channel)
//   layer 3 is linear, so it is applied once per cell after the K-sum-pool:
//     sum_k (W3 h2_k + b3) = W3 sum_k h2_k + n_valid b3.
// Only layer 2 (the ReLU sandwich) is evaluated per neighbour.  Results differ from the naive
// formulation by fp32 re-association only (checked at 1e-4 against the brute-force oracle).
//
// k_fusion_simt is the bring-up / cross-check path (CF_MODE_FP32_SIMT); the production path is the
// tcgen05 kernel in cf_mlp_tc.cu.
#include "cf_common.cuh"

namespace cf {

// ---------------------------------------------------------------------------------------------
// T[b,m,n] = sum_k feat[b,m,k] W1[n,k] + sum_d W1[n,Ci+d] p[b,m,d] + b1[n]      (m < num_points[b])
// 64x64 tile, BK=16, 256 threads, 4x4 micro-tile.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_point_mlp1(const float *__restrict__ feat, const float *__restrict__ points,
                                                    const int64_t *__restrict__ num_points, int32_t N, int32_t Ci,
                                                    int32_t C, const float *__restrict__ W1,
                                                    const float *__restrict__ b1, float *__restrict__ T)
{
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int b = blockIdx.z;
    const int32_t n_pts = valid_points(num_points, b, N);
    const int32_t m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
    if (m0 >= n_pts) return;
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, each 4(m) x 4(n)
    const int32_t ldw = Ci + 3;
    const float *A = feat + (size_t)b * N * Ci;
    float acc[4][4] = {};
    const int a_row = tid >> 2, a_k = (tid & 3) * 4;
    for (int32_t k0 = 0; k0 < Ci; k0 += 16) {
        {   // A tile: 64 rows x 16 k, one float4 per thread (Ci % 4 == 0 keeps it aligned)
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int32_t m = m0 + a_row;
            if (m < n_pts && k0 + a_k < Ci) v = __ldg(reinterpret_cast<const float4 *>(A + (size_t)m * Ci + k0 + a_k));
            As[a_k + 0][a_row] = v.x; As[a_k + 1][a_row] = v.y; As[a_k + 2][a_row] = v.z; As[a_k + 3][a_row] = v.w;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {  // B tile: 64 n x 16 k, scalar loads (row stride Ci+3 is not 16B aligned)
            const int idx = tid + r * 256;
            const int nn = idx >> 4, kk = idx & 15;
            const int32_t n = n0 + nn, k = k0 + kk;
            Bs[kk][nn] = (n < C && k < Ci) ? __ldg(W1 + (size_t)n * ldw + k) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            const float4 av = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float a[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int32_t m = m0 + ty * 4 + i;
        if (m >= n_pts) continue;
        const float *p = points + ((size_t)b * N + m) * 3;
        const float px = __ldg(p), py = __ldg(p + 1), pz = __ldg(p + 2);
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int32_t n = n0 + tx * 4 + j;
            float v = 0.0f;
            if (n < C) {
                const float *w = W1 + (size_t)n * ldw + Ci;
                v = acc[i][j] + (__ldg(w) * px + __ldg(w + 1) * py + __ldg(w + 2) * pz) + __ldg(b1 + n);
            }
            o[j] = v;
        }
        float *dst = T + ((size_t)b * N + m) * C + n0 + tx * 4;
        if (n0 + tx * 4 + 3 < C && (C & 3) == 0) {
            *reinterpret_cast<float4 *>(dst) = make_float4(o[0], o[1], o[2], o[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (n0 + tx * 4 + j < C) dst[j] = o[j];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// CUDA-core fused layers 1b/2/3 + pool + add.  Tile = 32 consecutive cells, 256 threads.
// Wt2/Wt3 are the transposed weights (in, out) so that lanes (consecutive out) read coalesced.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_transpose_sq(const float *__restrict__ W, int32_t C, float *__restrict__ Wt)
{
    const int32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * C) return;
    const int32_t o = idx / C, i = idx - o * C;
    Wt[(size_t)i * C + o] = W[idx];
}

template <typename MT>   // map element: float, or __nv_bfloat16 (CF_IO_BF16: widened on load, rounded once on store)
__global__ void __launch_bounds__(256) k_fusion_simt(const MT *__restrict__ bev, const float *__restrict__ T,
                                                     const int32_t *__restrict__ knn, int32_t N, int32_t C, int32_t H,
                                                     int32_t W, int32_t K, float x0, float y0, float dx, float dy,
                                                     const float *__restrict__ W1, int32_t Ci,
                                                     const float *__restrict__ Wt2, const float *__restrict__ b2,
                                                     const float *__restrict__ Wt3, const float *__restrict__ b3,
                                                     MT *__restrict__ out)
{
    extern __shared__ float smem[];
    const int32_t ldp = C + 1;
    float *h1 = smem;                   // [32][C]
    float *pooled = h1 + 32 * C;        // [32][C+1]
    float *w1x = pooled + 32 * ldp;     // [C]
    float *w1y = w1x + C;               // [C]
    float *ccx = w1y + C;               // [32]
    float *ccy = ccx + 32;              // [32]
    int32_t *sidx = reinterpret_cast<int32_t *>(ccy + 32);  // [32][K]
    int32_t *nval = sidx + 32 * CF_MAX_K;                   // [32]

    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    const int64_t cells = (int64_t)H * W;
    const int32_t ldw = Ci + 3;
    for (int c = tid; c < C; c += 256) {
        w1x[c] = __ldg(W1 + (size_t)c * ldw + Ci);
        w1y[c] = __ldg(W1 + (size_t)c * ldw + Ci + 1);
    }
    const float *Tb = T + (size_t)b * N * C;
    const int64_t tiles = ceil_div64(cells, 32);
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t cell0 = tile * 32;
        __syncthreads();
        if (tid < 32) {
            const int64_t cell = cell0 + tid;
            int32_t nv = 0;
            float cx = 0.f, cy = 0.f;
            if (cell < cells) {
                const int32_t i = (int32_t)(cell / W), j = (int32_t)(cell - (int64_t)i * W);
                cx = __fadd_rn(x0, __fmul_rn((float)i, dx));
                cy = __fadd_rn(y0, __fmul_rn((float)j, dy));
                for (int k = 0; k < K; ++k) {
                    const int32_t p = __ldg(knn + ((size_t)b * cells + cell) * K + k);
                    sidx[tid * CF_MAX_K + k] = p;
                    nv += p >= 0;
                }
            } else {
                for (int k = 0; k < K; ++k) sidx[tid * CF_MAX_K + k] = -1;
            }
            ccx[tid] = cx;
            ccy[tid] = cy;
            nval[tid] = nv;
        }
        for (int idx = tid; idx < 32 * ldp; idx += 256) pooled[idx] = 0.0f;
        __syncthreads();
        for (int k = 0; k < K; ++k) {
            for (int idx = tid; idx < 32 * C; idx += 256) {
                const int r = idx / C, c = idx - r * C;
                const int32_t p = sidx[r * CF_MAX_K + k];
                float v = 0.0f;
                if (p >= 0) v = fmaxf(__ldg(Tb + (size_t)p * C + c) - (w1x[c] * ccx[r] + w1y[c] * ccy[r]), 0.0f);
                h1[idx] = v;
            }
            __syncthreads();
            for (int idx = tid; idx < 32 * C; idx += 256) {
                const int r = idx / C, c = idx - r * C;
                if (sidx[r * CF_MAX_K + k] < 0) continue;
                float s = __ldg(b2 + c);
                const float *hr = h1 + r * C;
#pragma unroll 8
                for (int kk = 0; kk < C; ++kk) s = fmaf(hr[kk], __ldg(Wt2 + (size_t)kk * C + c), s);
                pooled[r * ldp + c] += fmaxf(s, 0.0f);
            }
            __syncthreads();
        }
        for (int idx = tid; idx < 32 * C; idx += 256) {
            const int c = idx >> 5, r = idx & 31;
            const int64_t cell = cell0 + r;
            if (cell >= cells) continue;
            float s = (float)nval[r] * __ldg(b3 + c);
            const float *pr = pooled + r * ldp;
#pragma unroll 8
            for (int kk = 0; kk < C; ++kk) s = fmaf(pr[kk], __ldg(Wt3 + (size_t)kk * C + c), s);
            const size_t o = ((size_t)b * C + c) * cells + cell;
            map_st(out + o, map_ldg(bev + o) + s);
        }
    }
}

int point_mlp1_simt(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N,
                    int32_t Ci, int32_t C, const float *d_W1, const float *d_b1, float *d_T, cudaStream_t st)
{
    dim3 grid((unsigned)((N + 63) / 64), (unsigned)((C + 63) / 64), (unsigned)B);
    k_point_mlp1<<<grid, 256, 0, st>>>(d_feat, d_points, d_num_points, N, Ci, C, d_W1, d_b1, d_T);
    count_launches(1);
    return launch_status("cf_point_mlp1");
}

size_t fusion_simt_workspace_bytes(int32_t C) { return (size_t)2 * C * C * sizeof(float); }

int fusion_simt(const float *d_bev, const float *d_T, const int32_t *d_knn, int32_t B, int32_t N, int32_t C,
                int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy, const float *d_W1,
                int32_t Ci, const float *d_W2, const float *d_b2, const float *d_W3, const float *d_b3,
                float *d_out, bool io16, void *d_workspace, cudaStream_t st)
{
    float *Wt2 = (float *)d_workspace, *Wt3 = Wt2 + (size_t)C * C;
    const int tb = (C * C + 255) / 256;
    k_transpose_sq<<<tb, 256, 0, st>>>(d_W2, C, Wt2);
    k_transpose_sq<<<tb, 256, 0, st>>>(d_W3, C, Wt3);
    const size_t smem = (size_t)(32 * C + 32 * (C + 1) + 2 * C + 64) * sizeof(float) +
                        (size_t)(32 * CF_MAX_K + 32) * sizeof(int32_t);
    static bool attr_set = false;
    if (!attr_set) {
        CF_TRY(cuda_status(cudaFuncSetAttribute(k_fusion_simt<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024),
                           "k_fusion_simt smem attribute"));
        CF_TRY(cuda_status(cudaFuncSetAttribute(k_fusion_simt<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024),
                           "k_fusion_simt smem attribute"));
        attr_set = true;
    }
    const int64_t tiles = ceil_div64((int64_t)H * W, 32);
    const int gx = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 8);
    if (io16)
        k_fusion_simt<<<dim3(gx, B), 256, smem, st>>>(reinterpret_cast<const __nv_bfloat16 *>(d_bev), d_T, d_knn, N, C, H, W, K, x0,
                                                      y0, dx, dy, d_W1, Ci, Wt2, d_b2, Wt3, d_b3, reinterpret_cast<__nv_bfloat16 *>(d_out));
    else
        k_fusion_simt<<<dim3(gx, B), 256, smem, st>>>(d_bev, d_T, d_knn, N, C, H, W, K, x0, y0, dx, dy, d_W1, Ci, Wt2,
                                                      d_b2, Wt3, d_b3, d_out);
    count_launches(3);
    return launch_status("cf_fusion_fwd (simt)");
}

}  // namespace cf

namespace cf {
size_t point_mlp1_tc_workspace_bytes(int32_t Ci, int32_t C, int32_t mode);
int point_mlp1_tc(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N,
                  int32_t Ci, int32_t C, const float *d_W1, const float *d_b1, float *d_T, int32_t mode,
                  const void *d_packed, void *d_workspace, cudaStream_t st);
int point_mlp1_tc_pack(const float *d_W1, int32_t Ci, int32_t C, int32_t mode, void *d_packed, cudaStream_t st);
int point_mlp1_multi_tc(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N,
                        int32_t Ci, int32_t n_scales, const int32_t *h_C, const float *const *h_W1,
                        const float *const *h_b1, float *const *h_T, int32_t mode, const void *const *h_packed,
                        cudaStream_t st);
}  // namespace cf

extern "C" int cf_point_mlp1_pack_weights(const float *d_W1, int32_t Ci, int32_t C, int32_t mode, void *d_packed, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    mode = mode_base(mode);
    CF_REQUIRE(d_W1 && d_packed && aligned16(d_packed), CF_ERR_ARG, "cf_point_mlp1_pack_weights: bad pointer");
    CF_REQUIRE(mode == CF_MODE_FP32 || mode == CF_MODE_BF16 || mode == CF_MODE_BF16_TABLES, CF_ERR_ARG,
               "cf_point_mlp1_pack_weights: mode %d has no packed form", mode);
    return point_mlp1_tc_pack(d_W1, Ci, C, mode, d_packed, (cudaStream_t)stream);
}

extern "C" size_t cf_point_mlp1_workspace_bytes(int32_t Ci, int32_t C, int32_t mode)
{
    mode = cf::mode_base(mode);
    if (mode == CF_MODE_FP32_SIMT || Ci <= 0 || C <= 0) return 0;
    return cf::point_mlp1_tc_workspace_bytes(Ci, C, mode);
}

extern "C" int cf_point_mlp1(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B,
                             int32_t N, int32_t Ci, int32_t C, const float *d_W1, const float *d_b1, float *d_T,
                             int32_t mode, const void *d_packed, void *d_workspace, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    mode = mode_base(mode);
    CF_REQUIRE(d_feat && d_points && d_num_points && d_W1 && d_b1 && d_T, CF_ERR_ARG, "cf_point_mlp1: null pointer");
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && Ci > 0 && C > 0, CF_ERR_ARG, "cf_point_mlp1: bad extents");
    CF_REQUIRE(Ci % 4 == 0, CF_ERR_ARG, "cf_point_mlp1: Ci=%d must be a multiple of 4", Ci);
    CF_REQUIRE(mode == CF_MODE_FP32 || mode == CF_MODE_BF16 || mode == CF_MODE_FP32_SIMT || mode == CF_MODE_BF16_TABLES, CF_ERR_ARG,
               "cf_point_mlp1: unknown mode %d", mode);
    CF_REQUIRE(aligned16(d_feat) && aligned16(d_T), CF_ERR_ALIGN, "cf_point_mlp1: feat/T must be 16-byte aligned");
    if (mode == CF_MODE_BF16_TABLES) {   // bf16 rows: the multi-scale kernel with one scale (no FFMA fallback)
        CF_REQUIRE(d_packed != nullptr || d_workspace != nullptr, CF_ERR_ARG, "cf_point_mlp1: CF_MODE_BF16_TABLES needs packed weights or a workspace");
        CF_REQUIRE(aligned16(d_workspace) && aligned16(d_packed) && (reinterpret_cast<uintptr_t>(d_feat) & 31u) == 0 &&
                       (reinterpret_cast<uintptr_t>(d_T) & 31u) == 0,
                   CF_ERR_ALIGN, "cf_point_mlp1: CF_MODE_BF16_TABLES needs 32-byte aligned feat / T and 16-byte aligned weights");
        const void *img = d_packed;
        if (!img) {
            CF_TRY(point_mlp1_tc_pack(d_W1, Ci, C, mode, d_workspace, (cudaStream_t)stream));
            img = d_workspace;
        }
        const int rc = point_mlp1_multi_tc(d_feat, d_points, d_num_points, B, N, Ci, 1, &C, &d_W1, &d_b1, &d_T, mode, &img, (cudaStream_t)stream);
        if (rc == CF_ERR_UNSUPPORTED) set_error("cf_point_mlp1: CF_MODE_BF16_TABLES does not support Ci=%d, C=%d", Ci, C);
        return rc;
    }
    if (mode != CF_MODE_FP32_SIMT && (d_workspace != nullptr || d_packed != nullptr)) {
        CF_REQUIRE(aligned16(d_workspace) && aligned16(d_packed), CF_ERR_ALIGN, "cf_point_mlp1: workspace / packed weights must be 16-byte aligned");
        const int rc = point_mlp1_tc(d_feat, d_points, d_num_points, B, N, Ci, C, d_W1, d_b1, d_T, mode, d_packed,
                                     d_workspace, (cudaStream_t)stream);
        if (rc != CF_ERR_UNSUPPORTED) return rc;  // shapes without a tensor-core instantiation use the FFMA kernel
    }
    return point_mlp1_simt(d_feat, d_points, d_num_points, B, N, Ci, C, d_W1, d_b1, d_T, (cudaStream_t)stream);
}

extern "C" int cf_point_mlp1_multi(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B,
                                   int32_t N, int32_t Ci, int32_t n_scales, const int32_t *h_C,
                                   const float *const *h_W1, const float *const *h_b1, float *const *h_T, int32_t mode,
                                   const void *const *h_packed, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    mode = mode_base(mode);
    CF_REQUIRE(d_feat && d_points && d_num_points && h_C && h_W1 && h_b1 && h_T && h_packed, CF_ERR_ARG,
               "cf_point_mlp1_multi: null pointer");
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && Ci > 0 && n_scales > 0, CF_ERR_ARG, "cf_point_mlp1_multi: bad extents");
    CF_REQUIRE(mode == CF_MODE_FP32 || mode == CF_MODE_BF16 || mode == CF_MODE_BF16_TABLES, CF_ERR_ARG,
               "cf_point_mlp1_multi: mode %d has no tensor-core path", mode);
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_feat) & 31u) == 0, CF_ERR_ALIGN, "cf_point_mlp1_multi: feat must be 32-byte aligned");
    for (int s = 0; s < n_scales && s < 64; ++s) {
        CF_REQUIRE(h_W1[s] && h_b1[s] && h_T[s] && h_packed[s], CF_ERR_ARG, "cf_point_mlp1_multi: null pointer for scale %d", s);
        CF_REQUIRE((reinterpret_cast<uintptr_t>(h_T[s]) & 31u) == 0 && aligned16(h_packed[s]), CF_ERR_ALIGN,
                   "cf_point_mlp1_multi: T of scale %d must be 32-byte aligned, its packed weights 16-byte aligned", s);
    }
    const int rc = point_mlp1_multi_tc(d_feat, d_points, d_num_points, B, N, Ci, n_scales, h_C, h_W1, h_b1, h_T, mode,
                                       h_packed, (cudaStream_t)stream);
    if (rc == CF_ERR_UNSUPPORTED) set_error("cf_point_mlp1_multi: shapes not supported by the multi-scale kernel (Ci=%d, %d scales)", Ci, n_scales);
    return rc;
}
