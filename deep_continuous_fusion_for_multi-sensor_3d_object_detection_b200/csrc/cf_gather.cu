// cf_gather.cu -- K-3: camera projection + bilinear gather of the image feature map, per LiDAR point.
//
//   (u,v) = [x y z 1] @ CRT / w   (data_import_carla.py:196-201; or the dataset's projected_loc_uv)
//   uf = (u+0.5)*Wf/img_w - 0.5,  vf = (v+0.5)*Hf/img_h - 0.5   (pixel-centre convention = grid_sample
//   align_corners=False), 4 taps, taps outside the map read 0.         SURVEY Appendix A6/A7.
//
// The gather wants pixel-major rows (all Ci channels of one pixel contiguous) so that each tap is one
// coalesced, float4-vectorised read; a channel-major (NCHW) map is first re-laid pixel-major by a
// shared-memory tile transpose (coalesced on both sides).  A channels_last map (sc == 1) is used in place.
// A bf16 map (cf_point_gather_bf16) stays bf16 in its pixel-major copy; every tap is widened exactly to fp32 and blended
// with the same fp32 sequence, so the features equal those of the widened fp32 map.
#include "cf_common.cuh"

namespace cf {

// (B, Ci, HW) with strides -> (B, HW, Ci) dense.  32x32 tile through smem, +1 padding: conflict free.
template <typename MT>
__global__ void __launch_bounds__(256) k_to_pixel_major(const MT *__restrict__ src, int64_t sb, int64_t sc,
                                                        int64_t sh, int64_t sw, int32_t Ci, int32_t Hf, int32_t Wf,
                                                        MT *__restrict__ dst)
{
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int32_t HW = Hf * Wf;
    const int32_t p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int32_t c = c0 + r, p = p0 + tx;
        float v = 0.0f;
        if (c < Ci && p < HW) {
            const int32_t h = p / Wf, w = p - h * Wf;
            v = map_ldg(src + b * sb + c * sc + h * sh + w * sw);
        }
        tile[r][tx] = v;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int32_t p = p0 + r, c = c0 + tx;
        if (p < HW && c < Ci) map_st(dst + ((size_t)b * HW + p) * Ci + c, tile[tx][r]);
    }
}

struct Calib {
    float m[12];  // CRT (4,3) row-major
};

// four channels of a pixel-major row, widened to fp32 (a bf16 row: one 8-byte load)
__device__ __forceinline__ float4 ld_px4(const float *row, int32_t c4) { return __ldg(reinterpret_cast<const float4 *>(row) + c4); }
__device__ __forceinline__ float4 ld_px4(const __nv_bfloat16 *row, int32_t c4)
{
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(row) + c4);
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xFFFF0000u));
}

// one warp per point; lanes stride over float4 channel groups
template <typename MT>
__global__ void __launch_bounds__(256) k_point_gather(const MT *__restrict__ pix,  // (B, Hf*Wf, Ci) pixel-major
                                                      int64_t pb, int64_t ph, int64_t pw,  // element strides (pc == 1)
                                                      int32_t Ci, int32_t Hf, int32_t Wf,
                                                      const float *__restrict__ points, const float *__restrict__ uv,
                                                      Calib cal, int use_calib, const int64_t *__restrict__ num_points,
                                                      int32_t N, float sx, float sy, float *__restrict__ feat)
{
    const int b = blockIdx.y;
    const int32_t n = valid_points(num_points, b, N);
    const int lane = threadIdx.x & 31;
    const int32_t warps_per_grid = gridDim.x * (blockDim.x >> 5);
    for (int32_t p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < N; p += warps_per_grid) {
        if (p >= n) {  // zero padding rows: nothing downstream may ever see uninitialised memory
            float4 *z = reinterpret_cast<float4 *>(feat + ((size_t)b * N + p) * Ci);
            for (int32_t c4 = lane; c4 < (Ci >> 2); c4 += 32) z[c4] = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        float u, v;
        if (use_calib) {
            const float *q = points + ((size_t)b * N + p) * 3;
            const float x = __ldg(q), y = __ldg(q + 1), z = __ldg(q + 2);
            float r[3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
                r[c] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, cal.m[c]), __fmul_rn(y, cal.m[3 + c])),
                                           __fmul_rn(z, cal.m[6 + c])),
                                 cal.m[9 + c]);
            u = __fdiv_rn(r[0], r[2]);
            v = __fdiv_rn(r[1], r[2]);
        } else {
            const float2 t = __ldg(reinterpret_cast<const float2 *>(uv) + (size_t)b * N + p);
            u = t.x;
            v = t.y;
        }
        const float uf = __fsub_rn(__fmul_rn(__fadd_rn(u, 0.5f), sx), 0.5f);
        const float vf = __fsub_rn(__fmul_rn(__fadd_rn(v, 0.5f), sy), 0.5f);
        float4 *o = reinterpret_cast<float4 *>(feat + ((size_t)b * N + p) * Ci);
        const int32_t c4n = Ci >> 2;
        if (!(uf > -1.0f && uf < (float)Wf && vf > -1.0f && vf < (float)Hf)) {
            for (int32_t c4 = lane; c4 < c4n; c4 += 32) o[c4] = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        const float fx = floorf(uf), fy = floorf(vf);
        const int32_t ix = (int32_t)fx, iy = (int32_t)fy;
        const float wx1 = __fsub_rn(uf, fx), wy1 = __fsub_rn(vf, fy);
        const float wx0 = __fsub_rn(1.0f, wx1), wy0 = __fsub_rn(1.0f, wy1);
        const bool okx0 = ix >= 0 && ix < Wf, okx1 = ix + 1 >= 0 && ix + 1 < Wf;
        const bool oky0 = iy >= 0 && iy < Hf, oky1 = iy + 1 >= 0 && iy + 1 < Hf;
        const float w00 = (okx0 && oky0) ? __fmul_rn(wx0, wy0) : 0.0f;
        const float w01 = (okx1 && oky0) ? __fmul_rn(wx1, wy0) : 0.0f;
        const float w10 = (okx0 && oky1) ? __fmul_rn(wx0, wy1) : 0.0f;
        const float w11 = (okx1 && oky1) ? __fmul_rn(wx1, wy1) : 0.0f;
        const int32_t x0c = okx0 ? ix : 0, x1c = okx1 ? ix + 1 : 0, y0c = oky0 ? iy : 0, y1c = oky1 ? iy + 1 : 0;
        const MT *r00 = pix + b * pb + y0c * ph + x0c * pw;
        const MT *r01 = pix + b * pb + y0c * ph + x1c * pw;
        const MT *r10 = pix + b * pb + y1c * ph + x0c * pw;
        const MT *r11 = pix + b * pb + y1c * ph + x1c * pw;
        for (int32_t c4 = lane; c4 < c4n; c4 += 32) {
            const float4 a = ld_px4(r00, c4), bq = ld_px4(r01, c4), c = ld_px4(r10, c4), d = ld_px4(r11, c4);
            float4 r;
            r.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.x), __fmul_rn(w01, bq.x)), __fmul_rn(w10, c.x)), __fmul_rn(w11, d.x));
            r.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.y), __fmul_rn(w01, bq.y)), __fmul_rn(w10, c.y)), __fmul_rn(w11, d.y));
            r.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.z), __fmul_rn(w01, bq.z)), __fmul_rn(w10, c.z)), __fmul_rn(w11, d.z));
            r.w = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.w), __fmul_rn(w01, bq.w)), __fmul_rn(w10, c.w)), __fmul_rn(w11, d.w));
            o[c4] = r;
        }
    }
}

template <typename MT>
int point_gather(const MT *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B, int32_t Ci, int32_t Hf,
                 int32_t Wf, const float *d_points, const float *d_uv, const float *h_calib, const int64_t *d_num_points,
                 int32_t N, float img_w, float img_h, float *d_feat, void *d_workspace, void *stream)
{
    CF_TRY(require_sm100());
    CF_REQUIRE(d_img_feat && d_points && d_num_points && d_feat, CF_ERR_ARG, "cf_point_gather: null pointer");
    CF_REQUIRE((d_uv != nullptr) != (h_calib != nullptr), CF_ERR_ARG,
               "cf_point_gather: pass exactly one of d_uv / h_calib");
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && Ci > 0 && Hf > 0 && Wf > 0, CF_ERR_ARG, "cf_point_gather: bad extents");
    CF_REQUIRE(Ci % 4 == 0, CF_ERR_ARG, "cf_point_gather: Ci=%d must be a multiple of 4", Ci);
    CF_REQUIRE(img_w > 0.0f && img_h > 0.0f, CF_ERR_ARG, "cf_point_gather: bad image size");
    CF_REQUIRE(aligned16(d_feat), CF_ERR_ALIGN, "cf_point_gather: d_feat must be 16-byte aligned");
    CF_REQUIRE(d_uv == nullptr || (reinterpret_cast<uintptr_t>(d_uv) & 7u) == 0, CF_ERR_ALIGN,
               "cf_point_gather: d_uv must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const MT *pix = d_img_feat;
    int64_t pb = sb, ph = sh, pw = sw;
    if (sc != 1) {
        CF_REQUIRE(d_workspace != nullptr, CF_ERR_ARG, "cf_point_gather: workspace required for channel-major maps");
        CF_REQUIRE(aligned16(d_workspace), CF_ERR_ALIGN, "cf_point_gather: workspace must be 16-byte aligned");
        const int32_t HW = Hf * Wf;
        dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((Ci + 31) / 32), (unsigned)B);
        k_to_pixel_major<<<grid, 256, 0, st>>>(d_img_feat, sb, sc, sh, sw, Ci, Hf, Wf, (MT *)d_workspace);
        count_launches(1);
        pix = (const MT *)d_workspace;
        pb = (int64_t)HW * Ci;
        ph = (int64_t)Wf * Ci;
        pw = Ci;
    } else {
        // four channels per load: 16 bytes of fp32, 8 bytes of bf16
        CF_REQUIRE((reinterpret_cast<uintptr_t>(d_img_feat) & (4 * sizeof(MT) - 1)) == 0 && sb % 4 == 0 && sh % 4 == 0 &&
                       sw % 4 == 0,
                   CF_ERR_ALIGN, "cf_point_gather: channels_last map must be %d-byte aligned per pixel", (int)(4 * sizeof(MT)));
    }
    Calib cal{};
    if (h_calib)
        for (int i = 0; i < 12; ++i) cal.m[i] = h_calib[i];
    const float sx = (float)Wf / img_w, sy = (float)Hf / img_h;
    const int blocks = (int)std::min<int64_t>(ceil_div64(N, 8), 148 * 16);
    k_point_gather<<<dim3(blocks, B), 256, 0, st>>>(pix, pb, ph, pw, Ci, Hf, Wf, d_points, d_uv, cal,
                                                    h_calib != nullptr, d_num_points, N, sx, sy, d_feat);
    count_launches(1);
    return launch_status("cf_point_gather");
}

}  // namespace cf

extern "C" size_t cf_gather_workspace_bytes(int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, int64_t sc)
{
    if (sc == 1) return 0;
    return (size_t)B * (size_t)Ci * (size_t)Hf * (size_t)Wf * sizeof(float);
}

extern "C" int cf_point_gather(const float *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                               int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                               const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w,
                               float img_h, float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather(d_img_feat, sb, sc, sh, sw, B, Ci, Hf, Wf, d_points, d_uv, h_calib, d_num_points, N, img_w, img_h,
                            d_feat, d_workspace, stream);
}

extern "C" int cf_point_gather_bf16(const void *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                                    int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                                    const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w,
                                    float img_h, float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather(static_cast<const __nv_bfloat16 *>(d_img_feat), sb, sc, sh, sw, B, Ci, Hf, Wf, d_points, d_uv,
                            h_calib, d_num_points, N, img_w, img_h, d_feat, d_workspace, stream);
}
