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
// A camera rig (cf_point_gather_multi*) projects with device-side (B,M,4,3) calibrations (w > 0 in front) and averages the
// blends of the cameras that see a point (semantics: include/cf_b200.h).  Each camera has its own map, extent and image
// size (cf_point_gather_rig*); the (B,M,Ci,Hf,Wf) rig and the single-camera entry points run the same kernel with M equal
// descriptors (M = 1 for one camera); only where the map coordinates come from differs (CamSource).
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

// four channels of a pixel-major row, widened to fp32 (a bf16 row: one 8-byte load)
__device__ __forceinline__ float4 ld_px4(const float *row, int32_t c4) { return __ldg(reinterpret_cast<const float4 *>(row) + c4); }
__device__ __forceinline__ float4 ld_px4(const __nv_bfloat16 *row, int32_t c4)
{
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(row) + c4);
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xFFFF0000u));
}

// One warp per point.  Lane m < M resolves camera m (M = 1 for the single-camera entry points); a ballot gives the visible
// set.  Each visible camera's clamped taps and masked weights are shuffled to the warp in ascending camera order, the warp
// blends its Ci channels (float4 per lane) from that camera's map (base and strides from the block's camera table) and sums
// the blends in registers; one division by n_vis (none for one camera), one store.
template <typename MT>
__global__ void __launch_bounds__(256) k_point_gather(const RigCams cams,  // map: pixel-major rows (channel stride 1)
                                                      int32_t M, int32_t Ci, const CamSource src,
                                                      const int64_t *__restrict__ num_points, int32_t N,
                                                      float *__restrict__ feat)
{
    __shared__ CamTable ct;
    const int b = blockIdx.y;
    const int32_t n = valid_points(num_points, b, N);  // loaded before the barrier: its latency overlaps the staging
    stage_cams<MT>(ct, cams, M, b);
    const int lane = threadIdx.x & 31;
    const int32_t warps_per_grid = gridDim.x * (blockDim.x >> 5);
    const int32_t c4n = Ci >> 2;
    const int cl = lane < M ? lane : 0;  // this lane's camera
    for (int32_t p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < N; p += warps_per_grid) {
        float4 *o = reinterpret_cast<float4 *>(feat + ((size_t)b * N + p) * Ci);
        unsigned vis = 0;
        float uf = 0.0f, vf = 0.0f;
        const int32_t Hf = ct.Hf[cl], Wf = ct.Wf[cl];
        if (p < n)
            vis = __ballot_sync(0xffffffffu, lane < M && cam_project(src, b, N, p, lane, M, ct.sx[cl], ct.sy[cl], Hf, Wf, uf, vf));
        if (vis == 0) {  // padding row, or no camera sees the point
            for (int32_t c4 = lane; c4 < c4n; c4 += 32) o[c4] = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        // this lane's camera (meaningful on the visible lanes only): taps outside the map weigh 0 and read corner 0
        const Taps tp = bilinear_taps(uf, vf, Hf, Wf);
        const float l00 = tp.in(0) ? tp.w[0] : 0.0f, l01 = tp.in(1) ? tp.w[1] : 0.0f;
        const float l10 = tp.in(2) ? tp.w[2] : 0.0f, l11 = tp.in(3) ? tp.w[3] : 0.0f;
        const int32_t lx0 = tp.okx[0] ? tp.x : 0, lx1 = tp.okx[1] ? tp.x + 1 : 0;
        const int32_t ly0 = tp.oky[0] ? tp.y : 0, ly1 = tp.oky[1] ? tp.y + 1 : 0;
        const int nv = __popc(vis);
        for (int32_t cb = 0; cb < c4n; cb += 32) {  // warp-uniform trip count: every lane takes part in the shuffles
            const int32_t c4 = cb + lane;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            bool first = true;
            for (unsigned mk = vis; mk; mk &= mk - 1) {
                const int m = __ffs(mk) - 1;
                const float w00 = __shfl_sync(0xffffffffu, l00, m), w01 = __shfl_sync(0xffffffffu, l01, m);
                const float w10 = __shfl_sync(0xffffffffu, l10, m), w11 = __shfl_sync(0xffffffffu, l11, m);
                const int32_t x0c = __shfl_sync(0xffffffffu, lx0, m), x1c = __shfl_sync(0xffffffffu, lx1, m);
                const int32_t y0c = __shfl_sync(0xffffffffu, ly0, m), y1c = __shfl_sync(0xffffffffu, ly1, m);
                if (c4 < c4n) {
                    const MT *base = static_cast<const MT *>(ct.base[m]);
                    const int64_t ph = ct.sh[m], pw = ct.sw[m];
                    const float4 a = ld_px4(base + y0c * ph + x0c * pw, c4), bq = ld_px4(base + y0c * ph + x1c * pw, c4);
                    const float4 c = ld_px4(base + y1c * ph + x0c * pw, c4), d = ld_px4(base + y1c * ph + x1c * pw, c4);
                    float4 r;
                    r.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.x), __fmul_rn(w01, bq.x)), __fmul_rn(w10, c.x)), __fmul_rn(w11, d.x));
                    r.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.y), __fmul_rn(w01, bq.y)), __fmul_rn(w10, c.y)), __fmul_rn(w11, d.y));
                    r.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.z), __fmul_rn(w01, bq.z)), __fmul_rn(w10, c.z)), __fmul_rn(w11, d.z));
                    r.w = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, a.w), __fmul_rn(w01, bq.w)), __fmul_rn(w10, c.w)), __fmul_rn(w11, d.w));
                    if (first) {
                        acc = r;  // not 0 + r: a -0.0 blend keeps its sign
                    } else {
                        acc.x = __fadd_rn(acc.x, r.x);
                        acc.y = __fadd_rn(acc.y, r.y);
                        acc.z = __fadd_rn(acc.z, r.z);
                        acc.w = __fadd_rn(acc.w, r.w);
                    }
                }
                first = false;
            }
            if (c4 < c4n) {
                if (nv > 1) {
                    const float fn = (float)nv;
                    acc = make_float4(__fdiv_rn(acc.x, fn), __fdiv_rn(acc.y, fn), __fdiv_rn(acc.z, fn), __fdiv_rn(acc.w, fn));
                }
                o[c4] = acc;
            }
        }
    }
}

// True when camera m of the descriptors is camera 0 moved by m * sm elements with camera 0's extent and strides: the B*M maps
// of a (B,M,Ci,Hf,Wf) tensor with camera stride sm (sm = sb for one camera)
template <typename MT>
static bool one_shape(const cf_camera_map *h, int32_t M, int64_t &sm)
{
    const intptr_t d = M > 1 ? (intptr_t)h[1].d_map - (intptr_t)h[0].d_map : (intptr_t)(h[0].sb * (int64_t)sizeof(MT));
    if (d % (intptr_t)sizeof(MT)) return false;
    sm = (int64_t)(d / (intptr_t)sizeof(MT));
    for (int m = 1; m < M; ++m)
        if ((intptr_t)h[m].d_map != (intptr_t)h[0].d_map + (intptr_t)(m * sm * (int64_t)sizeof(MT)) || h[m].Hf != h[0].Hf ||
            h[m].Wf != h[0].Wf || h[m].sb != h[0].sb || h[m].sc != h[0].sc || h[m].sh != h[0].sh || h[m].sw != h[0].sw)
            return false;
    return true;
}

// K-3 for the M cameras of h_cams and one source; `fn` names the entry point in the error texts
template <typename MT>
int point_gather(const char *fn, const cf_camera_map *h_cams, int32_t B, int32_t M, int32_t Ci, const CamSource &src,
                 const int64_t *d_num_points, int32_t N, float *d_feat, void *d_workspace, void *stream)
{
    const bool rig = src.kind == CamSource::kRig;
    CF_TRY(require_sm100());
    CF_TRY(check_cams(fn, h_cams, M));
    CF_REQUIRE(src.points && (src.dev || src.kind == CamSource::kHostCrt) && d_num_points && d_feat, CF_ERR_ARG,
               "%s: null pointer", fn);
    CF_REQUIRE(B > 0 && (int64_t)B * M <= 65535 && N > 0 && Ci > 0, CF_ERR_ARG, "%s: bad extents", fn);
    CF_REQUIRE(Ci % 4 == 0, CF_ERR_ARG, "%s: Ci=%d must be a multiple of 4", fn, Ci);
    CF_REQUIRE(aligned16(d_feat), CF_ERR_ALIGN, "%s: d_feat must be 16-byte aligned", fn);
    bool relay = false;
    for (int m = 0; m < M; ++m) {
        const cf_camera_map &c = h_cams[m];
        CF_REQUIRE(c.d_map != nullptr, CF_ERR_ARG, "%s: null pointer (camera %d map)", fn, m);
        if (c.sc != 1) {
            relay = true;
        } else {
            // four channels per load: 16 bytes of fp32, 8 bytes of bf16
            CF_REQUIRE((reinterpret_cast<uintptr_t>(c.d_map) & (4 * sizeof(MT) - 1)) == 0 && c.sb % 4 == 0 && c.sh % 4 == 0 &&
                           c.sw % 4 == 0,
                       CF_ERR_ALIGN, "%s: channels_last map%s must be %d-byte aligned per pixel", fn, rig ? "s" : "",
                       (int)(4 * sizeof(MT)));
        }
    }
    if (relay) {
        CF_REQUIRE(d_workspace != nullptr, CF_ERR_ARG, "%s: workspace required for channel-major maps", fn);
        CF_REQUIRE(aligned16(d_workspace), CF_ERR_ALIGN, "%s: workspace must be 16-byte aligned", fn);
    }
    int64_t total, sm = 0;
    RigCams cams = rig_cams(h_cams, M, &total);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned gy = (unsigned)((Ci + 31) / 32);
    if (relay && one_shape<MT>(h_cams, M, sm)) {
        // the B*M maps of one (B,M,Ci,Hf,Wf) tensor, re-laid (B, M, Hf*Wf, Ci)
        const cf_camera_map &c = h_cams[0];
        const int32_t HW = c.Hf * c.Wf;
        const MT *img = static_cast<const MT *>(c.d_map);
        MT *dst = (MT *)d_workspace;
        const unsigned gx = (unsigned)((HW + 31) / 32);
        if (c.sb == (int64_t)M * sm) {  // the B*M maps are one run of stride sm: one launch re-lays them all
            k_to_pixel_major<<<dim3(gx, gy, (unsigned)(B * M)), 256, 0, st>>>(img, sm, c.sc, c.sh, c.sw, Ci, c.Hf, c.Wf, dst);
            count_launches(1);
        } else {
            for (int32_t b = 0; b < B; ++b)
                k_to_pixel_major<<<dim3(gx, gy, (unsigned)M), 256, 0, st>>>(img + b * c.sb, sm, c.sc, c.sh, c.sw, Ci, c.Hf,
                                                                          c.Wf, dst + (size_t)b * M * HW * Ci);
            count_launches(B);
        }
        for (int m = 0; m < M; ++m) {
            cams.map[m] = dst + (size_t)m * HW * Ci;
            cams.sb[m] = (int64_t)M * HW * Ci;
            cams.sh[m] = (int64_t)c.Wf * Ci;
            cams.sw[m] = Ci;
        }
    } else if (relay) {
        // one launch per channel-major camera, into its own (B, Hf_m*Wf_m, Ci) part of the workspace
        char *ws = (char *)d_workspace;
        for (int m = 0; m < M; ++m) {
            const cf_camera_map &c = h_cams[m];
            if (c.sc == 1) continue;
            const int32_t HW = c.Hf * c.Wf;
            MT *dst = (MT *)ws;
            k_to_pixel_major<<<dim3((unsigned)((HW + 31) / 32), gy, (unsigned)B), 256, 0, st>>>(
                static_cast<const MT *>(c.d_map), c.sb, c.sc, c.sh, c.sw, Ci, c.Hf, c.Wf, dst);
            count_launches(1);
            cams.map[m] = dst;
            cams.sb[m] = (int64_t)HW * Ci;
            cams.sh[m] = (int64_t)c.Wf * Ci;
            cams.sw[m] = Ci;
            ws += (size_t)B * HW * Ci * sizeof(float);   // the workspace bound of cf_gather_rig_workspace_bytes
        }
    }
    // at most five blocks per SM and frame: each warp takes a few points, which pays for the block's camera table
    const int blocks = (int)std::min<int64_t>(ceil_div64(N, 8), 148 * 5);
    k_point_gather<MT><<<dim3(blocks, B), 256, 0, st>>>(cams, M, Ci, src, d_num_points, N, d_feat);
    count_launches(1);
    return launch_status(fn);
}

// one camera (logical (B,Ci,Hf,Wf) map): the rig path with M = 1
template <typename MT>
int point_gather_one(const MT *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B, int32_t Ci, int32_t Hf,
                     int32_t Wf, const float *d_points, const float *d_uv, const float *h_calib, const int64_t *d_num_points,
                     int32_t N, float img_w, float img_h, float *d_feat, void *d_workspace, void *stream)
{
    CF_REQUIRE((d_uv != nullptr) != (h_calib != nullptr), CF_ERR_ARG, "cf_point_gather: pass exactly one of d_uv / h_calib");
    CF_REQUIRE(d_uv == nullptr || (reinterpret_cast<uintptr_t>(d_uv) & 7u) == 0, CF_ERR_ALIGN,
               "cf_point_gather: d_uv must be 8-byte aligned");
    cf_camera_map cam;
    equal_cams(&cam, d_img_feat, sizeof(MT), sb, sb, sc, sh, sw, 1, Hf, Wf, img_w, img_h);
    return point_gather<MT>("cf_point_gather", &cam, B, 1, Ci, camera_source(d_points, d_uv, h_calib), d_num_points, N, d_feat,
                            d_workspace, stream);
}

template <typename MT>
int point_gather_rig(const char *fn, const cf_camera_map *h_cams, int32_t B, int32_t M, int32_t Ci, const float *d_points,
                     const float *d_calib, const int64_t *d_num_points, int32_t N, float *d_feat, void *d_workspace,
                     void *stream)
{
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_calib) & 3u) == 0, CF_ERR_ALIGN, "%s: d_calib must be 4-byte aligned", fn);
    return point_gather<MT>(fn, h_cams, B, M, Ci, rig_source(d_points, d_calib), d_num_points, N, d_feat, d_workspace, stream);
}

// a (B,M,Ci,Hf,Wf) rig: M equal descriptors
template <typename MT>
int point_gather_multi(const MT *d_img_feat, int64_t sb, int64_t sm, int64_t sc, int64_t sh, int64_t sw, int32_t B, int32_t M,
                       int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_calib,
                       const int64_t *d_num_points, int32_t N, float img_w, float img_h, float *d_feat, void *d_workspace,
                       void *stream)
{
    CF_REQUIRE(M >= 1 && M <= CF_MAX_CAMERAS, CF_ERR_ARG, "cf_point_gather_multi: M=%d cameras, expected 1..%d", M,
               CF_MAX_CAMERAS);
    CF_REQUIRE(d_img_feat != nullptr, CF_ERR_ARG, "cf_point_gather_multi: null pointer");
    cf_camera_map cams[CF_MAX_CAMERAS];
    equal_cams(cams, d_img_feat, sizeof(MT), sb, sm, sc, sh, sw, M, Hf, Wf, img_w, img_h);
    return point_gather_rig<MT>("cf_point_gather_multi", cams, B, M, Ci, d_points, d_calib, d_num_points, N, d_feat,
                                d_workspace, stream);
}

}  // namespace cf

extern "C" size_t cf_gather_multi_workspace_bytes(int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf, int64_t sc)
{
    if (sc == 1) return 0;
    return (size_t)B * (size_t)M * (size_t)Ci * (size_t)Hf * (size_t)Wf * sizeof(float);
}

extern "C" size_t cf_gather_workspace_bytes(int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, int64_t sc)
{
    return cf_gather_multi_workspace_bytes(B, 1, Ci, Hf, Wf, sc);
}

// the channel-major cameras' pixel-major copies, one after the other (fp32 size: an upper bound for bf16)
extern "C" size_t cf_gather_rig_workspace_bytes(int32_t B, int32_t M, int32_t Ci, const cf_camera_map *h_cams)
{
    if (h_cams == nullptr || B <= 0 || M <= 0 || M > CF_MAX_CAMERAS || Ci <= 0) return 0;
    size_t bytes = 0;
    for (int m = 0; m < M; ++m)
        if (h_cams[m].sc != 1 && h_cams[m].Hf > 0 && h_cams[m].Wf > 0)
            bytes += (size_t)B * (size_t)Ci * (size_t)h_cams[m].Hf * (size_t)h_cams[m].Wf * sizeof(float);
    return bytes;
}

extern "C" int cf_point_gather(const float *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                               int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                               const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w,
                               float img_h, float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather_one(d_img_feat, sb, sc, sh, sw, B, Ci, Hf, Wf, d_points, d_uv, h_calib, d_num_points, N, img_w,
                                img_h, d_feat, d_workspace, stream);
}

extern "C" int cf_point_gather_bf16(const void *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                                    int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                                    const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w,
                                    float img_h, float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather_one(static_cast<const __nv_bfloat16 *>(d_img_feat), sb, sc, sh, sw, B, Ci, Hf, Wf, d_points, d_uv,
                                h_calib, d_num_points, N, img_w, img_h, d_feat, d_workspace, stream);
}

extern "C" int cf_point_gather_multi(const float *d_img_feat, int64_t sb, int64_t sm, int64_t sc, int64_t sh, int64_t sw,
                                     int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                                     const float *d_calib, const int64_t *d_num_points, int32_t N, float img_w, float img_h,
                                     float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather_multi(d_img_feat, sb, sm, sc, sh, sw, B, M, Ci, Hf, Wf, d_points, d_calib, d_num_points, N, img_w,
                                  img_h, d_feat, d_workspace, stream);
}

extern "C" int cf_point_gather_multi_bf16(const void *d_img_feat, int64_t sb, int64_t sm, int64_t sc, int64_t sh, int64_t sw,
                                          int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                                          const float *d_calib, const int64_t *d_num_points, int32_t N, float img_w,
                                          float img_h, float *d_feat, void *d_workspace, void *stream)
{
    return cf::point_gather_multi(static_cast<const __nv_bfloat16 *>(d_img_feat), sb, sm, sc, sh, sw, B, M, Ci, Hf, Wf,
                                  d_points, d_calib, d_num_points, N, img_w, img_h, d_feat, d_workspace, stream);
}

extern "C" int cf_point_gather_rig(const cf_camera_map *h_cams, int32_t B, int32_t M, int32_t Ci, const float *d_points,
                                   const float *d_calib, const int64_t *d_num_points, int32_t N, float *d_feat,
                                   void *d_workspace, void *stream)
{
    return cf::point_gather_rig<float>("cf_point_gather_rig", h_cams, B, M, Ci, d_points, d_calib, d_num_points, N, d_feat,
                                       d_workspace, stream);
}

extern "C" int cf_point_gather_rig_bf16(const cf_camera_map *h_cams, int32_t B, int32_t M, int32_t Ci, const float *d_points,
                                        const float *d_calib, const int64_t *d_num_points, int32_t N, float *d_feat,
                                        void *d_workspace, void *stream)
{
    return cf::point_gather_rig<__nv_bfloat16>("cf_point_gather_rig_bf16", h_cams, B, M, Ci, d_points, d_calib, d_num_points,
                                               N, d_feat, d_workspace, stream);
}
