// cf_common.cuh -- shared host/device helpers for libcf_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "cf_b200.h"

namespace cf {

// thread-local error text behind cf_last_error()
void set_error(const char *fmt, ...);
// maps a CUDA runtime error to CF_ERR_LAUNCH (+ text); returns CF_OK when err == cudaSuccess
int cuda_status(cudaError_t err, const char *what);
// cudaGetLastError() after a launch
int launch_status(const char *what);
// 0 when the current device is compute capability 10.x (cached per device)
int require_sm100();
int sm_count();
// bookkeeping behind cf_launch_count(): every kernel launch of this library is counted
void count_launches(int n);

#define CF_REQUIRE(cond, code, ...)      \
    do {                                 \
        if (!(cond)) {                   \
            ::cf::set_error(__VA_ARGS__); \
            return (code);               \
        }                                \
    } while (0)

#define CF_TRY(expr)                  \
    do {                              \
        int _cf_rc = (expr);          \
        if (_cf_rc != CF_OK) return _cf_rc; \
    } while (0)

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Row splits of the fixed-order reductions of the deterministic backward (cf_bwd_det.cu): a constant, so the summation
// order depends on shapes and live counts only, not on the SM count of the GPU.
constexpr int kDetSplits = 128;

// `mode` without its flag bits: the MLP arithmetic (CF_MODE_*) that picks kernels, operand layouts and workspace sizes
constexpr int32_t kModeFlags = CF_BWD_DETERMINISTIC | CF_IO_BF16 | CF_IO_NHWC;
static inline int32_t mode_base(int32_t mode) { return mode & ~kModeFlags; }

__host__ __device__ static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Map element access (CF_IO_BF16).  MT = float or __nv_bfloat16; a bf16 element is widened exactly to fp32 on load and an
// fp32 value is rounded once, to nearest even, on store.  The float overloads are the plain fp32 accesses.
__device__ __forceinline__ float map_ldcs(const float *p) { return __ldcs(p); }
__device__ __forceinline__ float map_ldcs(const __nv_bfloat16 *p) { return __bfloat162float(__ldcs(p)); }
__device__ __forceinline__ float map_ldg(const float *p) { return __ldg(p); }
__device__ __forceinline__ float map_ldg(const __nv_bfloat16 *p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ void map_stcs(float *p, float v) { __stcs(p, v); }
__device__ __forceinline__ void map_stcs(__nv_bfloat16 *p, float v)
{
    __stcs(reinterpret_cast<unsigned short *>(p), __bfloat16_as_ushort(__float2bfloat16_rn(v)));
}
__device__ __forceinline__ void map_st(float *p, float v) { *p = v; }
__device__ __forceinline__ void map_st(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }
// the bit pattern a plain copy of a map element moves
template <typename MT> struct MapBits { using type = float; };
template <> struct MapBits<__nv_bfloat16> { using type = unsigned short; };

// number of valid points of frame b, clamped to [0, N]
__device__ __forceinline__ int32_t valid_points(const int64_t *num_points, int b, int32_t N)
{
    int64_t n = num_points[b];
    n = n < 0 ? 0 : n;
    n = n > N ? N : n;
    return (int32_t)n;
}

// Where the camera gather (K-3) and its adjoints take the map coordinates of camera m of point p.  The kind is a run-time
// field, uniform over a launch, so that each gather kernel compiles once per map type.
struct CamSource {
    enum Kind : int32_t {
        kUv,       // one camera: the dataset's projected_loc_uv (B,N,2) at `dev`
        kHostCrt,  // one camera: the reference's CRT_tensor (4,3) in `crt`, passed by value; no depth test
        kRig,      // M cameras: (B,M,4,3) device CRTs at `dev`, w > 0 in front of the camera
    };
    Kind kind;
    const float *points;  // (B,N,3) LiDAR points, projected by the CRT kinds
    const float *dev;
    float crt[12];
};

// one camera from exactly one of d_uv / h_calib (host memory, read here)
static inline CamSource camera_source(const float *d_points, const float *d_uv, const float *h_calib)
{
    CamSource s{};
    s.points = d_points;
    s.kind = h_calib ? CamSource::kHostCrt : CamSource::kUv;
    s.dev = d_uv;
    if (h_calib)
        for (int i = 0; i < 12; ++i) s.crt[i] = h_calib[i];
    return s;
}

static inline CamSource rig_source(const float *d_points, const float *d_calib)
{
    CamSource s{};
    s.kind = CamSource::kRig;
    s.points = d_points;
    s.dev = d_calib;
    return s;
}

// Per-camera constants of the K-3 kernels, passed by value.  Read only at compile-time indices (cam_get, an unrolled select,
// and stage_cam), which keep the parameter arrays in the constant bank: a dynamically indexed parameter array can be
// copied to local memory.  `map` is camera m's frame-0 map: the forward's pixel-major rows (sc unused), or the adjoints' fp32 gradient.
struct RigCams {
    const void *map[CF_MAX_CAMERAS];
    int64_t sb[CF_MAX_CAMERAS], sc[CF_MAX_CAMERAS], sh[CF_MAX_CAMERAS], sw[CF_MAX_CAMERAS];  // element strides
    int32_t Hf[CF_MAX_CAMERAS], Wf[CF_MAX_CAMERAS];
    float sx[CF_MAX_CAMERAS], sy[CF_MAX_CAMERAS];  // Wf_m / img_w_m, Hf_m / img_h_m
    int32_t plane[CF_MAX_CAMERAS];  // fixed-order adjoint: first pixel of camera m in a frame's pixel space (prefix of Hf*Wf)
};

struct Cam {
    const void *map;
    int64_t sb, sc, sh, sw;
    int32_t Hf, Wf, plane;
    float sx, sy;
};

// camera m's constants (m need not be known at compile time)
__device__ __forceinline__ Cam cam_get(const RigCams &r, int m)
{
    Cam c{r.map[0], r.sb[0], r.sc[0], r.sh[0], r.sw[0], r.Hf[0], r.Wf[0], r.plane[0], r.sx[0], r.sy[0]};
#pragma unroll
    for (int k = 1; k < CF_MAX_CAMERAS; ++k)
        if (m == k) c = Cam{r.map[k], r.sb[k], r.sc[k], r.sh[k], r.sw[k], r.Hf[k], r.Wf[k], r.plane[k], r.sx[k], r.sy[k]};
    return c;
}

// The camera constants of frame b, staged in shared memory by the first M threads of a block: a warp reads camera m's
// entries at a warp-uniform index (a broadcast), so they take no registers across the loops of the gather kernels.
struct CamTable {
    const void *base[CF_MAX_CAMERAS];  // camera m's map of frame b
    int64_t sc[CF_MAX_CAMERAS], sh[CF_MAX_CAMERAS], sw[CF_MAX_CAMERAS];
    int32_t Hf[CF_MAX_CAMERAS], Wf[CF_MAX_CAMERAS];
    float sx[CF_MAX_CAMERAS], sy[CF_MAX_CAMERAS];
};

template <typename T, int k>
__device__ __forceinline__ void stage_cam(CamTable &t, const RigCams &r, int b)
{
    t.base[k] = static_cast<const T *>(r.map[k]) + b * r.sb[k];
    t.sc[k] = r.sc[k], t.sh[k] = r.sh[k], t.sw[k] = r.sw[k];
    t.Hf[k] = r.Hf[k], t.Wf[k] = r.Wf[k];
    t.sx[k] = r.sx[k], t.sy[k] = r.sy[k];
}

// thread m < M writes camera m's entries (one branch per camera: a one-camera call runs one short branch), then the block
// synchronises
template <typename T>
__device__ __forceinline__ void stage_cams(CamTable &t, const RigCams &r, int32_t M, int b)
{
    static_assert(CF_MAX_CAMERAS == 8, "one case per camera");
    switch ((int)threadIdx.x < M ? (int)threadIdx.x : -1) {
    case 0: stage_cam<T, 0>(t, r, b); break;
    case 1: stage_cam<T, 1>(t, r, b); break;
    case 2: stage_cam<T, 2>(t, r, b); break;
    case 3: stage_cam<T, 3>(t, r, b); break;
    case 4: stage_cam<T, 4>(t, r, b); break;
    case 5: stage_cam<T, 5>(t, r, b); break;
    case 6: stage_cam<T, 6>(t, r, b); break;
    case 7: stage_cam<T, 7>(t, r, b); break;
    default: break;
    }
    __syncthreads();
}

// host side: the RigCams of M camera descriptors (maps and strides as given; the caller replaces them where it re-lays a
// map or passes gradients).  `total` receives the pixels of one frame, Sum_m Hf_m * Wf_m.
static inline RigCams rig_cams(const cf_camera_map *h, int32_t M, int64_t *total)
{
    RigCams r{};
    int64_t acc = 0;
    for (int m = 0; m < M; ++m) {
        r.map[m] = h[m].d_map;
        r.sb[m] = h[m].sb, r.sc[m] = h[m].sc, r.sh[m] = h[m].sh, r.sw[m] = h[m].sw;
        r.Hf[m] = h[m].Hf, r.Wf[m] = h[m].Wf;
        r.sx[m] = (float)h[m].Wf / h[m].img_w;
        r.sy[m] = (float)h[m].Hf / h[m].img_h;
        r.plane[m] = (int32_t)acc;
        acc += (int64_t)h[m].Hf * h[m].Wf;
    }
    for (int m = M; m < CF_MAX_CAMERAS; ++m) r.plane[m] = INT32_MAX;   // never selected by a pixel of the frame
    *total = acc;
    return r;
}

// host side: the descriptor checks shared by every K-3 entry point -> CF_OK or CF_ERR_ARG (with the text)
static inline int check_cams(const char *fn, const cf_camera_map *h, int32_t M)
{
    CF_REQUIRE(h != nullptr, CF_ERR_ARG, "%s: null camera descriptors", fn);
    CF_REQUIRE(M >= 1 && M <= CF_MAX_CAMERAS, CF_ERR_ARG, "%s: M=%d cameras, expected 1..%d", fn, M, CF_MAX_CAMERAS);
    for (int m = 0; m < M; ++m)
        CF_REQUIRE(h[m].Hf > 0 && h[m].Wf > 0 && h[m].img_w > 0.0f && h[m].img_h > 0.0f, CF_ERR_ARG,
                   "%s: camera %d: bad extents (Hf=%d, Wf=%d, image %gx%g)", fn, m, h[m].Hf, h[m].Wf, (double)h[m].img_w,
                   (double)h[m].img_h);
    return CF_OK;
}

// M equal descriptors: camera m of a (B,M,Ci,Hf,Wf) map with element strides sb, sm, sc, sh, sw
static inline void equal_cams(cf_camera_map *h, const void *map, size_t elem, int64_t sb, int64_t sm, int64_t sc, int64_t sh,
                              int64_t sw, int32_t M, int32_t Hf, int32_t Wf, float img_w, float img_h)
{
    for (int m = 0; m < M; ++m)
        h[m] = cf_camera_map{(const char *)map + m * sm * (int64_t)elem, sb, sc, sh, sw, Hf, Wf, img_w, img_h};
}

__device__ __forceinline__ float crt_col(float x, float y, float z, float c0, float c3, float c6, float c9)
{
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, c0), __fmul_rn(y, c3)), __fmul_rn(z, c6)), c9);
}

// Map coordinates (uf, vf) of point p of frame b in camera m < M:  (u,v) = [x y z 1] @ CRT / w, or the given uv;
// uf = (u+0.5)*sx - 0.5, vf = (v+0.5)*sy - 0.5.  True when the camera sees the point: at least one of the four bilinear
// taps lies inside the (Hf, Wf) map and, for a rig camera, w > 0.
__device__ __forceinline__ bool cam_project(const CamSource &s, int b, int32_t N, int32_t p, int m, int32_t M, float sx,
                                            float sy, int32_t Hf, int32_t Wf, float &uf, float &vf)
{
    float u, v;
    if (s.kind == CamSource::kUv) {
        const float *t = s.dev + ((size_t)b * N + p) * 2;
        u = __ldg(t);
        v = __ldg(t + 1);
    } else {
        const float *q = s.points + ((size_t)b * N + p) * 3;
        const float x = __ldg(q), y = __ldg(q + 1), z = __ldg(q + 2);
        float r[3];
        if (s.kind == CamSource::kRig) {
            const float *c = s.dev + (b * M + m) * 12;  // B <= 65535, M <= 8: int offset (size_t costs a spill in the gather)
#pragma unroll
            for (int k = 0; k < 3; ++k) r[k] = crt_col(x, y, z, __ldg(c + k), __ldg(c + 3 + k), __ldg(c + 6 + k), __ldg(c + 9 + k));
            if (!(r[2] > 0.0f)) return false;
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) r[k] = crt_col(x, y, z, s.crt[k], s.crt[3 + k], s.crt[6 + k], s.crt[9 + k]);
        }
        u = __fdiv_rn(r[0], r[2]);
        v = __fdiv_rn(r[1], r[2]);
    }
    uf = __fsub_rn(__fmul_rn(__fadd_rn(u, 0.5f), sx), 0.5f);
    vf = __fsub_rn(__fmul_rn(__fadd_rn(v, 0.5f), sy), 0.5f);
    return uf > -1.0f && uf < (float)Wf && vf > -1.0f && vf < (float)Hf;
}

// The four bilinear taps of (uf, vf), t = (x,y), (x+1,y), (x,y+1), (x+1,y+1) with x = floor(uf), y = floor(vf): the
// unmasked weights w[t] and which corner columns / rows lie inside the (Hf, Wf) map.
struct Taps {
    int32_t x, y;
    float w[4];
    bool okx[2], oky[2];
    __device__ __forceinline__ bool in(int t) const { return okx[t & 1] && oky[t >> 1]; }
};

__device__ __forceinline__ Taps bilinear_taps(float uf, float vf, int32_t Hf, int32_t Wf)
{
    Taps tp;
    const float fx = floorf(uf), fy = floorf(vf);
    tp.x = (int32_t)fx;
    tp.y = (int32_t)fy;
    const float wx1 = __fsub_rn(uf, fx), wy1 = __fsub_rn(vf, fy);
    const float wx0 = __fsub_rn(1.0f, wx1), wy0 = __fsub_rn(1.0f, wy1);
    tp.w[0] = __fmul_rn(wx0, wy0);
    tp.w[1] = __fmul_rn(wx1, wy0);
    tp.w[2] = __fmul_rn(wx0, wy1);
    tp.w[3] = __fmul_rn(wx1, wy1);
    tp.okx[0] = tp.x >= 0 && tp.x < Wf;
    tp.okx[1] = tp.x + 1 >= 0 && tp.x + 1 < Wf;
    tp.oky[0] = tp.y >= 0 && tp.y < Hf;
    tp.oky[1] = tp.y + 1 >= 0 && tp.y + 1 < Hf;
    return tp;
}

// uniform bucket grid over the BEV plane (K-1/K-2)
struct BucketGrid {
    float gx0, gy0, cell, inv_cell;
    int32_t nbx, nby;
};

__device__ __forceinline__ int32_t bucket_coord(float v, float g0, float inv_cell, int32_t nb)
{
    float f = floorf((v - g0) * inv_cell);
    // clamp in float first so that NaN / huge values cannot overflow the int conversion
    f = fminf(fmaxf(f, 0.0f), (float)(nb - 1));
    return (int32_t)f;
}

}  // namespace cf
