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
