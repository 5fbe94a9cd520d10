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
constexpr int32_t kModeFlags = CF_BWD_DETERMINISTIC | CF_IO_BF16;
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

// Camera of a rig (cf_point_gather_multi*): projects (x,y,z) with the row-vector CRT at `crt` (12 floats, w > 0 in front)
// into map coordinates, with the fp32 sequence of k_point_gather.  True when the camera sees the point: w > 0 and at least
// one of the four bilinear taps lies inside the (Hf, Wf) map.
__device__ __forceinline__ bool rig_project(const float *__restrict__ crt, float x, float y, float z, float sx, float sy,
                                            int32_t Hf, int32_t Wf, float &uf, float &vf)
{
    float r[3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
        r[c] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, __ldg(crt + c)), __fmul_rn(y, __ldg(crt + 3 + c))),
                                   __fmul_rn(z, __ldg(crt + 6 + c))),
                         __ldg(crt + 9 + c));
    if (!(r[2] > 0.0f)) return false;
    uf = __fsub_rn(__fmul_rn(__fadd_rn(__fdiv_rn(r[0], r[2]), 0.5f), sx), 0.5f);
    vf = __fsub_rn(__fmul_rn(__fadd_rn(__fdiv_rn(r[1], r[2]), 0.5f), sy), 0.5f);
    return uf > -1.0f && uf < (float)Wf && vf > -1.0f && vf < (float)Hf;
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
