// cf_common.cuh -- shared host/device helpers for libcf_b200.so (sm_100a only).
#pragma once
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

__host__ __device__ static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// number of valid points of frame b, clamped to [0, N]
__device__ __forceinline__ int32_t valid_points(const int64_t *num_points, int b, int32_t N)
{
    int64_t n = num_points[b];
    n = n < 0 ? 0 : n;
    n = n > N ? N : n;
    return (int32_t)n;
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
