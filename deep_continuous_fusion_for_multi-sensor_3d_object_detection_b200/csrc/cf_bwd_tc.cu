// cf_bwd_tc.cu -- the GEMMs of K-4b (cf_bwd.cu) on the tcgen05 tensor cores.
//
// Two shapes cover the backward of the fused layer:
//   NN   Out[R x N]  = epilogue( X[R x Kd] * Wp^T )        R = live rows / live cells / points (long), N, Kd <= 256
//        (Z2 = H1 W2^T,  dPooled = G W3,  dA = (dZ2 W2) . [H1 > 0],  dF += dT W1[:, :Ci])
//   TN   dW[M x N]  += X[R x M]^T * [Y | Y2 | w]           reduction over the long dimension R, split over CTAs
//        (dW2 | db2 = dZ2^T [H1 | 1],  dW3 | db3 = G^T [pooled | n_valid],  dW1 | db1 = dT^T [F | 1],  dW1 offsets = dA^T off)
// fp32 operands are split into bf16 hi + bf16 lo on the fly; hi*hi + hi*lo + lo*hi accumulate in fp32 in TMEM
// (~2^-16 relative per product, the same arithmetic as CF_MODE_FP32 of the forward).  Operands are K-major,
// SWIZZLE_NONE core matrices written by the threads that convert them (cf_tcgen05.cuh); for the TN shape the reduction
// dimension is the ROW index of X / Y, so a thread owns one column and 8 consecutive rows: its 8 scalar loads are
// coalesced across the warp and its 8 values are exactly one 16-byte K-major unit.
// R may live in device memory (d_R): grids are sized for the dense bound and clamp themselves.
#include "cf_common.cuh"
#include "cf_tcgen05.cuh"

namespace cf {

namespace {

constexpr int kRows = 128;     // UMMA M
constexpr int kNT = 512;       // threads per CTA (16 warps, four per TMEM lane quarter: the kernels live on loads in flight)
constexpr int kTnKC = 64;      // rows of X / Y per pipeline stage of the TN kernel

__host__ __device__ constexpr int tmem_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : 256; }
__host__ __device__ constexpr int nn_kc(int Kd) { return Kd <= 128 ? Kd : (Kd % 128 == 0 ? 128 : 64); }

// fp32 (rows, cols) weights, row stride ld -> operand image of B[n, k]:  transpose == 0: B = W (n = row, k = col);
// transpose == 1: B = W^T (n = col, k = row).  Layout [k-chunk][hi | lo][n/8][k/8 in chunk][n%8][k%8] bf16.
__global__ void __launch_bounds__(256) k_bwd_pack(const float *__restrict__ W, int32_t ld, int32_t Nn, int32_t Kd, int32_t KC,
                                                  int transpose, uint8_t *__restrict__ img)
{
    const int32_t units = Nn * (Kd / 8);
    const int32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= units) return;
    const int32_t n = u / (Kd / 8), k8 = u - n * (Kd / 8);
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = transpose ? __ldg(W + (size_t)(k8 * 8 + i) * ld + n) : __ldg(W + (size_t)n * ld + k8 * 8 + i);
    uint4 hi, lo;
    tc::split_bf16x8(v, hi, lo, true);
    const int32_t kc_units = KC / 8, chunk = k8 / kc_units, ku = k8 - chunk * kc_units;
    const size_t split_bytes = (size_t)Nn * KC * 2;
    const size_t base = (size_t)chunk * 2 * split_bytes + tc::unit_offset(n, ku, kc_units);
    *reinterpret_cast<uint4 *>(img + base) = hi;
    *reinterpret_cast<uint4 *>(img + base + split_bytes) = lo;
}

// the same for up to four images in one launch (blockIdx.y = image)
struct PackJob {
    const float *W;
    int32_t ld, Nn, Kd, KC, transpose;
    uint8_t *img;
};
struct PackJobs {
    PackJob j[4];
};
__global__ void __launch_bounds__(256) k_bwd_pack_multi(const PackJobs jobs)
{
    const PackJob &q = jobs.j[blockIdx.y];
    const int32_t units = q.Nn * (q.Kd / 8);
    for (int32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < units; u += gridDim.x * blockDim.x) {
        const int32_t n = u / (q.Kd / 8), k8 = u - n * (q.Kd / 8);
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
            v[i] = q.transpose ? __ldg(q.W + (size_t)(k8 * 8 + i) * q.ld + n) : __ldg(q.W + (size_t)n * q.ld + k8 * 8 + i);
        uint4 hi, lo;
        tc::split_bf16x8(v, hi, lo, true);
        const int32_t kc_units = q.KC / 8, chunk = k8 / kc_units, ku = k8 - chunk * kc_units;
        const size_t split_bytes = (size_t)q.Nn * q.KC * 2;
        const size_t base = (size_t)chunk * 2 * split_bytes + tc::unit_offset(n, ku, kc_units);
        *reinterpret_cast<uint4 *>(q.img + base) = hi;
        *reinterpret_cast<uint4 *>(q.img + base + split_bytes) = lo;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// NN: tile = 128 rows of X.  The whole packed weight image stays in shared memory; X is converted K-chunk by K-chunk.
// ---------------------------------------------------------------------------------------------------------------
enum { EPI_STORE = 0, EPI_ACCUM = 1, EPI_BIAS_RELU = 2, EPI_MASK = 3 };

struct NnParams {
    const float *X;
    int64_t ldx, R;
    const int32_t *d_R;
    int32_t Kd, N, KC;
    const uint8_t *wimg;
    float *Out;
    int64_t ldo;
    int32_t epi;
    const float *aux;  // EPI_BIAS_RELU: bias[N];  EPI_MASK: mask (R x N, row stride ldaux), may alias Out
    int64_t ldaux;
    int32_t stage_cols;  // columns of the accumulator staged through shared memory per epilogue pass (multiple of 32)
};

__global__ void __launch_bounds__(kNT) k_bwd_gemm_nn_tc(const NnParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int64_t R = p.d_R ? min(p.R, (int64_t)__ldg(p.d_R)) : p.R;
    const int64_t tiles = ceil_div64(R, kRows);
    if ((int64_t)blockIdx.x >= tiles) return;
    const int Kd = p.Kd, N = p.N, KC = p.KC, kc_units = KC / 8, chunks = Kd / KC;
    const int w_bytes = 2 * N * Kd * 2;
    uint8_t *sW = smem, *sA = smem + w_bytes;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int cols = tmem_cols(N);
    if (tid == 0) {
        tc::mbar_init(&bar, 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(&tmem_slot, cols);
    for (int o = tid * 16; o < w_bytes; o += kNT * 16)
        *reinterpret_cast<uint4 *>(sW + o) = __ldg(reinterpret_cast<const uint4 *>(p.wimg + o));
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_acc = tmem_slot;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t sA_addr = tc::smem_u32(sA), sW_addr = tc::smem_u32(sW);
    const uint32_t idesc = tc::make_idesc_bf16(kRows, N);
    const uint32_t sbo = kc_units * 128, lbo = 128;
    const uint32_t a_split = kRows * KC * 2, w_split = N * KC * 2;
    const int row = tid & (kRows - 1), grp = tid >> 7;
    uint32_t phase = 0;

    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t r0 = tile * kRows;
        for (int ch = 0; ch < chunks; ++ch) {
            // a warp takes one 8-row group x 4 k-units per step: lane (r8 = lane % 8, u = lane / 8) reads 32 bytes of its row
            const float *xb = p.X + r0 * p.ldx + ch * KC;
            const int n_items = 16 * (kc_units / 4);
            for (int item = warp; item < n_items; item += 2 * (kNT / 32)) {  // two items per warp in flight
                float v[2][8];
                uint32_t off[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int it = item + u * (kNT / 32);
                    const int rg = it / (kc_units / 4), uq = it - rg * (kc_units / 4);
                    const int r = rg * 8 + (lane & 7), ku = uq * 4 + (lane >> 3);
                    off[u] = tc::unit_offset(r, ku, kc_units);
                    if (it < n_items && r0 + r < R) {
                        const float4 *src = reinterpret_cast<const float4 *>(xb + (int64_t)r * p.ldx + ku * 8);
                        const float4 t0 = src[0], t1 = src[1];
                        v[u][0] = t0.x; v[u][1] = t0.y; v[u][2] = t0.z; v[u][3] = t0.w;
                        v[u][4] = t1.x; v[u][5] = t1.y; v[u][6] = t1.z; v[u][7] = t1.w;
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[u][i] = 0.0f;
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    if (item + u * (kNT / 32) >= n_items) break;
                    uint4 hi, lo;
                    tc::split_bf16x8(v[u], hi, lo, true);
                    *reinterpret_cast<uint4 *>(sA + off[u]) = hi;
                    *reinterpret_cast<uint4 *>(sA + a_split + off[u]) = lo;
                }
            }
            tc::fence_proxy_async();
            tc::fence_before_sync();
            __syncthreads();
            if (tid == 0) {
                tc::fence_after_sync();
                const uint32_t wc = sW_addr + (uint32_t)ch * 2 * w_split;
                for (int kk = 0; kk < KC / 16; ++kk) {
                    const uint32_t koff = kk * 2 * lbo;
                    const uint64_t a_hi = tc::make_desc(sA_addr + koff, lbo, sbo), a_lo = tc::make_desc(sA_addr + a_split + koff, lbo, sbo);
                    const uint64_t w_hi = tc::make_desc(wc + koff, lbo, sbo), w_lo = tc::make_desc(wc + w_split + koff, lbo, sbo);
                    tc::mma_bf16(tmem_acc, a_hi, w_hi, idesc, (ch | kk) ? 1u : 0u);
                    tc::mma_bf16(tmem_acc, a_hi, w_lo, idesc, 1u);
                    tc::mma_bf16(tmem_acc, a_lo, w_hi, idesc, 1u);
                }
                tc::commit(&bar);
            }
            tc::mbar_wait(&bar, phase);  // the MMAs have read sA: the next chunk may overwrite it
            phase ^= 1u;
            tc::fence_after_sync();
        }
        // accumulator (lane = row) -> shared memory over the A buffer (the MMAs are done with it), 16-byte columns XOR-swizzled
        // by the row so that both the row-wise writes and the column-wise reads are conflict free -> epilogue with
        // consecutive lanes on consecutive 16-byte columns: a warp touches 512 contiguous bytes of Out instead of 32 rows
        const int n4 = p.stage_cols / 4;  // 16-byte columns per pass (all of N when the tile fits beside the weights)
        float4 *sD = reinterpret_cast<float4 *>(sA);
        const int live_rows = (int)min((int64_t)kRows, R - r0);
        __syncwarp();
#pragma unroll 1
        for (int c0 = 0; c0 < N; c0 += p.stage_cols) {
            if (c0) __syncthreads();  // the previous pass has been read
#pragma unroll 1
            for (int cc = grp; cc < p.stage_cols / 32; cc += kNT / kRows) {
                float z[32];
                tc::tmem_ld32(tmem_acc + lane_off + c0 + cc * 32, z);
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    sD[row * n4 + ((cc * 8 + q) ^ (row & 7))] = make_float4(z[q * 4], z[q * 4 + 1], z[q * 4 + 2], z[q * 4 + 3]);
            }
            tc::fence_before_sync();
            __syncthreads();
            for (int i = tid; i < live_rows * n4; i += kNT) {
                const int m = i / n4, c4 = i - m * n4;
                const float4 z = sD[m * n4 + (c4 ^ (m & 7))];
                float4 *dst = reinterpret_cast<float4 *>(p.Out + (r0 + m) * p.ldo + c0) + c4;
                if (p.epi == EPI_ACCUM) {
                    const float4 o = *dst;
                    *dst = make_float4(o.x + z.x, o.y + z.y, o.z + z.z, o.w + z.w);
                } else if (p.epi == EPI_BIAS_RELU) {
                    const float4 bv = __ldg(reinterpret_cast<const float4 *>(p.aux + c0) + c4);
                    *dst = make_float4(fmaxf(z.x + bv.x, 0.f), fmaxf(z.y + bv.y, 0.f), fmaxf(z.z + bv.z, 0.f), fmaxf(z.w + bv.w, 0.f));
                } else if (p.epi == EPI_MASK) {
                    // read before the (possibly aliasing) store of the same elements
                    const float4 mk = *(reinterpret_cast<const float4 *>(p.aux + (r0 + m) * p.ldaux + c0) + c4);
                    *dst = make_float4(mk.x > 0.f ? z.x : 0.f, mk.y > 0.f ? z.y : 0.f, mk.z > 0.f ? z.z : 0.f, mk.w > 0.f ? z.w : 0.f);
                } else {
                    *dst = z;
                }
            }
        }
        tc::fence_before_sync();
        __syncthreads();  // accumulator and staging buffer are drained before the next tile overwrites them
        tc::fence_after_sync();
    }
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem_acc, cols);
}

// ---------------------------------------------------------------------------------------------------------------
// TN: D[128 x Nt] (TMEM) = sum over this CTA's rows of  X[r, m0 + m] * Ycat[r, n],   then atomically added to dW / db.
// Ycat = [ Y (N columns) | Y2 (n2 columns) | w or 1 (one column, when db != nullptr) | zero padding to a multiple of 16 ].
// blockIdx.y = 128-column tile of X (M <= 256 -> 1 or 2), blockIdx.x = split of the row range.  Two shared-memory
// stages: the conversion of rows [i+1] runs under the MMAs of rows [i].
// ---------------------------------------------------------------------------------------------------------------
struct TnParams {
    const float *X;
    int64_t ldx;
    int32_t M;
    const float *Y;
    int64_t ldy;
    int32_t N;
    const float *Y2;    // extra columns: element (r, j) = Y2[r * rs2 + j * cs2]
    int64_t rs2, cs2;
    int32_t n2;
    const float *wcol;  // weights of the extra column (nullptr: ones)
    int32_t Nt;         // MMA N: N + n2 + (db ? 1 : 0) rounded up to 16
    int64_t R;
    const int32_t *d_R;
    float *dW;
    int64_t ldw;
    float *db;
    float *part;        // deterministic mode: this CTA's tile goes to part[split][M][n_out] instead of the atomics
};

__global__ void __launch_bounds__(kNT) k_bwd_gemm_tn_tc(const TnParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar[2];
    __shared__ uint32_t tmem_slot;
    const int64_t R = p.d_R ? min(p.R, (int64_t)__ldg(p.d_R)) : p.R;
    const int64_t chunks_total = ceil_div64(R, kTnKC), per = ceil_div64(chunks_total, gridDim.x);
    const int64_t c_begin = (int64_t)blockIdx.x * per, c_end = min(chunks_total, c_begin + per);
    if (c_begin >= c_end) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.y * kRows, Mv = min(kRows, p.M - m0);  // valid rows of D in this tile
    const int N = p.N, Nt = p.Nt, n_extra = Nt - N;
    constexpr int kc_units = kTnKC / 8;
    constexpr uint32_t a_split = kRows * kTnKC * 2;
    const uint32_t b_split = (uint32_t)Nt * kTnKC * 2;
    const uint32_t stage_bytes = 2 * a_split + 2 * b_split;
    const int cols = tmem_cols(Nt);
    if (tid == 0) {
        tc::mbar_init(&bar[0], 1);
        tc::mbar_init(&bar[1], 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(&tmem_slot, cols);
    // rows of the A operand beyond the valid columns of X stay zero in both stages
    if (Mv < kRows)
        for (int s = 0; s < 2; ++s)
            for (int o = tid * 16; o < (int)(2 * a_split); o += kNT * 16) *reinterpret_cast<uint4 *>(smem + s * stage_bytes + o) = make_uint4(0, 0, 0, 0);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_acc = tmem_slot;
    const uint32_t idesc = tc::make_idesc_bf16(kRows, Nt);
    constexpr uint32_t sbo = kc_units * 128, lbo = 128;
    const int items_a = (Mv / 32) * kc_units, items_b = (N / 32) * kc_units, items_e = n_extra ? kc_units : 0;

    for (int64_t c = c_begin; c < c_end; ++c) {
        const int64_t i = c - c_begin;
        const int s = (int)(i & 1);
        if (i >= 2) {  // stage s was read by the MMAs of chunk i - 2
            tc::mbar_wait(&bar[s], (uint32_t)(((i - 2) >> 1) & 1));
            tc::fence_after_sync();
        }
        uint8_t *sA = smem + s * stage_bytes, *sB = sA + 2 * a_split;
        const int64_t r0 = c * kTnKC;
        const int n_items = items_a + items_b + items_e;
        for (int item = warp; item < n_items; item += 2 * (kNT / 32)) {  // two items per warp in flight
            float v[2][8];
            uint8_t *dst[2];
            uint32_t split[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int it0 = item + u * (kNT / 32);
                dst[u] = nullptr;
                if (it0 >= n_items) continue;
                if (it0 < items_a + items_b) {
                    const bool isa = it0 < items_a;
                    const int it = isa ? it0 : it0 - items_a;
                    const int cb = it / kc_units, ku = it - cb * kc_units;
                    const int col = cb * 32 + lane;
                    const float *src = isa ? p.X + (r0 + ku * 8) * p.ldx + m0 + col : p.Y + (r0 + ku * 8) * p.ldy + col;
                    const int64_t ld = isa ? p.ldx : p.ldy;
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[u][j] = (r0 + ku * 8 + j < R) ? __ldg(src + j * ld) : 0.0f;
                    dst[u] = (isa ? sA : sB) + tc::unit_offset(col, ku, kc_units);
                    split[u] = isa ? a_split : b_split;
                } else {
                    if (lane >= n_extra) continue;
                    const int ku = it0 - items_a - items_b;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int64_t r = r0 + ku * 8 + j;
                        float x = 0.0f;
                        if (r < R) {
                            if (lane < p.n2) x = __ldg(p.Y2 + r * p.rs2 + lane * p.cs2);
                            else if (lane == p.n2 && p.db) x = p.wcol ? __ldg(p.wcol + r) : 1.0f;
                        }
                        v[u][j] = x;
                    }
                    dst[u] = sB + tc::unit_offset(N + lane, ku, kc_units);
                    split[u] = b_split;
                }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (!dst[u]) continue;
                uint4 hi, lo;
                tc::split_bf16x8(v[u], hi, lo, true);
                *reinterpret_cast<uint4 *>(dst[u]) = hi;
                *reinterpret_cast<uint4 *>(dst[u] + split[u]) = lo;
            }
        }
        tc::fence_proxy_async();
        tc::fence_before_sync();
        __syncthreads();
        if (tid == 0) {
            tc::fence_after_sync();
            const uint32_t a_addr = tc::smem_u32(sA), b_addr = tc::smem_u32(sB);
#pragma unroll
            for (int kk = 0; kk < kTnKC / 16; ++kk) {
                const uint32_t koff = kk * 2 * lbo;
                const uint64_t a_hi = tc::make_desc(a_addr + koff, lbo, sbo), a_lo = tc::make_desc(a_addr + a_split + koff, lbo, sbo);
                const uint64_t b_hi = tc::make_desc(b_addr + koff, lbo, sbo), b_lo = tc::make_desc(b_addr + b_split + koff, lbo, sbo);
                tc::mma_bf16(tmem_acc, a_hi, b_hi, idesc, (i | kk) ? 1u : 0u);
                tc::mma_bf16(tmem_acc, a_hi, b_lo, idesc, 1u);
                tc::mma_bf16(tmem_acc, a_lo, b_hi, idesc, 1u);
            }
            tc::commit(&bar[s]);
        }
    }
    {   // the last commit covers every MMA issued before it
        const int64_t last = c_end - c_begin - 1;
        tc::mbar_wait(&bar[last & 1], (uint32_t)((last >> 1) & 1));
        tc::fence_after_sync();
    }
    // D (lane = row m) -> shared memory [m][Nt + 1] (the stages are free now) -> atomics with lane = column n: a warp adds
    // to 128 contiguous bytes of one row of dW instead of to 32 different rows
    float *sD = reinterpret_cast<float *>(smem);
    const int ldd = Nt + 1;
    {
        const int m = (warp & 3) * 32 + lane;
        const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
#pragma unroll 1
        for (int cc = warp >> 2; cc < Nt / 16; cc += kNT / kRows) {
            float z[16];
            tc::tmem_ld16(tmem_acc + lane_off + cc * 16, z);
#pragma unroll
            for (int j = 0; j < 16; ++j) sD[m * ldd + cc * 16 + j] = z[j];
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    const int n_w = N + p.n2;  // columns [0, n_w) go to dW, column n_w to db
    const int n_out = n_w + (p.db ? 1 : 0);
    if (p.part) {
        float *dst = p.part + ((int64_t)blockIdx.x * p.M + m0) * n_out;
        for (int m = warp; m < Mv; m += kNT / 32)
            for (int n = lane; n < n_out; n += 32) dst[(int64_t)m * n_out + n] = sD[m * ldd + n];
    } else {
        for (int m = warp; m < Mv; m += kNT / 32) {
            float *dw = p.dW + (int64_t)(m0 + m) * p.ldw;
            for (int n = lane; n < n_out; n += 32) {
                const float v = sD[m * ldd + n];
                if (v == 0.0f) continue;
                if (n < n_w) atomicAdd(dw + n, v);
                else atomicAdd(p.db + m0 + m, v);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem_acc, cols);
}

}  // namespace

// ---- host side (internal to the library; cf_bwd.cu is the caller) ---------------------------------------------------------
size_t bwd_tc_packed_bytes(int32_t Nn, int32_t Kd) { return ((size_t)2 * Nn * Kd * 2 + 255) / 256 * 256; }

bool bwd_tc_nn_fits(int32_t Kd, int32_t N)
{
    return Kd % 32 == 0 && N % 32 == 0 && Kd <= 256 && N <= 256 &&
           (size_t)2 * N * Kd * 2 + (size_t)2 * kRows * nn_kc(Kd) * 2 <= 220 * 1024;
}

bool bwd_tc_tn_fits(int32_t M, int32_t N) { return M % 32 == 0 && N % 32 == 0 && M <= 256 && N <= 256; }

int bwd_tc_pack(const float *d_W, int32_t ld, int32_t Nn, int32_t Kd, int transpose, void *d_img, cudaStream_t st)
{
    const int32_t units = Nn * (Kd / 8);
    k_bwd_pack<<<(units + 255) / 256, 256, 0, st>>>(d_W, ld, Nn, Kd, nn_kc(Kd), transpose, (uint8_t *)d_img);
    count_launches(1);
    return launch_status("cf_fusion_bwd (pack)");
}

int bwd_tc_pack4(const float *const *Ws, const int32_t *lds, const int32_t *Nns, const int32_t *Kds, const int *transposes,
                 void *const *imgs, int n, cudaStream_t st)
{
    PackJobs jobs{};
    int32_t most = 0;
    for (int i = 0; i < n; ++i) {
        jobs.j[i] = PackJob{Ws[i], lds[i], Nns[i], Kds[i], nn_kc(Kds[i]), transposes[i], (uint8_t *)imgs[i]};
        most = std::max(most, Nns[i] * (Kds[i] / 8));
    }
    k_bwd_pack_multi<<<dim3((unsigned)std::min((most + 255) / 256, 64), (unsigned)n), 256, 0, st>>>(jobs);
    count_launches(1);
    return launch_status("cf_fusion_bwd (pack)");
}

int bwd_tc_gemm_nn(const float *X, int64_t ldx, int64_t R, const int32_t *d_R, int32_t Kd, int32_t N, const void *wimg,
                   float *Out, int64_t ldo, int epi, const float *aux, int64_t ldaux, cudaStream_t st)
{
    static int attr_done = 0;
    NnParams p{X, ldx, R, d_R, Kd, N, nn_kc(Kd), (const uint8_t *)wimg, Out, ldo, epi, aux, ldaux, 0};
    // weights + max(A chunk, staged accumulator columns): the 32-column groups of the 128-row tile that fit into the A
    // buffer, or into 32 KB where the A chunk is smaller (more would cost residency), as a divisor of N / 32 (full passes)
    const int w_bytes = 2 * N * Kd * 2, a_bytes = 2 * kRows * p.KC * 2, group_bytes = kRows * 32 * 4;
    int groups = std::max(1, std::min(N / 32, std::max(a_bytes, std::min(220 * 1024 - w_bytes, 32 * 1024)) / group_bytes));
    while ((N / 32) % groups) --groups;
    p.stage_cols = groups * 32;
    const int smem = w_bytes + std::max(a_bytes, groups * group_bytes);
    if (!attr_done) {
        CF_TRY(cuda_status(cudaFuncSetAttribute(k_bwd_gemm_nn_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024),
                           "cf_fusion_bwd (nn attr)"));
        attr_done = 1;
    }
    const int per_sm = std::max(1, std::min({(220 * 1024) / (smem + 1024), 512 / tmem_cols(N), 2048 / kNT}));
    const int64_t tiles = ceil_div64(R, kRows);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)sm_count() * per_sm));
    k_bwd_gemm_nn_tc<<<grid, kNT, smem, st>>>(p);
    count_launches(1);
    return launch_status("cf_fusion_bwd (nn)");
}

int det_reduce(const float *part, int32_t M, int32_t n_w, int32_t n_out, int32_t nsplit, int64_t R, const int32_t *d_R,
               int64_t unit, int64_t per_fixed, float *dW, int64_t ldw, int64_t cs, float *db, cudaStream_t st);

// part != nullptr (deterministic mode): kDetSplits / mtiles row splits whatever the GPU, partials summed in split order
int bwd_tc_gemm_tn(const float *X, int64_t ldx, int32_t M, const float *Y, int64_t ldy, int32_t N, const float *Y2,
                   int64_t rs2, int64_t cs2, int32_t n2, const float *wcol, int64_t R, const int32_t *d_R, float *dW,
                   int64_t ldw, float *db, cudaStream_t st, float *part)
{
    static int attr_done = 0;
    const int32_t Nt = (N + n2 + (db ? 1 : 0) + 15) / 16 * 16;
    if (Nt > 256) {
        set_error("cf_fusion_bwd (tn): %d columns exceed one MMA", Nt);
        return CF_ERR_ARG;
    }
    TnParams p{X, ldx, M, Y, ldy, N, Y2, rs2, cs2, n2, wcol, Nt, R, d_R, dW, ldw, db, part};
    const int smem = 2 * (2 * kRows * kTnKC * 2 + 2 * Nt * kTnKC * 2);
    if (!attr_done) {
        CF_TRY(cuda_status(cudaFuncSetAttribute(k_bwd_gemm_tn_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024),
                           "cf_fusion_bwd (tn attr)"));
        attr_done = 1;
    }
    const int mtiles = (M + kRows - 1) / kRows;
    const int per_sm = std::max(1, std::min({(220 * 1024) / (smem + 1024), 512 / tmem_cols(Nt), 2048 / kNT}));
    const int64_t chunks = ceil_div64(R, kTnKC);
    // at least 4 stages of rows per CTA, at most one wave of CTAs
    const int64_t ctas = part ? kDetSplits : (int64_t)sm_count() * per_sm;
    const int64_t splits = std::max<int64_t>(1, std::min<int64_t>(ceil_div64(chunks, 4), ctas / mtiles));
    k_bwd_gemm_tn_tc<<<dim3((unsigned)splits, (unsigned)mtiles), kNT, smem, st>>>(p);
    count_launches(1);
    CF_TRY(launch_status("cf_fusion_bwd (tn)"));
    if (part) {
        const int32_t n_w = N + n2;
        return det_reduce(part, M, n_w, n_w + (db ? 1 : 0), (int32_t)splits, R, d_R, kTnKC, 0, dW, ldw, 1, db, st);
    }
    return CF_OK;
}

}  // namespace cf

// ---- self-tests of the two GEMM shapes (tests/test_gpu_bwd_gemm.py); not part of the reference-facing surface ----------
extern "C" size_t cf_debug_bwd_packed_bytes(int32_t N, int32_t Kd) { return N > 0 && Kd > 0 ? cf::bwd_tc_packed_bytes(N, Kd) : 0; }

extern "C" int cf_debug_bwd_gemm_nn(const float *d_X, int64_t R, const int32_t *d_R, int32_t Kd, int32_t N, const float *d_W,
                                    int32_t transpose, float *d_Out, int32_t epi, const float *d_aux, void *d_packed,
                                    void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_X && d_W && d_Out && d_packed && R > 0, CF_ERR_ARG, "cf_debug_bwd_gemm_nn: null pointer / empty");
    CF_REQUIRE(bwd_tc_nn_fits(Kd, N), CF_ERR_ARG, "cf_debug_bwd_gemm_nn: Kd=%d N=%d has no tensor-core instantiation", Kd, N);
    CF_REQUIRE(epi >= EPI_STORE && epi <= EPI_MASK && (epi < EPI_BIAS_RELU || d_aux), CF_ERR_ARG, "cf_debug_bwd_gemm_nn: bad epilogue");
    CF_REQUIRE(aligned16(d_X) && aligned16(d_Out) && aligned16(d_packed) && (!d_aux || aligned16(d_aux)), CF_ERR_ALIGN,
               "cf_debug_bwd_gemm_nn: 16-byte alignment");
    cudaStream_t st = (cudaStream_t)stream;
    CF_TRY(bwd_tc_pack(d_W, transpose ? N : Kd, N, Kd, transpose, d_packed, st));
    return bwd_tc_gemm_nn(d_X, Kd, R, d_R, Kd, N, d_packed, d_Out, N, epi, d_aux, N, st);
}

// d_dW (M, N + n2) and d_db (M, may be NULL) are accumulated into
extern "C" int cf_debug_bwd_gemm_tn(const float *d_X, int32_t M, const float *d_Y, int32_t N, const float *d_Y2, int32_t n2,
                                    const float *d_wcol, int64_t R, const int32_t *d_R, float *d_dW, float *d_db, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_X && d_dW && R > 0 && (N == 0 || d_Y) && (n2 == 0 || d_Y2) && n2 >= 0 && n2 <= 15, CF_ERR_ARG,
               "cf_debug_bwd_gemm_tn: bad arguments");
    CF_REQUIRE(bwd_tc_tn_fits(M, N), CF_ERR_ARG, "cf_debug_bwd_gemm_tn: M=%d N=%d has no tensor-core instantiation", M, N);
    return bwd_tc_gemm_tn(d_X, M, M, d_Y, N, N, d_Y2, n2, 1, n2, d_wcol, R, d_R, d_dW, N + n2, d_db, (cudaStream_t)stream,
                          nullptr);
}
