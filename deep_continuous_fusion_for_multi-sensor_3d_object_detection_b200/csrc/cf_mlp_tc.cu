// cf_mlp_tc.cu -- K-4 on the 5th-generation tensor cores: per-neighbour MLP layer 2, K-sum-pool, layer 3 and
// the BEV add for one backbone scale, fused so that neither the gathered rows nor the hidden activations
// ever leave the SM.
//
// Tile = 128 BEV cells (= the M of a cta_group::1 UMMA, one TMEM lane per cell) taken from the compacted list of
// cells that have at least one neighbour.  Per tile:
//   for each neighbour slot k:
//     A_k[128 x C]  = relu(T[idx_k] - e_cell)            built by CUDA cores straight into shared memory in the
//                                                         UMMA operand layout, bf16 (+ bf16 residual in fp32 mode)
//     acc[128 x C]  = valid_k * b2 + A_k * W2^T           tcgen05.mma, accumulator in TMEM; the bias rides on an extra
//                                                         K=16 step whose A column is the row's valid flag, so rows
//                                                         without a k-th neighbour come out as exactly 0
//     pooled       += relu(acc)                           tcgen05.ld -> registers -> tcgen05.st (pooled lives in TMEM)
//   acc = n_valid * b3 + pooled * W3^T                    tcgen05.mma (bias column = the row's neighbour count)
//   out = bev + acc                                       epilogue: coalesced NCHW read of bev, write of out
// The same CTAs also copy bev -> out for the cells WITHOUT a neighbour (the other end of the compacted list), so the
// memory-bound copy overlaps the issue-bound MLP tiles of the CTAs that share the SM.
//
// Instruction diet of the two per-(neighbour, channel) loops (they bound the kernel, not HBM or the tensor pipe):
//   operand build  T - (w1x cx + w1y cy): two FFMA2 per channel PAIR; ReLU folded into the bf16 conversions
//                  (cvt.rz.relu / cvt.rn.relu), hi/lo residual with one FADD2 per pair
//   slot epilogue  relu + pooled add: FMNMX + half a FADD2 per channel; no bias add, no valid-mask select
//
// Precision modes
//   CF_MODE_BF16: operands rounded to bf16, fp32 accumulate (tolerance 1e-2, Appendix A12).
//   CF_MODE_FP32: every fp32 operand x is split into bf16 hi + bf16 lo (x ~ hi + lo to 2^-16); the product is
//                 hi*hi + hi*lo + lo*hi, three MMAs into the same fp32 accumulator: relative error ~2^-15 per
//                 product, which keeps the fused features within 1e-4 of the fp32 oracle.
//
// Weights are pre-packed once per call (k_pack_weights) into the shared-memory operand image, chunked along K;
// up to C = 128 both layers stay resident in shared memory for the life of the CTA, above that chunks of 64 input
// channels are streamed from L2 per use.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "cf_common.cuh"
#include "cf_tcgen05.cuh"

namespace cf {

// debugging aids, read from the environment ONCE, when the library first launches a fused kernel.  Neither selects a
// kernel for speed: CF_DEBUG_LAUNCH only prints, and CF_NO_TMA_STORE reaches the direct-store fallback (the path taken
// when the tensor maps cannot be encoded) so that tests can compare it with the TMA-store path.
struct Tuning {
    bool debug_launch = false;    // CF_DEBUG_LAUNCH: print the launch shape
    bool no_tma_store = false;    // CF_NO_TMA_STORE: the layer-1 kernel stores every tile directly (the path taken without tensor maps)
};
static const Tuning &tuning()
{
    static const Tuning t = [] {
        Tuning v;
        v.debug_launch = getenv("CF_DEBUG_LAUNCH") != nullptr;
        v.no_tma_store = getenv("CF_NO_TMA_STORE") != nullptr;
        return v;
    }();
    return t;
}

namespace {

constexpr int kTile = 128;  // cells per tile == UMMA M
constexpr int kThreads = 128;

struct TcParams {
    const float *bev;      // bev / out: elements of the kernel's map type MT (float, or bf16 with CF_IO_BF16)
    const float *T;
    const int32_t *knn;
    float *out;
    const uint8_t *wimg2;  // packed W2 image (chunked)
    const uint8_t *wimg3;
    const float *W1;       // for the offset columns
    const float *b2;
    const float *b3;
    int32_t B, N, H, W, K, Ci;
    float x0, y0, dx, dy;
    int64_t tiles_per_frame, tiles_total;
    // (B, cells) per frame: indices of the cells that have a neighbour from the front, the others from the back
    const int32_t *cell_list;
    const int32_t *cell_count;  // (B) number of cells with a neighbour
    int32_t copy_dead;          // this kernel copies bev -> out for the cells without a neighbour
};

__host__ __device__ constexpr int kc_for(int C, int NS)
{
    // resident when both layers' packed weights + the A tile fit in shared memory, else stream 64-wide chunks
    return C <= 128 ? C : 64;
}

__host__ __device__ constexpr int tmem_cols_for(int cols)
{
    return cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
}

constexpr int kEW = 16;  // TMEM columns per epilogue step
constexpr int kCopyBatch = 16;  // channels per copy unit and thread loaded before the first store
constexpr int kRowBatch = 4;    // NHWC copy units: 16-byte vectors per lane loaded before the first store

// NHWC maps (CF_IO_NHWC): the kEW channels of an epilogue chunk are 16 consecutive elements of the cell's row, moved as
// 16-byte vectors.  Widening and rounding are those of map_ldcs / map_stcs, so the values equal the NCHW path's bit for bit.
__device__ __forceinline__ void row_ldcs16(const float *p, float *v)
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 t = __ldcs(reinterpret_cast<const float4 *>(p) + q);
        v[4 * q] = t.x;
        v[4 * q + 1] = t.y;
        v[4 * q + 2] = t.z;
        v[4 * q + 3] = t.w;
    }
}
__device__ __forceinline__ void row_ldcs16(const __nv_bfloat16 *p, float *v)
{
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const uint4 t = __ldcs(reinterpret_cast<const uint4 *>(p) + q);
        const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            v[8 * q + 2 * i] = __uint_as_float(w[i] << 16);
            v[8 * q + 2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
        }
    }
}
__device__ __forceinline__ void row_stcs16(float *p, const float *v)
{
#pragma unroll
    for (int q = 0; q < 4; ++q) __stcs(reinterpret_cast<float4 *>(p) + q, make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
}
__device__ __forceinline__ void row_stcs16(__nv_bfloat16 *p, const float *v)
{
    auto bits = [](float x) { return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(x)); };
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = bits(v[8 * q + 2 * i]) | (bits(v[8 * q + 2 * i + 1]) << 16);
        __stcs(reinterpret_cast<uint4 *>(p) + q, make_uint4(w[0], w[1], w[2], w[3]));
    }
}
// first element of cell `cell` of frame b (channel 0) in an NCHW or NHWC map
template <bool NHWC>
__device__ __forceinline__ size_t map_cell(int b, int32_t cell, int C, int64_t cells)
{
    return NHWC ? ((size_t)b * cells + cell) * C : (size_t)b * C * cells + cell;
}

// the "row" a cell without a k-th neighbour gathers: relu(-1e30 - e) = 0, so the operand build needs no select
#define CF_NEG8 -1e30f, -1e30f, -1e30f, -1e30f, -1e30f, -1e30f, -1e30f, -1e30f
#define CF_NEG64 CF_NEG8, CF_NEG8, CF_NEG8, CF_NEG8, CF_NEG8, CF_NEG8, CF_NEG8, CF_NEG8
__device__ __align__(32) float g_neg_row[256] = {CF_NEG64, CF_NEG64, CF_NEG64, CF_NEG64};
#undef CF_NEG64
#undef CF_NEG8
// the same row for bf16 tables (CF_MODE_BF16_TABLES): 0xF14A = bf16(-1e30)
#define CF_NEGH8 0xF14A, 0xF14A, 0xF14A, 0xF14A, 0xF14A, 0xF14A, 0xF14A, 0xF14A
#define CF_NEGH64 CF_NEGH8, CF_NEGH8, CF_NEGH8, CF_NEGH8, CF_NEGH8, CF_NEGH8, CF_NEGH8, CF_NEGH8
__device__ __align__(32) uint16_t g_neg_row_h[256] = {CF_NEGH64, CF_NEGH64, CF_NEGH64, CF_NEGH64};
#undef CF_NEGH64
#undef CF_NEGH8

// element type of the layer-1 tables a fused kernel gathers from, and its all-(-1e30) row
template <bool TH>
struct TableT {
    using type = float;
    static __device__ __forceinline__ const float *neg() { return g_neg_row; }
};
template <>
struct TableT<true> {
    using type = __nv_bfloat16;
    static __device__ __forceinline__ const __nv_bfloat16 *neg() { return reinterpret_cast<const __nv_bfloat16 *>(g_neg_row_h); }
};

template <int C, int NS>
struct TcLayout {
    static constexpr int KC = kc_for(C, NS);
    static constexpr bool kResident = KC == C;
    static constexpr int kChunks = C / KC;
    static_assert(C % KC == 0 && KC % 32 == 0, "channel count must be a multiple of the K-chunk");
    static constexpr int kWChunkBytes = NS * C * KC * 2;            // one K-chunk of one layer, all splits
    static constexpr int kWBytes = 2 * kWChunkBytes;                // resident: W2 | W3;  streamed: two chunk buffers
    static constexpr int kABytes = NS * kTile * KC * 2;             // one A tile (all splits)
    static constexpr int kOffA = kWBytes;
    static constexpr int kOffAb = kOffA + kABytes;                  // bias A operand: 128 rows x 16 bf16 (2 units / row)
    static constexpr int kAbBytes = kTile * 32;
    static constexpr int kOffWb = kOffAb + kAbBytes;                // bias B operands: 2 layers x (C rows x 16 bf16)
    static constexpr int kWbBytes = C * 32;
    static constexpr int kOffCtr = kOffWb + 2 * kWbBytes;           // float4 (cx,cx,cy,cy) [2][128]
    static constexpr int kOffCell = kOffCtr + 2 * kTile * 16;       // int32 cell of each row [2][128]
    static constexpr int kOffW1 = kOffCell + 2 * kTile * 4;         // float w1x[C], w1y[C]
    static constexpr int kOffBar = kOffW1 + 2 * C * 4;              // mbarrier (8 B), tmem ptr (4 B), pad, int wmax[2][4], weight-chunk mbarriers [2]
    static constexpr int kOffIdx = kOffBar + 64;                    // int32 [2][K][128] (K known at launch)
    static __host__ __device__ constexpr int smem_bytes(int K) { return kOffIdx + 2 * K * kTile * 4; }
    static constexpr int kTmemCols = tmem_cols_for(2 * C);          // accumulator + the pooled sum
    static_assert(smem_bytes(CF_MAX_K) <= 227 * 1024, "layout exceeds the shared memory of an SM");
};

// ---------------------------------------------------------------------------------------------------------------
// fp32 (rows, cols) weights with row stride ld -> packed operand image:
//   [chunk][split][n/8][k/8 in chunk][n%8][k%8] bf16, chunk = KC consecutive input channels
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_weights(const float *__restrict__ W, int32_t rows, int32_t cols, int32_t ld,
                                                      int32_t KC, int32_t NS, uint8_t *__restrict__ img)
{
    const int32_t units = rows * (cols / 8);  // one 16-byte unit = 8 consecutive k of one n
    const int32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= units) return;
    const int32_t n = u / (cols / 8), k8 = u - n * (cols / 8);
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = W[(size_t)n * ld + k8 * 8 + i];
    uint4 hi, lo;
    tc::split_bf16x8(v, hi, lo, NS == 2);
    const int32_t kc_units = KC / 8;
    const int32_t chunk = k8 / kc_units, ku = k8 - chunk * kc_units;
    const size_t chunk_bytes = (size_t)rows * KC * 2;
    const size_t base = (size_t)chunk * NS * chunk_bytes + tc::unit_offset(n, ku, kc_units);
    *reinterpret_cast<uint4 *>(img + base) = hi;
    if (NS == 2) *reinterpret_cast<uint4 *>(img + base + chunk_bytes) = lo;
}

// linear copy of a packed weight chunk (global/L2 -> shared), 16 bytes per thread per step
template <int NT>
__device__ __forceinline__ void copy_chunk(uint8_t *dst, const uint8_t *__restrict__ src, int bytes)
{
    for (int o = threadIdx.x * 16; o < bytes; o += NT * 16)
        *reinterpret_cast<uint4 *>(dst + o) = __ldg(reinterpret_cast<const uint4 *>(src + o));
}

// issue the MMAs of one K-chunk: acc (+)= A[128 x KC] * Wchunk[C x KC]^T, all split products
template <int C, int NS, int KC>
__device__ __forceinline__ void issue_chunk(uint32_t a_addr, uint32_t w_addr, uint32_t tmem_acc, bool accumulate)
{
    constexpr uint32_t idesc = tc::make_idesc_bf16(kTile, C);
    constexpr uint32_t sbo = (KC / 8) * 128, lbo = 128;
    constexpr uint32_t a_split = kTile * KC * 2, w_split = C * KC * 2;
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int kk = 0; kk < KC / 16; ++kk) {
        const uint32_t koff = kk * 2 * lbo;  // 16 bf16 = two 16-byte k-units
        const uint64_t a_hi = tc::make_desc(a_addr + koff, lbo, sbo);
        const uint64_t w_hi = tc::make_desc(w_addr + koff, lbo, sbo);
        tc::mma_bf16(tmem_acc, a_hi, w_hi, idesc, acc);
        acc = 1u;
        if (NS == 2) {
            const uint64_t a_lo = tc::make_desc(a_addr + a_split + koff, lbo, sbo);
            const uint64_t w_lo = tc::make_desc(w_addr + w_split + koff, lbo, sbo);
            tc::mma_bf16(tmem_acc, a_hi, w_lo, idesc, 1u);
            tc::mma_bf16(tmem_acc, a_lo, w_hi, idesc, 1u);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Cell compaction.  Only ~1/3 of the BEV cells of a LiDAR frame have a point within the radius.  This pass splits
// the cells of each frame into two lists that share one array of `cells` ints: cells WITH a neighbour from the front,
// cells WITHOUT one from the back (block-local order, one atomicAdd per block and list, so each list is a
// concatenation of ascending runs: neighbouring list entries are neighbouring cells and the fused kernel's BEV
// accesses stay coalesced).  count[b] = cells with a neighbour, count[64 + b] = cells without.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cell_compact(const int32_t *__restrict__ knn, int32_t K, int64_t cells,
                                                      int32_t *__restrict__ list, int32_t *__restrict__ count)
{
    __shared__ int32_t warp_live[8], warp_dead[8];
    __shared__ int32_t base_live, base_dead;
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t cell = (int64_t)blockIdx.x * 256 + tid;
    const bool inside = cell < cells;
    const bool live = inside && __ldg(knn + ((size_t)b * cells + cell) * K) >= 0;
    const bool dead = inside && !live;
    const unsigned bal_live = __ballot_sync(0xffffffffu, live), bal_dead = __ballot_sync(0xffffffffu, dead);
    if (lane == 0) {
        warp_live[warp] = __popc(bal_live);
        warp_dead[warp] = __popc(bal_dead);
    }
    __syncthreads();
    if (tid == 0) {
        int32_t run_l = 0, run_d = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const int32_t cl = warp_live[w], cd = warp_dead[w];
            warp_live[w] = run_l;
            warp_dead[w] = run_d;
            run_l += cl;
            run_d += cd;
        }
        base_live = run_l ? atomicAdd(count + b, run_l) : 0;
        base_dead = run_d ? atomicAdd(count + 64 + b, run_d) : 0;
    }
    __syncthreads();
    const unsigned below = (1u << lane) - 1u;
    int32_t *fl = list + (size_t)b * cells;
    if (live) fl[base_live + warp_live[warp] + __popc(bal_live & below)] = (int32_t)cell;
    if (dead) fl[cells - 1 - (base_dead + warp_dead[warp] + __popc(bal_dead & below))] = (int32_t)cell;
}

// Thread layout: G groups of 128 threads.  Thread (row = tid % 128, grp = tid / 128) owns BEV cell `row` of the
// tile; the G threads of a row split the 16-byte operand units of the A tile and the 16-column chunks of the
// epilogues between them (warp w may only touch TMEM lanes 32*(w%4)..+31, which is exactly its rows).
// Launch shape of the two small-C instantiations (measured on B200, BASELINE configs[1]: several small CTAs per SM --
// more independent tiles in flight -- beat fewer barrier rounds per tile; see profiles/README.md).
template <int C>
struct TcShape {
    static constexpr int G = C <= 32 ? 1 : C <= 64 ? 2 : C == 96 || C == 192 ? 3 : 4;
    static constexpr int kMinBlocks = C <= 32 ? 4 : C <= 64 ? 2 : 1;
};

// ---------------------------------------------------------------------------------------------------------------
// Pieces shared by the two fused kernels, k_fusion_tc and k_fusion_sk, which must give bit-identical results.  What
// differs between the kernels (A-buffer address, K-chunk, bias-operand size) is an argument.
// ---------------------------------------------------------------------------------------------------------------

// One-time setup of the negated offset weights and the bias operands (contains a CTA barrier).  The kernel's bias A
// operands (ab_bytes from sAb) are followed by the bias B operands of layer 2 and layer 3 (C rows x 16 bf16 each).
template <int C, int NT>
__device__ __forceinline__ void setup_offsets_and_bias(const TcParams &p, int tid, float *swn, uint8_t *sAb, int ab_bytes)
{
    // negated offset weights, per block of 8 channels: -w1x[8] | -w1y[8]  (what one lane of the operand build needs)
    for (int c = tid; c < C; c += NT) {
        swn[(c >> 3) * 16 + (c & 7)] = -__ldg(p.W1 + (size_t)c * (p.Ci + 3) + p.Ci);
        swn[(c >> 3) * 16 + 8 + (c & 7)] = -__ldg(p.W1 + (size_t)c * (p.Ci + 3) + p.Ci + 1);
    }
    // bias operands.  A side (rewritten per round): row r, k-columns 0 and 1 = the row's flag, the other 14 stay 0.
    // B side: row n = (hi(b[n]), lo(b[n]), 0 ...), so flag * (hi + lo) lands in the accumulator with one K=16 step.
    for (int o = tid * 16; o < ab_bytes + 2 * C * 32; o += NT * 16) *reinterpret_cast<uint4 *>(sAb + o) = make_uint4(0, 0, 0, 0);
    __syncthreads();
    uint8_t *sWb = sAb + ab_bytes;
    for (int n = tid; n < 2 * C; n += NT) {
        const int layer = n / C, c = n - layer * C;
        const float bv = __ldg((layer ? p.b3 : p.b2) + c);
        const __nv_bfloat16 h = __float2bfloat16_rn(bv);
        const __nv_bfloat16 l = __float2bfloat16_rn(bv - __bfloat162float(h));
        const uint32_t packed = (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(l) << 16);
        *reinterpret_cast<uint32_t *>(sWb + layer * C * 32 + tc::unit_offset(c, 0, 2)) = packed;
    }
}

// the bev values of this thread's first kPre output chunks -> tv (they ride in the registers of the gathered rows)
template <int C, int G, int kPre, bool NHWC, typename MT>
__device__ __forceinline__ void prefetch_bev(float *tv, const MT *src_bev, int64_t cells, int grp)
{
#pragma unroll
    for (int j = 0; j < kPre; ++j) {
        if (grp + j * G < C / kEW) {
            if constexpr (NHWC) {
                row_ldcs16(src_bev + (grp + j * G) * kEW, tv + j * kEW);
            } else {
#pragma unroll
                for (int i = 0; i < kEW; ++i) tv[j * kEW + i] = map_ldcs(src_bev + (size_t)((grp + j * G) * kEW + i) * cells);
            }
        }
    }
}

// the final epilogue of one output chunk cc of an NHWC map: out = bev (+ acc z when R > 0), with the bev values from tv
// (prefetched chunks, j < kPre) or loaded here.  The sums are those of the NCHW epilogue.
template <int kPre, typename MT>
__device__ __forceinline__ void final_chunk_nhwc(float *v, const MT *src_bev, int cc, int j, int R, const float *tv, const float *z)
{
    if (j < kPre) {
#pragma unroll
        for (int i = 0; i < kEW; ++i) v[i] = tv[(j & 1) * kEW + i];
    } else {
        row_ldcs16(src_bev + cc * kEW, v);
    }
    if (R > 0) {
#pragma unroll
        for (int i = 0; i < kEW; ++i) v[i] = v[i] + z[i];
    }
}


// ---- layer 3 operand: KC channels of pooled (TMEM, this warp's lanes) -> the A buffer at a_addr; with bias_col, the
// row's bias column = n_valid (acc = n_valid * b3 + pooled * W3^T) ------------------------------------------------
template <int NS, int KC, int G>
__device__ __forceinline__ void pooled_to_operand(uint32_t pool, uint32_t a_addr, int row, int grp, bool bias_col, uint32_t ab_row,
                                                  int n_valid)
{
    constexpr int EW = kEW;
    __syncwarp();
#pragma unroll 1
    for (int cc = grp; cc < KC / EW; cc += G) {
        float s[EW];
        tc::tmem_ld<EW>(pool + cc * EW, s);
#pragma unroll
        for (int q = 0; q < EW / 8; ++q) {
            float2 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = make_float2(s[q * 8 + 2 * i], s[q * 8 + 2 * i + 1]);
            uint4 hi, lo;
            tc::relu_split_bf16x8(v, hi, lo, NS == 2);   // pooled >= 0: the ReLU is the identity here
            const uint32_t off = a_addr + tc::unit_offset(row, cc * (EW / 8) + q, KC / 8);
            tc::sts_u32x4(off, hi);
            if (NS == 2) tc::sts_u32x4(off + kTile * KC * 2, lo);
        }
    }
    if (bias_col && grp == 0) {
        const uint32_t nv16 = __float_as_uint((float)n_valid) >> 16;   // small integers are exact in bf16
        tc::sts_u32(ab_row, nv16 | (nv16 << 16));
    }
}

__device__ __forceinline__ void store_ctr(float4 *s, float cx, float cy) { *s = make_float4(cx, cx, cy, cy); }   // k_fusion_tc
__device__ __forceinline__ void store_ctr(float2 *s, float cx, float cy) { *s = make_float2(cx, cy); }           // k_fusion_sk

// ---- tile sequencing (uniform across the CTA) ------------------------------------------------------------------
// Tile t covers entries [e0, e0 + 128) of frame b's lists: of the cells WITH a neighbour (an MLP tile) and, from the
// other end, of the cells WITHOUT one (a copy unit).  The CTA walks both sequences with two cursors and interleaves
// them, so the memory-bound copies overlap the MLP tiles of the CTAs that share the SM.
// Positions in the tile sequence are (frame b, tile q within the frame); this CTA visits every gridDim.x-th tile.
// The cursors stay in the kernel; Ctr is the kernel's format of a cell centre in the tile header.
template <typename Ctr>
struct TileWalk {
    const TcParams &p;
    const int64_t cells;
    const int32_t tpf;        // tiles per frame
    const int row;            // this thread's row of a tile
    const int K;
    const uint32_t sidx_addr; // tile header, double-buffered by tile parity: int32 [2][K][128] neighbour indices (slot-major),
    Ctr *const sctr;          // [2][128] cell centres
    int32_t *const scell;     // and [2][128] cells (-1: the list ends before the row)
    int32_t *const swmax;     // [2][4] per warp of group 0: its largest neighbour count

    __device__ __forceinline__ int32_t n_live_of(int b) const { return p.cell_list ? __ldg(p.cell_count + b) : (int32_t)cells; }
    __device__ __forceinline__ void advance(int32_t &b, int32_t &q, int32_t step) const
    {
        q += step;
        while (q >= tpf) {
            q -= tpf;
            ++b;
        }
    }
    // forward (inclusive) to the next tile that has rows; b == B: none
    __device__ __forceinline__ void seek_live(int32_t &b, int32_t &q) const
    {
        while (b < p.B && q * kTile >= n_live_of(b)) advance(b, q, (int32_t)gridDim.x);
    }
    // this CTA's first MLP tile (cb, cq) and copy unit (db, dq); fill: this thread prefetches its row of the first header
    __device__ __forceinline__ void start(int32_t &cb, int32_t &cq, int32_t &db, int32_t &dq, bool fill) const
    {
        advance(cb, cq, (int32_t)blockIdx.x);
        seek_live(cb, cq);
        if (p.copy_dead) advance(db, dq, (int32_t)blockIdx.x); else db = p.B;
        if (cb < p.B && fill) header_fill(cb, header_cell(cb, cq), 0);
    }
    // Tile header, prefetched one tile ahead by the 128 threads of group 0 (thread = row).
    //   stage 1: the row's cell (-1: the list ends before this row)
    //   stage 2: its K neighbour indices straight into shared memory (cp.async, slot-major), centre and cell
    __device__ __forceinline__ int32_t header_cell(int32_t b, int32_t q) const
    {
        const int32_t e = q * kTile + row;
        if (e >= n_live_of(b)) return -1;
        return p.cell_list ? __ldg(p.cell_list + (size_t)b * cells + e) : e;
    }
    __device__ __forceinline__ void header_fill(int32_t b, int32_t cell, int par) const
    {
        const uint32_t dst = sidx_addr + (uint32_t)((par * K * kTile + row) * 4);
        float cx = 0.f, cy = 0.f;
        if (cell >= 0) {
            const int32_t *kr = p.knn + ((size_t)b * cells + cell) * K;
            for (int k = 0; k < K; ++k) tc::cp_async4(dst + k * kTile * 4, kr + k);
            const int32_t i = (int32_t)((uint32_t)cell / (uint32_t)p.W), j = cell - i * p.W;
            cx = __fadd_rn(p.x0, __fmul_rn((float)i, p.dx));
            cy = __fadd_rn(p.y0, __fmul_rn((float)j, p.dy));
        } else {
            for (int k = 0; k < K; ++k) tc::sts_u32(dst + k * kTile * 4, 0xFFFFFFFFu);
        }
        tc::cp_async_commit();
        store_ctr(sctr + par * kTile + row, cx, cy);
        scell[par * kTile + row] = cell;
    }
    // The prefetched header of the tile with parity par (contains a CTA barrier): returns the tile's round count, the
    // neighbour count of its best-connected cell; n_valid (group 0, grp0) = this row's neighbour count.
    __device__ __forceinline__ int read_header(int par, bool grp0, int lane, int warp, int &n_valid) const
    {
        if (grp0) {
            tc::cp_async_wait_all();
            for (int k = 0; k < K; ++k) n_valid += (int32_t)tc::lds_u32(sidx_addr + (uint32_t)(((par * K + k) * kTile + row) * 4)) >= 0;
            const int wm = __reduce_max_sync(0xffffffffu, n_valid);
            if (lane == 0) swmax[par * 4 + warp] = wm;
        }
        __syncthreads();
        const int4 wm = *reinterpret_cast<const int4 *>(swmax + par * 4);
        return max(max(wm.x, wm.y), max(wm.z, wm.w));
    }
    // the list entries of the next two copy units from cursor (db, dq): frame (uniform, -1: none left) and this thread's
    // cell (-1: past the end of the list)
    __device__ __forceinline__ void fetch_units(int32_t &db, int32_t &dq, int32_t (&uframe)[2], int32_t (&ucell)[2]) const
    {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            uframe[u] = -1;
            ucell[u] = -1;
            int32_t n_dead = 0;
            while (db < p.B) {
                n_dead = (int32_t)cells - n_live_of(db);
                if (dq * kTile < n_dead) break;
                advance(db, dq, (int32_t)gridDim.x);
            }
            if (db < p.B) {
                uframe[u] = db;
                const int32_t j = dq * kTile + row;
                if (j < n_dead) ucell[u] = __ldg(p.cell_list + (size_t)db * cells + (cells - 1 - j));
                advance(db, dq, (int32_t)gridDim.x);
            }
        }
    }
};

// ---- copy units: cells without a neighbour (back of the list): out = bev ----------------------------------------
// (thread = cell, the G thread groups split the channels; two units are interleaved after every MLP tile; their list
// entries were fetched at the start of the tile, so a unit costs one DRAM round trip per channel batch)
// NHWC: a cell's channels are one row, so the warp copies the rows of its 32 cells (this group's C / G channels of each)
// with 16-byte accesses, consecutive lanes on consecutive vectors of a row; the cell of row r comes from lane r.
template <int C, int G, typename MT, bool NHWC>
__device__ __forceinline__ void copy_units(const TcParams &p, const int32_t (&uframe)[2], const int32_t (&ucell)[2], int grp, int64_t cells)
{
    if constexpr (NHWC) {
        constexpr int V = C / G * (int)sizeof(MT) / 16;   // 16-byte vectors per row and group
        static_assert(V % kRowBatch == 0, "whole batches per row");
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (uframe[u] >= 0) {   // uniform
                const size_t o = (size_t)uframe[u] * cells * C + grp * (C / G);
                const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const MT *>(p.bev) + o);
                uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<MT *>(p.out) + o);
#pragma unroll 1
                for (int i0 = lane; i0 < 32 * V; i0 += 32 * kRowBatch) {
                    uint4 v[kRowBatch];
                    int64_t e[kRowBatch];
#pragma unroll
                    for (int t = 0; t < kRowBatch; ++t) {
                        const int i = i0 + 32 * t, r = i / V;
                        const int32_t cell = __shfl_sync(0xffffffffu, ucell[u], r);   // < 0: past the end of the list
                        e[t] = cell >= 0 ? (int64_t)cell * (C * (int)sizeof(MT) / 16) + (i - r * V) : -1;
                        if (e[t] >= 0) v[t] = __ldcs(src + e[t]);
                    }
#pragma unroll
                    for (int t = 0; t < kRowBatch; ++t)
                        if (e[t] >= 0) __stcs(dst + e[t], v[t]);
                }
            }
        }
        return;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        if (uframe[u] >= 0 && ucell[u] >= 0) {   // uframe is uniform; ucell < 0: a row past the end of the list
            constexpr int CG = C / G;
            const size_t o = ((size_t)uframe[u] * C + grp * CG) * cells + ucell[u];
            using RB = typename MapBits<MT>::type;   // a bf16 map is copied as raw 16-bit elements
            const RB *src = reinterpret_cast<const RB *>(p.bev) + o;
            RB *dst = reinterpret_cast<RB *>(p.out) + o;
#pragma unroll 1
            for (int c = 0; c < CG; c += kCopyBatch) {   // kCopyBatch loads in flight per thread, then the stores
                RB v[kCopyBatch];
#pragma unroll
                for (int i = 0; i < kCopyBatch; ++i) {
                    v[i] = __ldcs(src);
                    src += cells;
                }
#pragma unroll
                for (int i = 0; i < kCopyBatch; ++i) {
                    __stcs(dst, v[i]);
                    dst += cells;
                }
            }
        }
    }
}

// wait for the last copies, then free the tensor memory
__device__ __forceinline__ void teardown(uint32_t tmem_base, int tmem_cols, int warp)
{
    tc::cp_async_wait_all();
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem_base, tmem_cols);
}

template <int C, int NS, bool TH = false, typename MT = float, bool NHWC = false>
__global__ void __launch_bounds__(kTile * TcShape<C>::G, TcShape<C>::kMinBlocks) k_fusion_tc(const TcParams p)
{
    using TT = typename TableT<TH>::type;   // fp32 tables, or bf16 tables in CF_MODE_BF16_TABLES (NS == 1)
    const TT *const g_neg = TableT<TH>::neg();
    using L = TcLayout<C, NS>;
    constexpr int G = TcShape<C>::G, EW = kEW;
    constexpr int NT = kTile * G;
    constexpr int KC = L::KC;
    constexpr int kc_units = KC / 8;
    constexpr int kChunksE = C / EW;  // epilogue chunks over all C columns
    static_assert(C % G == 0 && (C / G) % 32 == 0, "column split between the thread groups");
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *sW = smem;
    uint8_t *sA = smem + L::kOffA;
    uint8_t *sAb = smem + L::kOffAb;
    uint8_t *sWb = smem + L::kOffWb;
    float4 *sctr = reinterpret_cast<float4 *>(smem + L::kOffCtr);
    int32_t *scell = reinterpret_cast<int32_t *>(smem + L::kOffCell);
    float *swn = reinterpret_cast<float *>(smem + L::kOffW1);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::kOffBar);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::kOffBar + 8);
    int32_t *swmax = reinterpret_cast<int32_t *>(smem + L::kOffBar + 16);   // [2][4]
    int32_t *sidx = reinterpret_cast<int32_t *>(smem + L::kOffIdx);         // [2][K][128]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & (kTile - 1), grp = tid / kTile;
    constexpr int NW = NT / 32;
    const int K = p.K;
    const int64_t cells = (int64_t)p.H * p.W;

    // ---- one-time setup -----------------------------------------------------------------------------------------
    const uint32_t wbar = tc::smem_u32(smem + L::kOffBar + 48);   // [2]: a streamed weight chunk has landed in its buffer
    if (tid == 0) {
        tc::mbar_init(bar, 1);
        tc::mbar_init(reinterpret_cast<uint64_t *>(smem + L::kOffBar + 48), 1);
        tc::mbar_init(reinterpret_cast<uint64_t *>(smem + L::kOffBar + 56), 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(tmem_slot, L::kTmemCols);
    setup_offsets_and_bias<C, NT>(p, tid, swn, sAb, L::kAbBytes);
    // Streamed weights (C > 128): chunks of KC input channels travel L2 -> shared memory as ONE bulk copy each (TMA engine,
    // cp.async.bulk; the packed chunk is contiguous) into two buffers, always one chunk ahead of the MMAs; only the thread that
    // issues the MMAs waits for a chunk (mbarrier complete_tx).  `wn` counts the chunks consumed so far: chunk wn lives in
    // buffer wn & 1 and is that buffer's (wn >> 1)-th use.  (Called by ONE thread.)
    uint32_t wn = 0;
    auto prefetch_wchunk = [&](const uint8_t *src, uint32_t buf) {
        tc::mbar_expect_tx(wbar + buf * 8, L::kWChunkBytes);
        tc::bulk_load_1d(tc::smem_u32(sW) + buf * L::kWChunkBytes, src, L::kWChunkBytes, wbar + buf * 8);
    };
    if (L::kResident) {
        copy_chunk<NT>(sW, p.wimg2, L::kWChunkBytes);
        copy_chunk<NT>(sW + L::kWChunkBytes, p.wimg3, L::kWChunkBytes);
    } else if (tid == 0) {
        prefetch_wchunk(p.wimg2, 0);
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_acc = tmem_base;                                // accumulator: columns [0, C)
    const uint32_t tmem_pool = tmem_base + C;                           // pooled sum:  columns [C, 2C)
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;        // this warp's TMEM lanes == its rows
    const uint32_t sA_addr = tc::smem_u32(sA), sW_addr = tc::smem_u32(sW);
    const uint32_t sAb_addr = tc::smem_u32(sAb), sWb_addr = tc::smem_u32(sWb);
    const uint32_t sidx_addr = tc::smem_u32(sidx), sctr_addr = tc::smem_u32(sctr);
    const uint32_t ab_row = sAb_addr + tc::unit_offset(row, 0, 2);
    constexpr uint32_t idesc = tc::make_idesc_bf16(kTile, C);
    uint32_t phase = 0, iter = 0;
    // the thread that issues the MMAs (called by every thread right behind a CTA barrier).  Wide shapes (1 CTA per SM, spare
    // registers): an elected lane of warp 0, so that ptxas keeps the descriptors in uniform registers and the 12 + MMAs of a chunk
    // step go out back to back; under `tid == 0` every UTCHMMA sits in its own ELECT / BRA.U.ANY loop (~70 cycles each), which
    // the narrow shapes accept because the elected form costs them registers (measured: spills, 266 -> 275 us at C = 32).
    auto issuer = [&]() -> bool {
        if constexpr (C >= 192) return warp == 0 && tc::elect_one();
        else return tid == 0;
    };

    // A-tile work split: a warp takes one 8-row group x 4 operand units (32 channels) per step, lane (r8 = lane % 8,
    // u = lane / 8).  Global side: the 4 lanes of a row read one contiguous 128-byte segment of the point's T row;
    // shared side: each quarter-warp (the unit of a 128-bit shared access) writes the 8 rows of one unit = 128 contiguous
    // bytes of the operand image: conflict free.  NW is a multiple of the unit-quads per row, so a warp always works on
    // the same 32 channels of a chunk and its negated offset weights stay in registers.
    constexpr int kQuads = kc_units / 4;
    static_assert(NW % kQuads == 0, "warps per CTA must be a multiple of the unit quads per row");
    constexpr int kStep = NW / kQuads;   // row groups between two items of a warp
    const int ku = (warp % kQuads) * 4 + (lane >> 3);
    const int r8 = lane & 7;
    const int rg0 = warp / kQuads;
    // -(w1x, w1y) of this lane's 8 channels:  T - (w1x cx + w1y cy) = two FFMA2 per channel pair.  Reloaded from shared
    // memory at the start of every round's build (4 LDS.128) rather than held across the whole tile.
    float2 nx[4], ny[4];
    const uint32_t swn_addr = tc::smem_u32(swn);
    auto load_offset_weights = [&](int ch) {
        const uint32_t a = swn_addr + (uint32_t)((ch * kc_units + ku) * 64);
        const float4 x0 = tc::lds_f32x4(a), x1 = tc::lds_f32x4(a + 16), y0 = tc::lds_f32x4(a + 32), y1 = tc::lds_f32x4(a + 48);
        nx[0] = make_float2(x0.x, x0.y); nx[1] = make_float2(x0.z, x0.w); nx[2] = make_float2(x1.x, x1.y); nx[3] = make_float2(x1.z, x1.w);
        ny[0] = make_float2(y0.x, y0.y); ny[1] = make_float2(y0.z, y0.w); ny[2] = make_float2(y1.x, y1.y); ny[3] = make_float2(y1.z, y1.w);
    };

    const TileWalk<float4> walk{p, cells, (int32_t)p.tiles_per_frame, row, K, sidx_addr, sctr, scell, swmax};

    // ---- operand build ---------------------------------------------------------------------------------------------
    // one item = 8 rows x 32 channels per warp: lane (r8, u) turns 8 channels of one neighbour row into two 16-byte
    // operand units (hi, lo).  Per item and lane: 2 LDS, 2 LDG.128, 8 FFMA2, 8 F2FP, 8 unpack, 4 FADD2, 2 STS.128 --
    // rows without a k-th neighbour read a row of -1e30, which the fused ReLU turns into zeros.
    auto gather = [&](const TT *Tc, const TT *neg, uint32_t idx_addr, float *t) {   // t[8]
        const int32_t pr = (int32_t)tc::lds_u32(idx_addr);
        // one 256-bit load per lane: the 4 lanes of a row fetch one full 128-byte line in a single request
        tc::ldg_row8(pr >= 0 ? Tc + (size_t)pr * C : neg, t);
    };
    auto build = [&](const float *t, const float4 &ctr, uint32_t dst_addr) {
        const float2 cxx = make_float2(ctr.x, ctr.y), cyy = make_float2(ctr.z, ctr.w);
        float2 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = tc::ffma2(nx[i], cxx, tc::ffma2(ny[i], cyy, make_float2(t[2 * i], t[2 * i + 1])));
        uint4 hi, lo;
        tc::relu_split_bf16x8(v, hi, lo, NS == 2);
        tc::sts_u32x4(dst_addr, hi);
        if (NS == 2) tc::sts_u32x4(dst_addr + kTile * KC * 2, lo);
    };

    int32_t cb = 0, cq = 0, db = 0, dq = 0;   // cursors: MLP tiles (cb, cq), copy units (db, dq)
    walk.start(cb, cq, db, dq, grp == 0);

    int32_t uframe[2] = {-1, -1}, ucell[2] = {-1, -1};   // the next two copy units (TileWalk::fetch_units)
    bool units_ready = false;

    while (cb < p.B || db < p.B) {
        if (cb < p.B) {
            const int par = iter & 1;
            ++iter;
            const int b = cb;
            // list entries of the copy units that follow this tile: in flight during the whole tile (at C = 32 this used to push
            // the mbarrier phase into local memory, 264 -> 283 us; with the gathers moved in front of the barrier it fits:
            // 260 -> 256 us)
            walk.fetch_units(db, dq, uframe, ucell);
            units_ready = true;
            int32_t nb = cb, nq = cq;
            walk.advance(nb, nq, (int32_t)gridDim.x);
            walk.seek_live(nb, nq);
            const bool has_next = nb < p.B;
            // ---- header of this tile (prefetched): rounds = neighbour count of its best-connected cell -----------------
            int n_valid = 0;
            const int R = walk.read_header(par, grp == 0, lane, warp, n_valid);
            const int32_t cell = scell[par * kTile + row];
            const bool in_range = cell >= 0;
            int32_t ncell = -1;   // stage 1 of the next tile's header: in flight during round 0
            if (grp == 0 && has_next) ncell = walk.header_cell(nb, nq);
            if (R == 0 && grp == 0 && has_next) walk.header_fill(nb, ncell, par ^ 1);

            const TT *Tb = reinterpret_cast<const TT *>(p.T) + (size_t)b * p.N * C;
            const uint32_t idx0 = sidx_addr + (uint32_t)((par * K * kTile + rg0 * 8 + r8) * 4);
            const uint32_t ctr0 = sctr_addr + (uint32_t)((par * kTile + rg0 * 8 + r8) * 16);
            const uint32_t dst0 = sA_addr + tc::unit_offset(r8, ku, kc_units) + (uint32_t)(rg0 * kc_units * 128);
            const MT *src_bev = reinterpret_cast<const MT *>(p.bev) + map_cell<NHWC>(b, cell, C, cells);
            // Pipelined shapes (both layers resident, 4 items per warp and round): tv holds the gathered neighbour rows
            // of the NEXT round while this round's MMA and epilogue run; in the last round the same 32 registers take the
            // bev values of this thread's first two output chunks instead.
            constexpr bool kPipe = L::kChunks == 1 && kStep == 4;
            constexpr int kPre = kPipe ? 2 : 0;   // output chunks whose bev values are prefetched
            constexpr bool kGatherEarly = kPipe && C <= 32;
            float tv[32];
            auto prefetch_tv = [&]() {
                if (in_range) prefetch_bev<C, G, kPre, NHWC>(tv, src_bev, cells, grp);
            };
            if (kPipe && R > 0) {
                const TT *Tc = Tb + ku * 8, *neg = g_neg + ku * 8;
#pragma unroll
                for (int i = 0; i < 4; ++i) gather(Tc, neg, idx0 + i * kStep * 32, tv + 8 * i);
            }
            // Chunked shapes (C > 128: a round is kChunks chunk steps of KC input channels): the neighbour rows of the NEXT
            // chunk step are gathered into registers right after this step's MMAs are issued and are built after its wait --
            // the L2 round trip of the gather (~1 us of a ~3 us chunk step) leaves the tile's chain.
            constexpr bool kPipe2 = !kPipe && L::kChunks > 1;
            static_assert(kPipe || kPipe2, "every shape builds its operands in one of the two pipelined forms");
            constexpr int kMaxItems = (16 + kStep - 1) / kStep;
            float pv[kPipe2 ? kMaxItems * 8 : 1];
            auto gather_chunk = [&](int k, int ch) {
                const TT *Tc = Tb + ch * KC + ku * 8, *neg = g_neg + ch * KC + ku * 8;
#pragma unroll
                for (int m = 0; m < kMaxItems; ++m)
                    if (rg0 + m * kStep < 16) gather(Tc, neg, idx0 + (uint32_t)(k * kTile * 4 + m * kStep * 32), pv + 8 * m);
            };
            if (kPipe2 && R > 0) gather_chunk(0, 0);
            if (R == 0) prefetch_tv();

            for (int k = 0; k < R; ++k) {
                const uint32_t idxk = idx0 + (uint32_t)(k * kTile * 4);
                for (int ch = 0; ch < L::kChunks; ++ch) {
                    if (kPipe) {
                        load_offset_weights(0);
                        // rows were gathered while the previous round's MMA and epilogue ran
                        // (the centre of item i+1 is loaded before item i is stored: the shared-memory latency hides
                        // behind the arithmetic of the previous item)
                        float4 ctr = tc::lds_f32x4(ctr0);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            float4 ctr_next = ctr;
                            if (i < 3) ctr_next = tc::lds_f32x4(ctr0 + (i + 1) * kStep * 128);
                            build(tv + 8 * i, ctr, dst0 + i * kStep * kc_units * 128);
                            ctr = ctr_next;
                        }
                    } else {
                        load_offset_weights(ch);
#pragma unroll
                        for (int m = 0; m < kMaxItems; ++m) {
                            if (rg0 + m * kStep < 16) {
                                const float4 cm = tc::lds_f32x4(ctr0 + m * kStep * 128);
                                build(pv + 8 * m, cm, dst0 + m * kStep * kc_units * 128);
                            }
                        }
                    }
                    if (ch == 0 && grp == 0)   // bias flag of the row: bf16 (1, 1) or (0, 0)
                        tc::sts_u32(ab_row, (int32_t)tc::lds_u32(sidx_addr + (uint32_t)(((par * K + k) * kTile + row) * 4)) >= 0 ? 0x3F803F80u : 0u);
                    if (kGatherEarly) {
                        // the next round's neighbour rows (their registers are free again): issued BEFORE the barrier and the MMA
                        // issue, so they get the barrier skew and the issue time as extra lead and the issuing warp does not lag
                        // (C = 32: 266 -> 260 us out of place, 184 -> 178 us in place; neutral at C = 64, where it adds spills)
                        if (k + 1 < R) {
                            const TT *Tc = Tb + ku * 8, *neg = g_neg + ku * 8;
#pragma unroll
                            for (int i = 0; i < 4; ++i) gather(Tc, neg, idxk + kTile * 4 + i * kStep * 32, tv + 8 * i);
                        } else {
                            prefetch_tv();
                        }
                    }
                    tc::fence_proxy_async();
                    tc::fence_before_sync();
                    __syncthreads();
                    if (issuer()) {
                        if (!L::kResident) tc::mbar_wait_a(wbar + (wn & 1) * 8, (wn >> 1) & 1u);   // this step's weight chunk has landed
                        tc::fence_after_sync();
                        if (ch == 0)
                            tc::mma_bf16(tmem_acc, tc::make_desc(sAb_addr, 128, 256), tc::make_desc(sWb_addr, 128, 256), idesc, 0u);
                        issue_chunk<C, NS, KC>(sA_addr, sW_addr + (L::kResident ? 0 : (wn & 1) * L::kWChunkBytes), tmem_acc, true);
                        tc::commit(bar);
                        if (!L::kResident) {
                            // next chunk in the tile's fixed sequence: W2 chunks of every round, then the W3 chunks; its buffer was
                            // last read by the previous chunk step's MMAs, which every thread has seen complete
                            const uint8_t *nsrc = ch + 1 < L::kChunks ? p.wimg2 + (size_t)(ch + 1) * L::kWChunkBytes
                                                  : k + 1 < R        ? p.wimg2
                                                                     : p.wimg3;
                            prefetch_wchunk(nsrc, (wn + 1) & 1);
                        }
                    }
                    if (!L::kResident) ++wn;
                    if (kPipe2) {   // the next chunk step's rows: this round's next chunk, or the first chunk of the next round
                        if (ch + 1 < L::kChunks) gather_chunk(k, ch + 1);
                        else if (k + 1 < R) gather_chunk(k + 1, 0);
                    }
                    if (ch == L::kChunks - 1) {
                        // work that overlaps this round's MMA and epilogue: the next tile's header, then the next round's
                        // gathers (or, in the last round, the bev values of the final epilogue)
                        if (k == 0 && grp == 0 && has_next) walk.header_fill(nb, ncell, par ^ 1);
                        if (k + 1 < R) {
                            if (kPipe && !kGatherEarly) {
                                const TT *Tc = Tb + ku * 8, *neg = g_neg + ku * 8;
#pragma unroll
                                for (int i = 0; i < 4; ++i) gather(Tc, neg, idxk + kTile * 4 + i * kStep * 32, tv + 8 * i);
                            }
                        } else if (!kGatherEarly) {
                            prefetch_tv();
                        }
                    }
                    tc::mbar_wait(bar, phase);
                    phase ^= 1u;
                    tc::fence_after_sync();
                }
                // ---- epilogue of the round: pooled (+)= relu(acc)   (bias and valid mask are already inside acc) -----------
                __syncwarp();
#pragma unroll 1
                for (int cc = grp; cc < kChunksE; cc += G) {
                    float z[EW], s[EW];
                    if (k > 0) {
                        tc::tmem_ld16x2(tmem_acc + lane_off + cc * EW, tmem_pool + lane_off + cc * EW, z, s);
#pragma unroll
                        for (int i = 0; i < EW; i += 2) {
                            const float2 a = tc::fadd2(make_float2(s[i], s[i + 1]), make_float2(fmaxf(z[i], 0.f), fmaxf(z[i + 1], 0.f)));
                            s[i] = a.x;
                            s[i + 1] = a.y;
                        }
                    } else {
                        tc::tmem_ld<EW>(tmem_acc + lane_off + cc * EW, z);
#pragma unroll
                        for (int i = 0; i < EW; ++i) s[i] = fmaxf(z[i], 0.f);
                    }
                    tc::tmem_st<EW>(tmem_pool + lane_off + cc * EW, s);
                }
                tc::fence_before_sync();  // TMEM accesses above are ordered before the next MMA by the next barrier
            }

            if (R > 0) {
                // ---- layer 3: acc = n_valid * b3 + pooled * W3^T -----------------------------------------------------------
                for (int ch = 0; ch < L::kChunks; ++ch) {
                    pooled_to_operand<NS, KC, G>(tmem_pool + lane_off + ch * KC, sA_addr, row, grp, ch == 0, ab_row, n_valid);
                    tc::fence_proxy_async();
                    tc::fence_before_sync();
                    __syncthreads();
                    if (issuer()) {
                        if (!L::kResident) tc::mbar_wait_a(wbar + (wn & 1) * 8, (wn >> 1) & 1u);
                        tc::fence_after_sync();
                        if (ch == 0)
                            tc::mma_bf16(tmem_acc, tc::make_desc(sAb_addr, 128, 256), tc::make_desc(sWb_addr + L::kWbBytes, 128, 256),
                                         idesc, 0u);
                        issue_chunk<C, NS, KC>(sA_addr, sW_addr + (L::kResident ? L::kWChunkBytes : (wn & 1) * L::kWChunkBytes), tmem_acc, true);
                        tc::commit(bar);
                        if (!L::kResident) {   // next: the following W3 chunk, or the first W2 chunk for the next tile
                            const uint8_t *nsrc = ch + 1 < L::kChunks ? p.wimg3 + (size_t)(ch + 1) * L::kWChunkBytes : p.wimg2;
                            prefetch_wchunk(nsrc, (wn + 1) & 1);
                        }
                    }
                    if (!L::kResident) ++wn;
                    tc::mbar_wait(bar, phase);
                    phase ^= 1u;
                    tc::fence_after_sync();
                }
            }
            // ---- final epilogue: out = bev + acc (thread = cell: a warp touches 128 contiguous bytes per channel) ---------
            __syncwarp();
            if (R > 0 || p.out != p.bev) {
                MT *dst_out = reinterpret_cast<MT *>(p.out) + map_cell<NHWC>(b, cell, C, cells);
#pragma unroll
                for (int j = 0; j < (kChunksE + G - 1) / G; ++j) {
                    const int cc = grp + j * G;
                    if (cc < kChunksE) {
                        float z[EW];
                        if (R > 0) tc::tmem_ld<EW>(tmem_acc + lane_off + cc * EW, z);
                        if constexpr (NHWC) {
                            if (in_range) {
                                float v[EW];
                                final_chunk_nhwc<kPre>(v, src_bev, cc, j, R, tv, z);
                                row_stcs16(dst_out + cc * EW, v);
                            }
                        } else if (in_range) {
                            if (j < kPre) {
#pragma unroll
                                for (int i = 0; i < EW; ++i)
                                    map_stcs(dst_out + (size_t)(cc * EW + i) * cells, R > 0 ? tv[(j & 1) * EW + i] + z[i] : tv[(j & 1) * EW + i]);
                            } else {
#pragma unroll
                                for (int h = 0; h < EW; h += 8) {   // 8 loads in flight, then 8 stores
                                    float bv[8];
#pragma unroll
                                    for (int i = 0; i < 8; ++i) bv[i] = map_ldcs(src_bev + (size_t)(cc * EW + h + i) * cells);
#pragma unroll
                                    for (int i = 0; i < 8; ++i)
                                        map_stcs(dst_out + (size_t)(cc * EW + h + i) * cells, R > 0 ? bv[i] + z[h + i] : bv[i]);
                                }
                            }
                        }
                    }
                }
            }
            // no barrier here: the tile header state (indices, centres, cells, round count) is double-buffered by tile
            // parity, and every other shared / tensor-memory buffer is only rewritten behind the next tile's first barrier
            tc::fence_before_sync();
            cb = nb;
            cq = nq;
        }
        if (!units_ready) walk.fetch_units(db, dq, uframe, ucell);
        units_ready = false;
        copy_units<C, G, MT, NHWC>(p, uframe, ucell, grp, cells);
    }

    if (!L::kResident && tid == 0) tc::mbar_wait_a(wbar + (wn & 1) * 8, (wn >> 1) & 1u);   // the weight chunk prefetched for a tile that never came
    teardown(tmem_base, L::kTmemCols, warp);
}

// ---------------------------------------------------------------------------------------------------------------
// k_fusion_sk: the fused kernel for C <= 128 with the MMAs taken off the tile's critical path.  Same tiles, same operand
// build, same epilogues and the same arithmetic as k_fusion_tc (bit-identical results), but two A buffers, two bias
// operands, two TMEM accumulators and two mbarriers: round k+1 is built and issued while the MMAs of round k run, and the
// epilogue of round k runs under the MMAs of round k+1:
//     prologue   build(0) | sync | issue(0) | gather(1)
//     round k    build(k+1) | sync | issue(k+1) | gather(k+2) | wait(k) | epilogue(k)
//     layer 3    pooled -> A | sync | issue | wait | out = bev + acc
// To keep the occupancy of k_fusion_tc with the second A buffer, W3 is not resident: it streams (cp.async) into the A
// buffer that the last round does not use, during the last-but-one round's epilogue.
// ---------------------------------------------------------------------------------------------------------------
template <int C, int NS>
struct SkLayout {
    static constexpr int kWBytes = NS * C * C * 2;                  // one layer's packed image (W2 resident; W3 streamed)
    static constexpr int kABytes = NS * kTile * C * 2;              // one A tile (all splits)
    static_assert(kWBytes <= kABytes, "W3 is staged in an A buffer");
    static constexpr int kOffA = kWBytes;                           // A[2]
    static constexpr int kAbBytes = kTile * 32;
    static constexpr int kOffAb = kOffA + 2 * kABytes;              // Ab[2]
    static constexpr int kWbBytes = C * 32;
    static constexpr int kOffWb = kOffAb + 2 * kAbBytes;            // bias B operands of layer 2 | layer 3
    static constexpr int kOffCtr = kOffWb + 2 * kWbBytes;           // float2 (cx, cy) [2][128]
    static constexpr int kOffCell = kOffCtr + 2 * kTile * 8;        // int32 [2][128]
    static constexpr int kOffW1 = kOffCell + 2 * kTile * 4;         // negated offset weights
    static constexpr int kOffBar = kOffW1 + 2 * C * 4;              // mbarrier[2] (16 B), tmem ptr (4 B), pad, int wmax[2][4]
    static constexpr int kOffIdx = kOffBar + 64;                    // int32 [2][K][128]
    static __host__ __device__ constexpr int smem_bytes(int K) { return kOffIdx + 2 * K * kTile * 4; }
    static constexpr int kTmemCols = tmem_cols_for(3 * C);          // two accumulators + the pooled sum
};

template <int C, int NS, bool TH = false, typename MT = float, bool NHWC = false>
__global__ void __launch_bounds__(kTile * TcShape<C>::G, TcShape<C>::kMinBlocks) k_fusion_sk(const TcParams p)
{
    using TT = typename TableT<TH>::type;
    const TT *const g_neg = TableT<TH>::neg();
    using L = SkLayout<C, NS>;
    constexpr int G = TcShape<C>::G, EW = kEW;
    constexpr int NT = kTile * G, NW = NT / 32;
    constexpr int kc_units = C / 8, kQuads = kc_units / 4, kStep = NW / kQuads;
    constexpr int kChunksE = C / EW;
    static_assert(NW % kQuads == 0 && 16 % kStep == 0 && 16 / kStep == 4, "4 operand items per warp and round");
    static_assert(C % G == 0 && (C / G) % 32 == 0, "column split between the thread groups");
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *sW = smem;
    uint8_t *sAb = smem + L::kOffAb;
    uint8_t *sWb = smem + L::kOffWb;
    float2 *sctr = reinterpret_cast<float2 *>(smem + L::kOffCtr);
    int32_t *scell = reinterpret_cast<int32_t *>(smem + L::kOffCell);
    float *swn = reinterpret_cast<float *>(smem + L::kOffW1);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::kOffBar);          // [2]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::kOffBar + 16);
    int32_t *swmax = reinterpret_cast<int32_t *>(smem + L::kOffBar + 32);     // [2][4]
    int32_t *sidx = reinterpret_cast<int32_t *>(smem + L::kOffIdx);           // [2][K][128]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & (kTile - 1), grp = tid / kTile;
    const int K = p.K;
    const int64_t cells = (int64_t)p.H * p.W;

    // ---- one-time setup -----------------------------------------------------------------------------------------
    if (tid == 0) {
        tc::mbar_init(&bar[0], 1);
        tc::mbar_init(&bar[1], 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(tmem_slot, L::kTmemCols);
    setup_offsets_and_bias<C, NT>(p, tid, swn, sAb, 2 * L::kAbBytes);
    copy_chunk<NT>(sW, p.wimg2, L::kWBytes);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_pool = tmem_base + 2 * C;                       // acc[a]: columns [a*C, (a+1)*C); pooled: [2C, 3C)
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t sW_addr = tc::smem_u32(sW), sA_addr = tc::smem_u32(smem + L::kOffA);
    const uint32_t sAb_addr = tc::smem_u32(sAb), sWb_addr = tc::smem_u32(sWb);
    const uint32_t sidx_addr = tc::smem_u32(sidx), sctr_addr = tc::smem_u32(sctr), swn_addr = tc::smem_u32(swn);
    const uint32_t ab_row = sAb_addr + tc::unit_offset(row, 0, 2);
    constexpr uint32_t idesc = tc::make_idesc_bf16(kTile, C);
    uint32_t ph = 0, iter = 0;   // ph: bit a = phase of mbarrier a

    const int ku = (warp % kQuads) * 4 + (lane >> 3);
    const int r8 = lane & 7;
    const int rg0 = warp / kQuads;
    float2 nx[4], ny[4];
    auto load_offset_weights = [&]() {
        const uint32_t a = swn_addr + (uint32_t)(ku * 64);
        const float4 x0 = tc::lds_f32x4(a), x1 = tc::lds_f32x4(a + 16), y0 = tc::lds_f32x4(a + 32), y1 = tc::lds_f32x4(a + 48);
        nx[0] = make_float2(x0.x, x0.y); nx[1] = make_float2(x0.z, x0.w); nx[2] = make_float2(x1.x, x1.y); nx[3] = make_float2(x1.z, x1.w);
        ny[0] = make_float2(y0.x, y0.y); ny[1] = make_float2(y0.z, y0.w); ny[2] = make_float2(y1.x, y1.y); ny[3] = make_float2(y1.z, y1.w);
    };

    const TileWalk<float2> walk{p, cells, (int32_t)p.tiles_per_frame, row, K, sidx_addr, sctr, scell, swmax};
    auto wait_bar = [&](uint32_t a) {
        tc::mbar_wait(&bar[a], (ph >> a) & 1u);
        ph ^= 1u << a;
        tc::fence_after_sync();
    };

    int32_t cb = 0, cq = 0, db = 0, dq = 0;   // cursors: MLP tiles (cb, cq), copy units (db, dq)
    walk.start(cb, cq, db, dq, grp == 0);

    int32_t uframe[2] = {-1, -1}, ucell[2] = {-1, -1};   // the next two copy units (TileWalk::fetch_units)
    bool units_ready = false;

    while (cb < p.B || db < p.B) {
        if (cb < p.B) {
            const int par = iter & 1;
            ++iter;
            const int b = cb;
            walk.fetch_units(db, dq, uframe, ucell);   // list entries of the copy units that follow this tile: in flight during the whole tile
            units_ready = true;
            int32_t nb = cb, nq = cq;
            walk.advance(nb, nq, (int32_t)gridDim.x);
            walk.seek_live(nb, nq);
            const bool has_next = nb < p.B;
            int n_valid = 0;
            const int R = walk.read_header(par, grp == 0, lane, warp, n_valid);
            const int32_t cell = scell[par * kTile + row];
            const bool in_range = cell >= 0;
            int32_t ncell = -1;
            if (grp == 0 && has_next) ncell = walk.header_cell(nb, nq);

            const TT *Tc = reinterpret_cast<const TT *>(p.T) + (size_t)b * p.N * C + ku * 8, *neg = g_neg + ku * 8;
            const uint32_t idx0 = sidx_addr + (uint32_t)((par * K * kTile + rg0 * 8 + r8) * 4);
            const uint32_t ctr0 = sctr_addr + (uint32_t)((par * kTile + rg0 * 8 + r8) * 8);
            const uint32_t dst0 = sA_addr + tc::unit_offset(r8, ku, kc_units) + (uint32_t)(rg0 * kc_units * 128);
            const MT *src_bev = reinterpret_cast<const MT *>(p.bev) + map_cell<NHWC>(b, cell, C, cells);
            float tv[32];   // neighbour rows of the next round to build; in the last round: bev values of the final epilogue
            auto gather_round = [&](int k) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int32_t pr = (int32_t)tc::lds_u32(idx0 + (uint32_t)(k * kTile * 4 + i * kStep * 32));
                    tc::ldg_row8(pr >= 0 ? Tc + (size_t)pr * C : neg, tv + 8 * i);
                }
            };
            auto prefetch_tv = [&]() {
                if (in_range) prefetch_bev<C, G, 2, NHWC>(tv, src_bev, cells, grp);
            };
            // A[buf] = relu(T[idx_k] - e) for the rows gathered in tv; bias flag of round k -> Ab[buf]
            auto build_round = [&](int k, uint32_t buf) {
                load_offset_weights();
                const uint32_t dstb = dst0 + buf * L::kABytes;
                float2 ctr = tc::lds_f32x2(ctr0);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float2 ctr_next = ctr;
                    if (i < 3) ctr_next = tc::lds_f32x2(ctr0 + (i + 1) * kStep * 64);
                    const float2 cxx = make_float2(ctr.x, ctr.x), cyy = make_float2(ctr.y, ctr.y);
                    float2 v[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        v[e] = tc::ffma2(nx[e], cxx, tc::ffma2(ny[e], cyy, make_float2(tv[8 * i + 2 * e], tv[8 * i + 2 * e + 1])));
                    uint4 hi, lo;
                    tc::relu_split_bf16x8(v, hi, lo, NS == 2);
                    const uint32_t d = dstb + i * kStep * kc_units * 128;
                    tc::sts_u32x4(d, hi);
                    if (NS == 2) tc::sts_u32x4(d + kTile * C * 2, lo);
                    ctr = ctr_next;
                }
                if (grp == 0)
                    tc::sts_u32(ab_row + buf * L::kAbBytes,
                                (int32_t)tc::lds_u32(sidx_addr + (uint32_t)(((par * K + k) * kTile + row) * 4)) >= 0 ? 0x3F803F80u : 0u);
            };
            // acc[buf] = flag * b + A[buf] * W^T   (w_addr: the layer's packed image, wb: its bias operand)
            auto issue_round = [&](uint32_t buf, uint32_t acc, uint32_t w_addr, uint32_t wb_addr) {
                if (tid == 0) {
                    tc::fence_after_sync();
                    tc::mma_bf16(tmem_base + acc * C, tc::make_desc(sAb_addr + buf * L::kAbBytes, 128, 256),
                                 tc::make_desc(wb_addr, 128, 256), idesc, 0u);
                    issue_chunk<C, NS, C>(sA_addr + buf * L::kABytes, w_addr, tmem_base + acc * C, true);
                    tc::commit(&bar[acc]);
                }
            };
            auto stream_w3 = [&](uint32_t buf) {   // W3's packed image -> A[buf] (free: its last MMAs are complete)
                const uint32_t dst = sA_addr + buf * L::kABytes;
                for (int o = tid * 16; o < L::kWBytes; o += NT * 16) tc::cp_async16(dst + o, p.wimg3 + o);
                tc::cp_async_commit();
            };
            auto epilogue_round = [&](int k, uint32_t acc) {   // pooled (+)= relu(acc)
                __syncwarp();
#pragma unroll 1
                for (int cc = grp; cc < kChunksE; cc += G) {
                    float z[EW], s[EW];
                    if (k > 0) {
                        tc::tmem_ld16x2(tmem_base + acc * C + lane_off + cc * EW, tmem_pool + lane_off + cc * EW, z, s);
#pragma unroll
                        for (int i = 0; i < EW; i += 2) {
                            const float2 a = tc::fadd2(make_float2(s[i], s[i + 1]), make_float2(fmaxf(z[i], 0.f), fmaxf(z[i + 1], 0.f)));
                            s[i] = a.x;
                            s[i + 1] = a.y;
                        }
                    } else {
                        tc::tmem_ld<EW>(tmem_base + acc * C + lane_off + cc * EW, z);
#pragma unroll
                        for (int i = 0; i < EW; ++i) s[i] = fmaxf(z[i], 0.f);
                    }
                    tc::tmem_st<EW>(tmem_pool + lane_off + cc * EW, s);
                }
                tc::fence_before_sync();
            };

            if (R == 0) {
                if (grp == 0 && has_next) walk.header_fill(nb, ncell, par ^ 1);
                prefetch_tv();
            } else {
                // ---- prologue: round 0 -------------------------------------------------------------------------------------
                gather_round(0);
                build_round(0, 0);
                tc::fence_proxy_async();
                tc::fence_before_sync();
                __syncthreads();
                issue_round(0, 0, sW_addr, sWb_addr);
                if (grp == 0 && has_next) walk.header_fill(nb, ncell, par ^ 1);
                if (R > 1) {
                    gather_round(1);
                } else {
                    stream_w3(1);
                    prefetch_tv();
                }
                for (int k = 0; k < R; ++k) {
                    const uint32_t a = k & 1;
                    if (k + 1 < R) {   // build and issue round k+1 while the MMAs of round k run
                        build_round(k + 1, a ^ 1);
                        tc::fence_proxy_async();
                        tc::fence_before_sync();
                        __syncthreads();
                        issue_round(a ^ 1, a ^ 1, sW_addr, sWb_addr);
                        if (k + 2 < R) gather_round(k + 2); else prefetch_tv();
                    }
                    wait_bar(a);
                    if (k == R - 2) stream_w3(a);   // A[a] is free now; the last round uses A[a ^ 1]
                    epilogue_round(k, a);
                }
                // ---- layer 3: acc = n_valid * b3 + pooled * W3^T  (pooled -> A[l]; W3 sits in A[l ^ 1]) --------------------
                const uint32_t l = (R - 1) & 1;
                pooled_to_operand<NS, C, G>(tmem_pool + lane_off, sA_addr + l * L::kABytes, row, grp, true, ab_row + l * L::kAbBytes, n_valid);
                tc::cp_async_wait_all();   // this thread's part of W3 has landed
                tc::fence_proxy_async();
                tc::fence_before_sync();
                __syncthreads();
                issue_round(l, l, sA_addr + (l ^ 1) * L::kABytes, sWb_addr + L::kWbBytes);
                wait_bar(l);
            }
            // ---- final epilogue: out = bev + acc -----------------------------------------------------------------------------
            __syncwarp();
            if (R > 0 || p.out != p.bev) {
                const uint32_t acc_l = tmem_base + (uint32_t)(((R - 1) & 1) * C) + lane_off;
                MT *dst_out = reinterpret_cast<MT *>(p.out) + map_cell<NHWC>(b, cell, C, cells);
#pragma unroll
                for (int j = 0; j < (kChunksE + G - 1) / G; ++j) {
                    const int cc = grp + j * G;
                    if (cc < kChunksE) {
                        float z[EW];
                        if (R > 0) tc::tmem_ld<EW>(acc_l + cc * EW, z);
                        if constexpr (NHWC) {
                            if (in_range) {
                                float v[EW];
                                final_chunk_nhwc<2>(v, src_bev, cc, j, R, tv, z);
                                row_stcs16(dst_out + cc * EW, v);
                            }
                        } else if (in_range) {
                            if (j < 2) {
#pragma unroll
                                for (int i = 0; i < EW; ++i)
                                    map_stcs(dst_out + (size_t)(cc * EW + i) * cells, R > 0 ? tv[(j & 1) * EW + i] + z[i] : tv[(j & 1) * EW + i]);
                            } else {
#pragma unroll
                                for (int h = 0; h < EW; h += 8) {
                                    float bv[8];
#pragma unroll
                                    for (int i = 0; i < 8; ++i) bv[i] = map_ldcs(src_bev + (size_t)(cc * EW + h + i) * cells);
#pragma unroll
                                    for (int i = 0; i < 8; ++i)
                                        map_stcs(dst_out + (size_t)(cc * EW + h + i) * cells, R > 0 ? bv[i] + z[h + i] : bv[i]);
                                }
                            }
                        }
                    }
                }
            }
            tc::fence_before_sync();
            cb = nb;
            cq = nq;
        }
        if (!units_ready) walk.fetch_units(db, dq, uframe, ucell);
        units_ready = false;
        copy_units<C, G, MT, NHWC>(p, uframe, ucell, grp, cells);
    }

    teardown(tmem_base, L::kTmemCols, warp);
}

// ---------------------------------------------------------------------------------------------------------------
// K-4a on tensor cores:  T_s[b, m, :] = feat[b, m, :] W1_s[:, :Ci]^T + W1_s[:, Ci:Ci+3] p_m + b1_s      (m < num_points[b])
// for one or SEVERAL scales s in one pass (cf_point_mlp1 is the one-scale call).  The camera features of a 128-point
// tile are split and packed into the UMMA A operand ONCE, then multiplied by every scale's W1 image part: the output
// channels of all scales form one long N dimension that is walked in chunks of <= 128 columns.  Per chunk: the packed
// weight rows stream L2 -> shared memory into one of two buffers, one thread issues the K = Ci MMAs into one of two TMEM
// accumulators, and the epilogue of the previous chunk runs under them.  The rank-3 offset term and the bias are added
// on CUDA cores in that epilogue (Ci + 3 = 131 is not an MMA-friendly K).
// ---------------------------------------------------------------------------------------------------------------
#ifndef CF_L1_PREFETCH
#define CF_L1_PREFETCH 1
#endif
constexpr int kMaxScales = 8, kMaxChunks = 24;
// 8 worker warps + the MMA issuer warp.  With 16 worker warps the kernel alone is a little faster, but its CTA then holds 52 k of
// the SM's 64 k registers and the KNN search, which runs beside it on another stream, gets one block per SM; with 8 it gets
// three (measured: configs[2] step 3.99 -> 3.93 ms, configs[1] 0.903 -> 0.895 ms; a high-priority stream for this kernel
// instead made both slower).
#ifndef CF_MULTI_THREADS
#define CF_MULTI_THREADS 288
#endif
constexpr int kMultiThreads = CF_MULTI_THREADS;
constexpr int kStageGroup = kTile * 128;              // one staged block: 128 rows of 128 bytes (32 fp32 / 64 bf16 columns), SWIZZLE_128B
// Per split count: output columns per chunk (UMMA N) and whether full tiles are staged for TMA stores.  The staged path pays
// when the tables leave for DRAM (bf16 mode at configs[2]: 2.5 GB per step); with two splits the operands leave no room
// for the staging sets, and at configs[1] the tables stay in L2 where the direct stores were measured faster (114 vs 125 us).
// TH (CF_MODE_BF16_TABLES): the tables are written as bf16 -- half the bytes per column, so a 128-column chunk fits the
// same two staged blocks.
template <int NS, bool TH = false>
struct MultiShape {
    static_assert(!TH || NS == 1, "bf16 tables belong to the bf16 operand mode");
    static constexpr int kChunkW = NS == 2 || TH ? 128 : 64;
    static constexpr int kGroupCols = TH ? 64 : 32;   // columns of one staged block
    static constexpr int kWBufs = 2;       // weight ring: a chunk is requested kWBufs chunks before its MMAs
                                           // (4 buffers and 3 staging sets measured the same 0.99 ms at configs[2]: the kernel is
                                           // bound by the DRAM write rate, 2.5 GB of tables at ~2.5 TB/s + 0.5 GB of reads)
    static constexpr bool kStaged = NS == 1;
    static constexpr int kStageSet = (kChunkW / kGroupCols) * kStageGroup;   // the staged output of one chunk
    static constexpr int kStageSets = 2;   // a staged block has kStageSets - 1 chunk iterations to be read by the TMA engine
    static constexpr int kStageBytes = kStaged ? kStageSets * kStageSet : 0;
};
struct Mlp1MultiParams {
    const float *feat;
    const float *points;
    const int64_t *num_points;
    int32_t B, N, Ci, tiles_per_frame, n_scales, n_chunks;
    int32_t tma_out;   // 1: full tiles leave through the tensor maps (every T 16-byte aligned)
    const uint8_t *wimg[kMaxScales];
    const float *W1[kMaxScales];
    const float *b1[kMaxScales];
    float *T[kMaxScales];
    int32_t C[kMaxScales], foff[kMaxScales];   // channels; offset (floats) of the scale's b1|wx|wy|wz table in shared memory
    int32_t chunk_scale[kMaxChunks], chunk_n0[kMaxChunks], chunk_len[kMaxChunks];
};
struct Mlp1Maps {
    CUtensorMap m[kMaxScales];   // T_s as (C_s, N, B) fp32, box 32 x 128 x 1, SWIZZLE_128B
};

// K-4a for several scales, one 128-point tile at a time.  Per chunk of <= 64 output columns: the packed weight rows stream
// L2 -> shared memory (TMA, one chunk ahead) into one of two buffers, one elected lane issues the K = Ci MMAs into one of two
// TMEM accumulators, and the epilogue of the previous chunk runs under them.  The epilogue of a FULL tile adds the rank-3
// offset and the bias and stages its 128 x 64 block in shared memory (rows of 128 bytes, 128-byte swizzle: conflict-free
// STS.128), and one thread hands the block to the TMA engine (cp.async.bulk.tensor.3d store): the table leaves the SM as full
// lines without passing the LSU again.  (A thread owns one ROW of the accumulator, so direct global stores touch 32 lines per
// instruction; that made the kernel LSU-bound at a third of the HBM write rate.)  The last, partial tile of a frame stores
// directly so that rows past num_points stay untouched.
template <int NS, bool TH = false>
__global__ void __launch_bounds__(kMultiThreads, 1) k_point_mlp1_multi(const Mlp1MultiParams p, const __grid_constant__ Mlp1Maps maps)
{
    using MS = MultiShape<NS, TH>;
    // warps 0 .. NW-1: workers (operand build, epilogues; NT / 128 threads per row split the columns of a chunk);
    // warp NW: one elected lane streams the weight chunks (two cp.async.bulk per chunk: TMA engine, mbarrier complete_tx) and
    // issues the MMAs (descriptors in uniform registers), so the tcgen05.mma of a chunk never sit in front of an epilogue
    constexpr int NT = kMultiThreads - 32, NW = NT / 32, kIssuer = NT, kColGroups = NT / kTile;
    constexpr int kChunkW = MS::kChunkW, kStageSet = MS::kStageSet, kStageBytes = MS::kStageBytes, kGroupCols = MS::kGroupCols;
    constexpr uint32_t kWBufs = MS::kWBufs, kStageSets = MS::kStageSets;
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar[2], wbar[kWBufs];   // MMAs of a chunk complete; weights of a chunk have landed
    __shared__ uint32_t tmem_slot;
    const int Ci = p.Ci, kc_units = Ci / 8;
    const int a_bytes = NS * kTile * Ci * 2, w_bytes = NS * kChunkW * Ci * 2;
    uint8_t *sStage = smem;                               // two sets of kStageSet bytes (1024-byte aligned)
    uint8_t *sA = smem + kStageBytes;
    uint8_t *sWb = sA + a_bytes;                          // ring of kWBufs buffers of w_bytes
    float *sF = reinterpret_cast<float *>(sWb + kWBufs * w_bytes);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & (kTile - 1), half = tid / kTile;
    const bool worker = tid < NT;

    if (tid == 0) {
        tc::mbar_init(&bar[0], 1);
        tc::mbar_init(&bar[1], 1);
        for (uint32_t i = 0; i < kWBufs; ++i) tc::mbar_init(&wbar[i], 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(&tmem_slot, 2 * kChunkW);
    for (int s = 0; s < p.n_scales; ++s) {
        const int C = p.C[s];
        float *f = sF + p.foff[s];   // per PAIR of output channels (c, c + 1): b1 b1 | wx wx | wy wy | wz wz (packed fp32 math)
        for (int c = tid; c < C; c += NT + 32) {
            const float *w = p.W1[s] + (size_t)c * (Ci + 3) + Ci;
            float *fp = f + (c >> 1) * 8 + (c & 1);
            fp[0] = __ldg(p.b1[s] + c); fp[2] = __ldg(w); fp[4] = __ldg(w + 1); fp[6] = __ldg(w + 2);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = tmem_slot;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t sA_addr = tc::smem_u32(sA), sW_addr = tc::smem_u32(sWb), stage_addr = tc::smem_u32(sStage);
    const uint32_t sbo = kc_units * 128, lbo = 128;
    uint32_t ph0 = 0, ph1 = 0;
    uint32_t cn = 0;   // chunks issued so far: accumulator and MMA mbarrier of a chunk = cn & 1, weight buffer = cn % kWBufs
    uint32_t en = 0;   // staging set of the next staged epilogue (they rotate)
    int pend_j = -1, pend_b = 0;   // the staged chunk whose stores have not been handed to the TMA engine yet (uniform)
    int32_t pend_m0 = 0;
    uint32_t pend_set = 0;
    // the chunk's rows of a packed image: hi rows, then lo rows (each a contiguous run of len * Ci * 2 bytes): one bulk copy
    // each, both completing on the buffer's mbarrier.  Called by ONE thread (the elected lane of the issuer warp).
    const uint32_t wbar_addr = tc::smem_u32(wbar);
    auto prefetch_w = [&](uint32_t g) {   // g = running chunk number: chunk g % n_chunks of some tile, buffer g % kWBufs
        const int j = (int)(g % (uint32_t)p.n_chunks);
        const uint32_t buf = g % kWBufs;
        const int s = p.chunk_scale[j], n0 = p.chunk_n0[j];
        const uint32_t piece = (uint32_t)(p.chunk_len[j] * Ci * 2);
        const uint8_t *src = p.wimg[s] + (size_t)(n0 / 8) * kc_units * 128;
        const uint32_t dst = sW_addr + buf * w_bytes;
        tc::mbar_expect_tx(wbar_addr + buf * 8, NS * piece);
        tc::bulk_load_1d(dst, src, piece, wbar_addr + buf * 8);
        if (NS == 2) tc::bulk_load_1d(dst + kChunkW * Ci * 2, src + (size_t)p.C[s] * Ci * 2, piece, wbar_addr + buf * 8);
    };
    // Called by every thread right after a __syncthreads that follows the staging writes (and their fence.proxy.async):
    // thread 0 hands the staged block to the TMA engine.  Thread 0 also waits, BEFORE every such barrier, until the engine
    // has read all but its latest kStageSets - 2 blocks, so the set written next (used kStageSets epilogues ago) is free.
    auto flush_pending = [&]() {
        if (pend_j >= 0 && tid == 0) {
            const int s = p.chunk_scale[pend_j], n0 = p.chunk_n0[pend_j], len = p.chunk_len[pend_j];
            for (int g = 0; g * kGroupCols < len; ++g)   // (a 32-column scale fills half a bf16 block: the map clips at C)
                tc::tma_store_3d(&maps.m[s], n0 + g * kGroupCols, pend_m0, pend_b, stage_addr + pend_set * kStageSet + g * kStageGroup);
            tc::bulk_commit();
        }
        pend_j = -1;
    };
    const bool issuer_warp = warp == kIssuer / 32;
    if (issuer_warp) {
        if (tc::elect_one())
            for (uint32_t g = 0; g < kWBufs; ++g) prefetch_w(g);
        __syncwarp();
    }

    const int64_t tiles_total = (int64_t)p.tiles_per_frame * p.B;
    for (int64_t tile = blockIdx.x; tile < tiles_total; tile += gridDim.x) {
        const int b = (int)(tile / p.tiles_per_frame);
        const int32_t m0 = (int32_t)(tile - (int64_t)b * p.tiles_per_frame) * kTile;
        const int32_t n_pts = valid_points(p.num_points, b, p.N);
        if (m0 >= n_pts) continue;  // uniform across the CTA
        const bool full = MS::kStaged && p.tma_out && m0 + kTile <= n_pts;
#if CF_L1_PREFETCH
        // the feature rows of this CTA's next tile start their way from DRAM into L2 now, one tile ahead of their A-operand build
        if (tid == kIssuer) {
            const int64_t nt = tile + gridDim.x;
            if (nt < tiles_total) {
                const int nb = (int)(nt / p.tiles_per_frame);
                const int32_t nm0 = (int32_t)(nt - (int64_t)nb * p.tiles_per_frame) * kTile;
                const int32_t rows = min(kTile, valid_points(p.num_points, nb, p.N) - nm0);
                if (rows > 0) tc::bulk_prefetch_l2(p.feat + ((size_t)nb * p.N + nm0) * Ci, (uint32_t)(rows * Ci * 4));
            }
        }
#endif
        // ---- A tile, once for all scales.  An item is one 8-row group x 4 operand units (hence Ci % 32 == 0), lane (r8 = lane % 8, u = lane / 8):
        // coalesced 128-byte row segments in, and each quarter-warp writes 128 contiguous bytes of the operand image (conflict
        // free).  The feature rows stream from DRAM: the loads of a batch of items are all issued before the first one is
        // split and stored -----------------------------------------------------------------------------------------------
        const float *fb = p.feat + ((size_t)b * p.N + m0) * Ci;
        const int n_items = 16 * (kc_units / 4);
        constexpr int kBatch = 4;
        for (int item0 = warp; worker && item0 < n_items; item0 += NW * kBatch) {
            float t[kBatch][8];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int item = item0 + u * NW;
                const int rg = item / (kc_units / 4), uq = item - rg * (kc_units / 4);
                const int r = rg * 8 + (lane & 7), ku = uq * 4 + (lane >> 3);
#pragma unroll
                for (int i = 0; i < 8; ++i) t[u][i] = 0.0f;
                // one 256-bit load per lane: the 4 lanes of a row fetch one full 128-byte line per request
                if (item < n_items && m0 + r < n_pts) tc::ldg_nc_f32x8(fb + (size_t)r * Ci + ku * 8, t[u]);
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int item = item0 + u * NW;
                if (item < n_items) {
                    const int rg = item / (kc_units / 4), uq = item - rg * (kc_units / 4);
                    const int r = rg * 8 + (lane & 7), ku = uq * 4 + (lane >> 3);
                    uint4 hi, lo;
                    tc::split_bf16x8(t[u], hi, lo, NS == 2);
                    const uint32_t off = tc::unit_offset(r, ku, kc_units);
                    *reinterpret_cast<uint4 *>(sA + off) = hi;
                    if (NS == 2) *reinterpret_cast<uint4 *>(sA + kTile * Ci * 2 + off) = lo;
                }
            }
        }
        const int32_t m = m0 + row;
        const bool live = worker && m < n_pts;
        float px = 0.f, py = 0.f, pz = 0.f;
        if (live) {
            const float *q = p.points + ((size_t)b * p.N + m) * 3;
            px = __ldg(q); py = __ldg(q + 1); pz = __ldg(q + 2);
        }
        // epilogue of chunk j: T_s[m, n0 + c] = acc + W1[:, Ci:Ci+3] p + b1
        auto epilogue = [&](int j, uint32_t buf) {
            const int s = p.chunk_scale[j], n0 = p.chunk_n0[j], len = p.chunk_len[j], C = p.C[s];
            const float4 *f = reinterpret_cast<const float4 *>(sF + p.foff[s]);
            const uint32_t acc = tmem_base + buf * kChunkW + lane_off;
            float *trow = p.T[s] + (TH ? 0 : ((size_t)b * p.N + m) * C + n0);
            __nv_bfloat16 *trow_h = reinterpret_cast<__nv_bfloat16 *>(p.T[s]) + ((size_t)b * p.N + m) * C + n0;
            uint8_t *srow = sStage + en * kStageSet + row * 128;
#pragma unroll 1
            for (int c = half * 16; worker && c < len; c += 16 * kColGroups) {
                float z[16];
                tc::tmem_ld16(acc + c, z);
                if (full || live) {
#pragma unroll
                    for (int q8 = 0; q8 < 2; ++q8) {
                        float o[8];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {   // two columns per FMUL2 / FFMA2 / FADD2: z + ((wx px + wy py) + wz pz) + b1
                            const float4 fa = f[(n0 + c + q8 * 8) + 2 * i], fb = f[(n0 + c + q8 * 8) + 2 * i + 1];
                            float2 t = tc::fmul2(make_float2(fa.z, fa.w), make_float2(px, px));
                            t = tc::ffma2(make_float2(fb.x, fb.y), make_float2(py, py), t);
                            t = tc::ffma2(make_float2(fb.z, fb.w), make_float2(pz, pz), t);
                            t = tc::fadd2(tc::fadd2(make_float2(z[q8 * 8 + 2 * i], z[q8 * 8 + 2 * i + 1]), t), make_float2(fa.x, fa.y));
                            o[2 * i] = t.x;
                            o[2 * i + 1] = t.y;
                        }
                        if (TH) {   // 8 columns -> one 16-byte chunk of bf16 (round to nearest even)
                            const uint4 h = make_uint4(tc::pack_bf16x2(o[0], o[1]), tc::pack_bf16x2(o[2], o[3]), tc::pack_bf16x2(o[4], o[5]),
                                                       tc::pack_bf16x2(o[6], o[7]));
                            if (full) {
                                uint8_t *grp = srow + (c >> 6) * kStageGroup;
                                const int q = ((c & 63) >> 3) + q8;
                                *reinterpret_cast<uint4 *>(grp + ((q ^ (row & 7)) << 4)) = h;
                            } else {
                                *reinterpret_cast<uint4 *>(trow_h + c + q8 * 8) = h;
                            }
                        } else if (full) {   // 16-byte chunk q of the row's 128-byte line sits at q ^ (row & 7)
                            uint8_t *grp = srow + (c >> 5) * kStageGroup;
                            const int q = ((c & 31) >> 2) + q8 * 2;
                            *reinterpret_cast<float4 *>(grp + (((q) ^ (row & 7)) << 4)) = make_float4(o[0], o[1], o[2], o[3]);
                            *reinterpret_cast<float4 *>(grp + (((q + 1) ^ (row & 7)) << 4)) = make_float4(o[4], o[5], o[6], o[7]);
                        } else {
                            tc::stg_f32x8(trow + c + q8 * 8, o);   // 256-bit stores: every lane writes full 32-byte sectors of its row
                        }
                    }
                }
            }
            if (full) {
                pend_j = j; pend_b = b; pend_m0 = m0; pend_set = en;
                en = en + 1 == kStageSets ? 0 : en + 1;
            }
            tc::fence_before_sync();
        };
        // iteration j issues the MMAs of chunk j and runs the epilogue of chunk j - 1 (the last iteration only the epilogue)
        for (int j = 0; j <= p.n_chunks; ++j) {
            tc::fence_proxy_async();
            tc::fence_before_sync();
            if (tid == 0) tc::bulk_wait_read<kStageSets - 2>();   // all but the latest kStageSets - 2 blocks have been read
            __syncthreads();
            flush_pending();
            if (j < p.n_chunks) {
                if (issuer_warp && tc::elect_one()) {
                    tc::mbar_wait_a(wbar_addr + (cn % kWBufs) * 8, (cn / kWBufs) & 1u);   // the chunk's weights have landed (requested kWBufs chunks ago)
                    tc::fence_after_sync();
                    const uint32_t idesc = tc::make_idesc_bf16(kTile, p.chunk_len[j]);
                    const uint32_t w0 = sW_addr + (uint32_t)((cn % kWBufs) * w_bytes), acc = tmem_base + (uint32_t)((cn & 1) * kChunkW);
                    uint32_t accum = 0;
                    for (int kk = 0; kk < Ci / 16; ++kk) {
                        const uint32_t koff = kk * 2 * lbo;
                        const uint64_t a_hi = tc::make_desc(sA_addr + koff, lbo, sbo), w_hi = tc::make_desc(w0 + koff, lbo, sbo);
                        tc::mma_bf16(acc, a_hi, w_hi, idesc, accum);
                        accum = 1;
                        if (NS == 2) {
                            const uint64_t a_lo = tc::make_desc(sA_addr + kTile * Ci * 2 + koff, lbo, sbo);
                            const uint64_t w_lo = tc::make_desc(w0 + kChunkW * Ci * 2 + koff, lbo, sbo);
                            tc::mma_bf16(acc, a_hi, w_lo, idesc, 1);
                            tc::mma_bf16(acc, a_lo, w_hi, idesc, 1);
                        }
                    }
                    tc::commit(&bar[cn & 1]);
                }
                ++cn;
            }
            if (j > 0) {   // the previous chunk's MMAs: once they are complete their weight buffer is free again
                const uint32_t pb = (cn - (j < p.n_chunks ? 2u : 1u)) & 1u;
                if (pb) { tc::mbar_wait(&bar[1], ph1); ph1 ^= 1u; } else { tc::mbar_wait(&bar[0], ph0); ph0 ^= 1u; }
                tc::fence_after_sync();
                if (issuer_warp) {   // the weight buffer of the chunk just completed is free: request the chunk that uses it next
                    const uint32_t done = cn - (j < p.n_chunks ? 2u : 1u);
                    if (tc::elect_one()) prefetch_w(done + kWBufs);
                    __syncwarp();
                }
                epilogue(j - 1, pb);   // runs under this chunk's MMAs and the weight prefetch
            }
        }
    }
    if (tid == kIssuer)   // the chunks requested for tiles that never came
        for (uint32_t g = cn; g < cn + kWBufs; ++g) tc::mbar_wait_a(wbar_addr + (g % kWBufs) * 8, (g / kWBufs) & 1u);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    flush_pending();
    if (tid == 0) tc::bulk_wait0();   // the staged blocks have been written before the shared memory goes away
    if (warp == 0) tc::tmem_free(tmem_base, 2 * kChunkW);
}

// a standalone D[128 x N] = A[128 x Kd] * B[N x Kd]^T through exactly the same packing / descriptor / TMEM code,
// so operand-layout mistakes can be told apart from fusion-logic mistakes (cf_debug_umma_gemm).
template <int N, int NS>
__global__ void __launch_bounds__(kThreads) k_umma_selftest(const float *__restrict__ A, const float *__restrict__ Bm,
                                                            int32_t Kd, float *__restrict__ D)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int kc_units = Kd / 8;
    uint8_t *sA = smem;
    uint8_t *sB = smem + NS * kTile * Kd * 2;
    if (tid == 0) {
        tc::mbar_init(&bar, 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(&tmem_slot, N <= 32 ? 32 : N <= 64 ? 64 : N <= 128 ? 128 : 256);
    for (int ku = 0; ku < kc_units; ++ku) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = A[(size_t)tid * Kd + ku * 8 + i];
        uint4 hi, lo;
        tc::split_bf16x8(v, hi, lo, NS == 2);
        *reinterpret_cast<uint4 *>(sA + tc::unit_offset(tid, ku, kc_units)) = hi;
        if (NS == 2) *reinterpret_cast<uint4 *>(sA + kTile * Kd * 2 + tc::unit_offset(tid, ku, kc_units)) = lo;
    }
    for (int u = tid; u < N * kc_units; u += kThreads) {
        const int n = u / kc_units, ku = u - n * kc_units;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = Bm[(size_t)n * Kd + ku * 8 + i];
        uint4 hi, lo;
        tc::split_bf16x8(v, hi, lo, NS == 2);
        *reinterpret_cast<uint4 *>(sB + tc::unit_offset(n, ku, kc_units)) = hi;
        if (NS == 2) *reinterpret_cast<uint4 *>(sB + N * Kd * 2 + tc::unit_offset(n, ku, kc_units)) = lo;
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = tmem_slot;
    if (tid == 0) {
        const uint32_t idesc = tc::make_idesc_bf16(kTile, N);
        const uint32_t sbo = kc_units * 128, lbo = 128;
        const uint32_t a0 = tc::smem_u32(sA), b0 = tc::smem_u32(sB);
        uint32_t acc = 0;
        for (int kk = 0; kk < Kd / 16; ++kk) {
            const uint32_t koff = kk * 2 * lbo;
            const uint64_t a_hi = tc::make_desc(a0 + koff, lbo, sbo), b_hi = tc::make_desc(b0 + koff, lbo, sbo);
            tc::mma_bf16(tmem_base, a_hi, b_hi, idesc, acc);
            acc = 1;
            if (NS == 2) {
                const uint64_t a_lo = tc::make_desc(a0 + kTile * Kd * 2 + koff, lbo, sbo);
                const uint64_t b_lo = tc::make_desc(b0 + N * Kd * 2 + koff, lbo, sbo);
                tc::mma_bf16(tmem_base, a_hi, b_lo, idesc, 1);
                tc::mma_bf16(tmem_base, a_lo, b_hi, idesc, 1);
            }
        }
        tc::commit(&bar);
    }
    tc::mbar_wait(&bar, 0);
    tc::fence_after_sync();
    for (int cc = 0; cc < N / 32; ++cc) {
        float z[32];
        tc::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + cc * 32, z);
#pragma unroll
        for (int i = 0; i < 32; ++i) D[(size_t)tid * N + cc * 32 + i] = z[i];
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem_base, N <= 32 ? 32 : N <= 64 ? 64 : N <= 128 ? 128 : 256);
}

// CTAs per SM of a persistent fused kernel: every CTA of the grid should be resident at once (static tile -> CTA map), so
// the count is the minimum over shared memory, registers, threads and TMEM columns (512 per SM, never oversubscribed:
// a CTA that cannot allocate would spin inside tcgen05.alloc).
template <typename Kern>
int resident_ctas(Kern kern, int threads, int smem, int tmem_cols, int *regs_cache, int *out)
{
    if (!*regs_cache) {
        cudaFuncAttributes fa;
        CF_TRY(cuda_status(cudaFuncGetAttributes(&fa, kern), "fused kernel attributes"));
        *regs_cache = (fa.numRegs + 7) / 8 * 8;
    }
    const int by_smem = (228 * 1024) / (smem + 1024);
    const int by_regs = 65536 / (*regs_cache * threads);
    *out = std::max(0, std::min(std::min(std::min(by_smem, by_regs), 2048 / threads), std::min(512 / tmem_cols, 8)));
    return CF_OK;
}

template <bool SK, int C, int NS, bool TH, typename MT, bool NHWC>
int launch_kernel(const TcParams &p, cudaStream_t st)
{
    using L = std::conditional_t<SK, SkLayout<C, NS>, TcLayout<C, NS>>;
    void (*kern)(TcParams);
    if constexpr (SK) kern = k_fusion_sk<C, NS, TH, MT, NHWC>; else kern = k_fusion_tc<C, NS, TH, MT, NHWC>;
    const char *name = SK ? "k_fusion_sk" : "k_fusion_tc";
    constexpr int NT = kTile * TcShape<C>::G;
    const int smem = L::smem_bytes(p.K);
    static int attr_bytes = 0, regs = 0;
    if (smem > attr_bytes) {
        CF_TRY(cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "fused kernel smem attribute"));
        attr_bytes = smem;
    }
    int per_sm = 1;
    CF_TRY(resident_ctas(kern, NT, smem, L::kTmemCols, &regs, &per_sm));
    per_sm = std::max(1, per_sm);
    const int64_t grid = std::min<int64_t>(p.tiles_total, (int64_t)sm_count() * per_sm);
    if (tuning().debug_launch) fprintf(stderr, "%s<%d,%d>: %d CTAs/SM grid %lld smem %d\n", name, C, NS, per_sm, (long long)grid, smem);
    kern<<<(unsigned)grid, NT, smem, st>>>(p);
    return CF_OK;
}

// Kernel choice.  Measured on B200 (profiles/README.md): the double-buffered k_fusion_sk wins where the MMAs of a round are
// long (C = 128: 165 -> 148 us), is a wash at C = 64 and loses at C = 32, where the round is all operand build.  At C = 96
// and 128 it keeps the residency of k_fusion_tc (1 CTA per SM: registers, and its 3C TMEM columns), so it runs wherever its
// shared memory fits: always, except at C = 128 in fp32 mode (NS = 2) from K = 15 on.
template <int C, int NS, bool TH, typename MT, bool NHWC>
int launch_fused(const TcParams &p, cudaStream_t st)
{
    if constexpr (C == 96 || (C == 128 && NS == 1)) {
        static_assert(SkLayout<C, NS>::smem_bytes(CF_MAX_K) <= 227 * 1024, "k_fusion_sk fits every K at this width");
        return launch_kernel<true, C, NS, TH, MT, NHWC>(p, st);
    } else if constexpr (C == 128) {
        if (SkLayout<C, NS>::smem_bytes(p.K) <= 227 * 1024) return launch_kernel<true, C, NS, TH, MT, NHWC>(p, st);
        return launch_kernel<false, C, NS, TH, MT, NHWC>(p, st);
    } else {
        return launch_kernel<false, C, NS, TH, MT, NHWC>(p, st);
    }
}

// the fused launch of one width for the mode (NS, bf16 tables th) and the map type (io16: bf16 maps) and layout
template <int C, bool NHWC>
int launch_fused_layout(const TcParams &p, int NS, bool th, bool io16, cudaStream_t st)
{
    if (io16)
        return NS == 2 ? launch_fused<C, 2, false, __nv_bfloat16, NHWC>(p, st)
               : th    ? launch_fused<C, 1, true, __nv_bfloat16, NHWC>(p, st)
                       : launch_fused<C, 1, false, __nv_bfloat16, NHWC>(p, st);
    return NS == 2 ? launch_fused<C, 2, false, float, NHWC>(p, st)
           : th    ? launch_fused<C, 1, true, float, NHWC>(p, st)
                   : launch_fused<C, 1, false, float, NHWC>(p, st);
}
template <int C>
int launch_fused_width(const TcParams &p, int NS, bool th, bool io16, bool nhwc, cudaStream_t st)
{
    return nhwc ? launch_fused_layout<C, true>(p, NS, th, io16, st) : launch_fused_layout<C, false>(p, NS, th, io16, st);
}

}  // namespace

static size_t tc_weight_bytes(int32_t C, int NS) { return ((size_t)2 * NS * C * C * 2 + 255) / 256 * 256; }

size_t fusion_tc_packed_bytes(int32_t C, int32_t mode) { return tc_weight_bytes(C, mode_base(mode) == CF_MODE_FP32 ? 2 : 1); }

int fusion_tc_pack(const float *d_W2, const float *d_W3, int32_t C, int32_t mode, void *d_packed, cudaStream_t st)
{
    CF_REQUIRE(C % 32 == 0 && C >= 32 && C <= 256, CF_ERR_UNSUPPORTED, "cf_fusion_pack_weights: C=%d", C);
    const int NS = mode_base(mode) == CF_MODE_FP32 ? 2 : 1;
    const int KC = kc_for(C, NS);
    const int pack_blocks = (C * (C / 8) + 255) / 256;
    k_pack_weights<<<pack_blocks, 256, 0, st>>>(d_W2, C, C, C, KC, NS, (uint8_t *)d_packed);
    k_pack_weights<<<pack_blocks, 256, 0, st>>>(d_W3, C, C, C, KC, NS, (uint8_t *)d_packed + (size_t)NS * C * C * 2);
    count_launches(2);
    return launch_status("cf_fusion_pack_weights");
}

size_t fusion_tc_workspace_bytes(int32_t C, int32_t mode, int32_t B, int32_t H, int32_t W)
{
    const int NS = mode_base(mode) == CF_MODE_FP32 ? 2 : 1;
    // packed W2/W3 images | per-frame counts (with / without a neighbour) | per-frame cell lists
    return tc_weight_bytes(C, NS) + 512 + (size_t)B * H * W * sizeof(int32_t);
}

int fusion_tc(const float *d_bev, const float *d_T, const int32_t *d_knn, int32_t B, int32_t N, int32_t C, int32_t H,
              int32_t W, int32_t K, float x0, float y0, float dx, float dy, const float *d_W1, int32_t Ci,
              const float *d_W2, const float *d_b2, const float *d_W3, const float *d_b3, float *d_out, int32_t mode,
              const void *d_packed, void *d_workspace, cudaStream_t st)
{
    CF_REQUIRE(C % 32 == 0, CF_ERR_UNSUPPORTED, "cf_fusion_fwd: tensor-core path needs C %% 32 == 0 (C=%d)", C);
    const bool io16 = (mode & CF_IO_BF16) != 0;   // d_bev / d_out hold bf16 maps
    const bool nhwc = (mode & CF_IO_NHWC) != 0;   // d_bev / d_out are (B,H,W,C) maps
    CF_REQUIRE(!nhwc || (aligned16(d_bev) && aligned16(d_out)), CF_ERR_ALIGN, "cf_fusion_fwd: NHWC maps must be 16-byte aligned");
    mode = mode_base(mode);
    const int NS = mode == CF_MODE_FP32 ? 2 : 1;
    // packed W2 | W3 operand images: the caller's cached copy (cf_fusion_pack_weights) or packed here
    const uint8_t *img2 = d_packed ? (const uint8_t *)d_packed : (const uint8_t *)d_workspace;
    const uint8_t *img3 = img2 + (size_t)NS * C * C * 2;
    int32_t *cell_count = (int32_t *)((uint8_t *)d_workspace + tc_weight_bytes(C, NS));
    int32_t *cell_list = cell_count + 128;
    CF_REQUIRE(B <= 64, CF_ERR_ARG, "cf_fusion_fwd: batch %d > 64 frames per call", B);
    const int64_t n_cells = (int64_t)H * W;
    // Compaction pays when there are many more tiles than SMs.  On the small coarse scales the cells with a neighbour are
    // one contiguous blob, so the tiles are already either full or empty (empty tiles just copy bev -> out) and
    // compaction only adds a launch (measured: 123 -> 148 us at 88x100x192).
    const int64_t min_tiles = 4 * (int64_t)sm_count();
    if (!d_packed) CF_TRY(fusion_tc_pack(d_W2, d_W3, C, mode, d_workspace, st));
    const bool compact = ceil_div64(n_cells, kTile) * B >= min_tiles;
    if (compact) {
        CF_TRY(cuda_status(cudaMemsetAsync(cell_count, 0, 512, st), "cf_fusion_fwd memset"));
        k_cell_compact<<<dim3((unsigned)ceil_div64(n_cells, 256), (unsigned)B), 256, 0, st>>>(d_knn, K, n_cells, cell_list,
                                                                                            cell_count);
        count_launches(1);
    }
    TcParams p;
    p.bev = d_bev; p.T = d_T; p.knn = d_knn; p.out = d_out; p.wimg2 = img2; p.wimg3 = img3; p.W1 = d_W1;
    p.b2 = d_b2; p.b3 = d_b3; p.B = B; p.N = N; p.H = H; p.W = W; p.K = K; p.Ci = Ci;
    p.x0 = x0; p.y0 = y0; p.dx = dx; p.dy = dy;
    p.tiles_per_frame = ceil_div64((int64_t)H * W, kTile);
    p.tiles_total = p.tiles_per_frame * B;
    p.cell_list = compact ? cell_list : nullptr;
    p.cell_count = cell_count;
    p.copy_dead = compact && d_out != d_bev;
    int rc = CF_ERR_UNSUPPORTED;
    const bool th = mode == CF_MODE_BF16_TABLES;   // d_T holds bf16 rows
    switch (C) {
        case 32: rc = launch_fused_width<32>(p, NS, th, io16, nhwc, st); break;
        case 64: rc = launch_fused_width<64>(p, NS, th, io16, nhwc, st); break;
        case 96: rc = launch_fused_width<96>(p, NS, th, io16, nhwc, st); break;
        case 128: rc = launch_fused_width<128>(p, NS, th, io16, nhwc, st); break;
        case 192: rc = launch_fused_width<192>(p, NS, th, io16, nhwc, st); break;
        case 256: rc = launch_fused_width<256>(p, NS, th, io16, nhwc, st); break;
        default:
            set_error("cf_fusion_fwd: unsupported C=%d on the tensor-core path", C);
            return CF_ERR_UNSUPPORTED;
    }
    CF_TRY(rc);
    count_launches(1);
    return launch_status("cf_fusion_fwd (tcgen05)");
}


int point_mlp1_tc_pack(const float *d_W1, int32_t Ci, int32_t C, int32_t mode, void *d_packed, cudaStream_t st)
{
    CF_REQUIRE(Ci % 16 == 0 && Ci <= 256 && C % 32 == 0, CF_ERR_UNSUPPORTED, "cf_point_mlp1_pack_weights: Ci=%d C=%d", Ci, C);
    const int NS = mode == CF_MODE_FP32 ? 2 : 1;
    k_pack_weights<<<(C * (Ci / 8) + 255) / 256, 256, 0, st>>>(d_W1, C, Ci, Ci + 3, Ci, NS, (uint8_t *)d_packed);
    count_launches(1);
    return launch_status("cf_point_mlp1_pack_weights");
}

size_t point_mlp1_tc_workspace_bytes(int32_t Ci, int32_t C, int32_t mode)
{
    const int NS = mode == CF_MODE_FP32 ? 2 : 1;
    return (size_t)NS * C * Ci * 2 + 256;
}

// 3-D tensor map over a table T (B, N, C) fp32 (or bf16): x = channel (fastest), y = point, z = frame; box 32 (64) x 128 x 1 with the
// 128-byte swizzle (the layout the epilogue stages).  Rows past N are clipped by the TMA engine.
static int make_table_map(CUtensorMap *tm, float *base, int32_t C, int32_t N, int32_t B, bool th)
{
    typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        CF_TRY(cuda_status(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q), "cuTensorMapEncodeTiled entry point"));
        CF_REQUIRE(f != nullptr && q == cudaDriverEntryPointSuccess, CF_ERR_LAUNCH, "cuTensorMapEncodeTiled is not available in this driver");
        fn = (EncodeTiledFn)f;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)N, (cuuint64_t)B};
    const cuuint64_t el_bytes = th ? 2 : 4;
    const cuuint64_t strides[2] = {(cuuint64_t)C * el_bytes, (cuuint64_t)N * C * el_bytes};
    const cuuint32_t box[3] = {th ? 64u : 32u, (cuuint32_t)kTile, 1};   // rows of 128 bytes
    const cuuint32_t el[3] = {1, 1, 1};
    const CUresult r = fn(tm, th ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, el,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_LAUNCH, "cuTensorMapEncodeTiled failed for a (%d, %d, %d) table (%d)", B, N, C, (int)r);
    return CF_OK;
}

// the chunk table (p.C, p.foff, p.chunk_*, p.n_chunks) and the shared memory of a k_point_mlp1_multi launch; returns
// CF_ERR_UNSUPPORTED (without setting an error) when the shapes do not fit the kernel
static int plan_mlp1_multi(Mlp1MultiParams &p, size_t &smem, int32_t Ci, int32_t n_scales, const int32_t *h_C, int32_t mode)
{
    const int NS = mode == CF_MODE_FP32 ? 2 : 1;
    if (n_scales < 1 || n_scales > kMaxScales || Ci % 32 != 0 || Ci > 256) return CF_ERR_UNSUPPORTED;
    const bool th = mode == CF_MODE_BF16_TABLES;
    const int chunk_w = NS == 2 ? MultiShape<2>::kChunkW : th ? MultiShape<1, true>::kChunkW : MultiShape<1>::kChunkW;
    const int stage_bytes = NS == 2 ? MultiShape<2>::kStageBytes : th ? MultiShape<1, true>::kStageBytes : MultiShape<1>::kStageBytes;
    int chunks = 0, foff = 0;
    for (int s = 0; s < n_scales; ++s) {
        const int C = h_C[s];
        if (C % 32 != 0 || C < 32 || C > 1024) return CF_ERR_UNSUPPORTED;
        p.C[s] = C; p.foff[s] = foff;
        foff += 4 * C;
        for (int n0 = 0; n0 < C; n0 += chunk_w) {
            if (chunks == kMaxChunks) return CF_ERR_UNSUPPORTED;
            p.chunk_scale[chunks] = s; p.chunk_n0[chunks] = n0; p.chunk_len[chunks] = std::min(chunk_w, C - n0);
            ++chunks;
        }
    }
    p.n_chunks = chunks;
    const int w_bufs = NS == 2 ? MultiShape<2>::kWBufs : MultiShape<1>::kWBufs;
    smem = (size_t)stage_bytes + (size_t)NS * (kTile + w_bufs * chunk_w) * Ci * 2 + (size_t)foff * 4;
    return smem > 225 * 1024 ? CF_ERR_UNSUPPORTED : CF_OK;
}

bool point_mlp1_multi_fits(int32_t Ci, int32_t C, int32_t mode)
{
    Mlp1MultiParams p;
    size_t smem;
    return plan_mlp1_multi(p, smem, Ci, 1, &C, mode) == CF_OK;
}

// returns CF_ERR_UNSUPPORTED (without setting an error) when the shapes do not fit the multi-scale kernel
int point_mlp1_multi_tc(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N,
                        int32_t Ci, int32_t n_scales, const int32_t *h_C, const float *const *h_W1,
                        const float *const *h_b1, float *const *h_T, int32_t mode, const void *const *h_packed,
                        cudaStream_t st)
{
    const int NS = mode == CF_MODE_FP32 ? 2 : 1;
    const bool th = mode == CF_MODE_BF16_TABLES;
    Mlp1MultiParams p;
    size_t smem;
    if (plan_mlp1_multi(p, smem, Ci, n_scales, h_C, mode) != CF_OK) return CF_ERR_UNSUPPORTED;
    p.feat = d_feat; p.points = d_points; p.num_points = d_num_points;
    p.B = B; p.N = N; p.Ci = Ci; p.tiles_per_frame = (N + kTile - 1) / kTile; p.n_scales = n_scales;
    for (int s = 0; s < n_scales; ++s) {
        if (!h_packed[s]) return CF_ERR_UNSUPPORTED;
        p.wimg[s] = (const uint8_t *)h_packed[s]; p.W1[s] = h_W1[s]; p.b1[s] = h_b1[s]; p.T[s] = h_T[s];
    }
    Mlp1Maps maps;
    memset(&maps, 0, sizeof(maps));
    p.tma_out = (NS == 2 ? MultiShape<2>::kStaged : MultiShape<1>::kStaged) && !tuning().no_tma_store;
    for (int s = 0; s < n_scales; ++s)
        if (((uintptr_t)h_T[s] & 15u) != 0) p.tma_out = 0;
    for (int s = 0; s < n_scales && p.tma_out; ++s)
        if (make_table_map(&maps.m[s], h_T[s], h_C[s], N, B, th) != CF_OK) p.tma_out = 0;   // no tensor maps (old driver): direct stores
    if (tuning().debug_launch) fprintf(stderr, "k_point_mlp1_multi<%d,%d>: %d chunks, staged TMA stores %d\n", NS, (int)th, p.n_chunks, p.tma_out);
    auto kern = NS == 2 ? k_point_mlp1_multi<2> : th ? k_point_mlp1_multi<1, true> : k_point_mlp1_multi<1>;
    CF_TRY(cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                       "k_point_mlp1_multi smem attribute"));
    const int64_t tiles = (int64_t)p.tiles_per_frame * B;
    // one CTA per SM (shared memory); an even share of tiles per CTA beats leaving a few CTAs with one tile more
    const int64_t waves = ceil_div64(tiles, sm_count());
    const int64_t grid = std::max<int64_t>(1, ceil_div64(tiles, waves));
    kern<<<(unsigned)grid, kMultiThreads, smem, st>>>(p, maps);
    count_launches(1);
    return launch_status("cf_point_mlp1_multi (tcgen05)");
}

int umma_selftest(const float *d_A, const float *d_B, int32_t N, int32_t Kd, int32_t split, float *d_D, cudaStream_t st)
{
    CF_REQUIRE(Kd % 16 == 0 && Kd >= 16 && Kd <= 256, CF_ERR_ARG, "cf_debug_umma_gemm: K=%d", Kd);
    const int NS = split ? 2 : 1;
    const size_t smem = (size_t)NS * (kTile + N) * Kd * 2;
    CF_REQUIRE(smem <= 200 * 1024, CF_ERR_ARG, "cf_debug_umma_gemm: operands do not fit in shared memory");
#define CF_ST_CASE(n)                                                                                                  \
    case n:                                                                                                            \
        if (NS == 2) {                                                                                                 \
            CF_TRY(cuda_status(cudaFuncSetAttribute(k_umma_selftest<n, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                    200 * 1024), "selftest attr"));                                   \
            k_umma_selftest<n, 2><<<1, kThreads, smem, st>>>(d_A, d_B, Kd, d_D);                                       \
        } else {                                                                                                       \
            CF_TRY(cuda_status(cudaFuncSetAttribute(k_umma_selftest<n, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                    200 * 1024), "selftest attr"));                                   \
            k_umma_selftest<n, 1><<<1, kThreads, smem, st>>>(d_A, d_B, Kd, d_D);                                       \
        }                                                                                                              \
        break;
    switch (N) {
        CF_ST_CASE(32) CF_ST_CASE(64) CF_ST_CASE(128) CF_ST_CASE(192) CF_ST_CASE(256)
        default:
            set_error("cf_debug_umma_gemm: N=%d not instantiated", N);
            return CF_ERR_ARG;
    }
#undef CF_ST_CASE
    count_launches(1);
    return launch_status("cf_debug_umma_gemm");
}

}  // namespace cf

// D (128,N) fp32 = A (128,K) * B (N,K)^T through the library's tcgen05 building blocks; split != 0 uses the
// bf16 hi/lo three-product scheme of CF_MODE_FP32.  Self-test entry point (tests/test_gpu_umma.py).
extern "C" int cf_debug_umma_gemm(const float *d_A, const float *d_B, int32_t N, int32_t K, int32_t split,
                                         float *d_D, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_A && d_B && d_D, CF_ERR_ARG, "cf_debug_umma_gemm: null pointer");
    return umma_selftest(d_A, d_B, N, K, split, d_D, (cudaStream_t)stream);
}
