// cf_bwd.cu -- K-4b: backward of the continuous-fusion layer (needed by the training configuration only).
//
// Forward (per scale, see cf_mlp_simt.cu / cf_mlp_tc.cu):
//   T_p   = W1[:, :Ci] f_p + W1[:, Ci:] p + b1                      per point
//   h1_r  = relu(T[j_r] - w1x*cx - w1y*cy)                          per row r = (cell, k) with a neighbour j_r
//   h2_r  = relu(W2 h1_r + b2);  pooled_c = sum_k h2_(c,k);  out_c = bev_c + W3 pooled_c + n_valid(c) b3
// Backward, given g = dL/dout (NCHW):   d bev = g   (returned by the host layer as the same tensor), and
//   G (cells x C)   = g transposed to cell-major
//   dW3 += G^T pooled        db3 += sum_c n_valid(c) G_c        dPooled = G W3
//   dZ2_r = dPooled_cell(r) * [h2_r > 0]      dW2 += dZ2^T H1      db2 += sum_r dZ2_r
//   dA_r  = (dZ2_r W2) * [h1_r > 0]           dT[j_r] += dA_r  (scatter-add, atomics)
//   dW1[:, Ci + j] += sum_r dA_r off_j(r),  off = (px - cx, py - cy, pz) of row r
//   dW1[:, :Ci] += dT^T F     db1 += sum_p dT_p     dF += dT W1[:, :Ci]
// Nothing is saved by the forward except indices, inputs and weights: H1, H2 and pooled are recomputed here and
// materialised in the caller-provided workspace.  Only (cell, k) slots that HOLD a neighbour exist there: k_bwd_compact
// turns knn_idx into a list of live cells and a list of live rows (the rows of a cell are contiguous), their two counts
// stay in device memory, and every later kernel is launched for the dense upper bound and clamps itself to the count
// (no host synchronisation; blocks beyond the count exit at once).  All arithmetic is fp32 on CUDA cores; reductions
// over rows use split accumulation + atomics, so gradients are reproducible to rounding, not bit for bit.
// With CF_BWD_DETERMINISTIC in `mode` the same kernels run with ordered list positions, per-split partials instead of
// atomics (summed in split order by cf_bwd_det.cu) and a gather for dT: gradients are then bit-identical run to run.
#include "cf_common.cuh"

namespace cf {

// cf_bwd_tc.cu: the same GEMMs on the tcgen05 tensor cores (fp32 operands split into bf16 hi + lo, fp32 accumulate)
enum { EPI_STORE = 0, EPI_ACCUM = 1, EPI_BIAS_RELU = 2, EPI_MASK = 3 };
size_t bwd_tc_packed_bytes(int32_t Nn, int32_t Kd);
bool bwd_tc_nn_fits(int32_t Kd, int32_t N);
bool bwd_tc_tn_fits(int32_t M, int32_t N);
int bwd_tc_pack(const float *d_W, int32_t ld, int32_t Nn, int32_t Kd, int transpose, void *d_img, cudaStream_t st);
int bwd_tc_pack4(const float *const *Ws, const int32_t *lds, const int32_t *Nns, const int32_t *Kds, const int *transposes,
                 void *const *imgs, int n, cudaStream_t st);
int bwd_tc_gemm_nn(const float *X, int64_t ldx, int64_t R, const int32_t *d_R, int32_t Kd, int32_t N, const void *wimg,
                   float *Out, int64_t ldo, int epi, const float *aux, int64_t ldaux, cudaStream_t st);
int bwd_tc_gemm_tn(const float *X, int64_t ldx, int32_t M, const float *Y, int64_t ldy, int32_t N, const float *Y2,
                   int64_t rs2, int64_t cs2, int32_t n2, const float *wcol, int64_t R, const int32_t *d_R, float *dW,
                   int64_t ldw, float *db, cudaStream_t st, float *part = nullptr);
// cf_bwd_det.cu: the pieces of the deterministic mode
size_t det_cell_blocks(int64_t ncell);
int det_compact_bases(const int32_t *knn, int64_t ncell, int32_t K, int32_t *blk, int32_t *counters, cudaStream_t st);
int det_reduce(const float *part, int32_t M, int32_t n_w, int32_t n_out, int32_t nsplit, int64_t R, const int32_t *d_R,
               int64_t unit, int64_t per_fixed, float *dW, int64_t ldw, int64_t cs, float *db, cudaStream_t st);
size_t det_dT_words(int64_t pts, int64_t rows);
int det_dT(const float *dA, int32_t C, const int32_t *row_pt, const int32_t *n_rows, int64_t rows, int64_t pts, float *dT,
           void *ws, cudaStream_t st);

namespace {

// ---------------------------------------------------------------------------------------------------------------
// C[R x N] (beta ? += : =) A[R x Kd] * B[Kd x N]; optional mask: C := 0 where mask[r,n] <= 0.   64x64x16 tiles.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sgemm_nn(const float *__restrict__ A, int64_t lda, const float *__restrict__ Bm,
                                                  int64_t ldb, float *__restrict__ Cm, int64_t ldc, int64_t R, int32_t N,
                                                  int32_t Kd, int beta, const float *__restrict__ mask, int64_t ldm,
                                                  const int32_t *__restrict__ d_R)
{
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t r0 = (int64_t)blockIdx.x * 64;
    const int32_t n0 = blockIdx.y * 64;
    if (d_R) R = min(R, (int64_t)__ldg(d_R));
    if (r0 >= R) return;
    float acc[4][4] = {};
    for (int32_t k0 = 0; k0 < Kd; k0 += 16) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int idx = tid + t * 256;
            {   // A tile: 64 rows x 16 k
                const int rr = idx >> 4, kk = idx & 15;
                const int64_t r = r0 + rr;
                As[kk][rr] = (r < R && k0 + kk < Kd) ? __ldg(A + r * lda + k0 + kk) : 0.0f;
            }
            {   // B tile: 16 k x 64 n
                const int kk = idx >> 6, nn = idx & 63;
                Bs[kk][nn] = (k0 + kk < Kd && n0 + nn < N) ? __ldg(Bm + (int64_t)(k0 + kk) * ldb + n0 + nn) : 0.0f;
            }
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
        const int64_t r = r0 + ty * 4 + i;
        if (r >= R) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int32_t n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (mask && !(__ldg(mask + r * ldm + n) > 0.0f)) v = 0.0f;
            float *dst = Cm + r * ldc + n;
            *dst = beta ? *dst + v : v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// C[M x N] += scale * A[R x M]^T * B[R x N]   (reduction over the long dimension R, split across blockIdx.z, atomics;
// part != nullptr: each split stores its tile to part[z][M][N] instead, for a fixed-order sum)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sgemm_tn(const float *__restrict__ A, int64_t lda, const float *__restrict__ Bm,
                                                  int64_t ldb, float *__restrict__ Cm, int64_t ldc, int64_t R, int32_t M,
                                                  int32_t N, int64_t rows_per_split, const int32_t *__restrict__ d_R,
                                                  float *__restrict__ part)
{
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int32_t m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
    if (d_R) R = min(R, (int64_t)__ldg(d_R));
    const int64_t r_begin = (int64_t)blockIdx.z * rows_per_split, r_end = min(R, r_begin + rows_per_split);
    if (r_begin >= R) return;
    float acc[4][4] = {};
    for (int64_t r0 = r_begin; r0 < r_end; r0 += 16) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int idx = tid + t * 256;
            const int rr = idx >> 6, cc = idx & 63;
            const int64_t r = r0 + rr;
            As[rr][cc] = (r < r_end && m0 + cc < M) ? __ldg(A + r * lda + m0 + cc) : 0.0f;
            Bs[rr][cc] = (r < r_end && n0 + cc < N) ? __ldg(Bm + r * ldb + n0 + cc) : 0.0f;
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
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int32_t m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
            if (m >= M || n >= N) continue;
            if (part) part[((int64_t)blockIdx.z * M + m) * N + n] = acc[i][j];
            else if (acc[i][j] != 0.0f) atomicAdd(Cm + (int64_t)m * ldc + n, acc[i][j]);
        }
}

// out[n] += scale * sum_r w[r] * X[r, n]   (w == nullptr: plain column sum).
// grid (row slabs of `slab` rows, column chunks of 32); a warp owns every 8th row of the slab, lane = column: 128-byte row
// segments, 4 independent partial sums per lane, then an 8-warp reduction in shared memory and one atomicAdd per column
// (slab_out != nullptr: the slab's sums are stored to slab_out[slab][N] instead, for a fixed-order sum).
__global__ void __launch_bounds__(256) k_colsum(const float *__restrict__ X, int64_t ldx, int64_t R, int32_t N,
                                                const float *__restrict__ w, float scale, float *__restrict__ out,
                                                int64_t out_stride, const int32_t *__restrict__ d_R, int64_t slab,
                                                float *__restrict__ slab_out)
{
    __shared__ float part[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int32_t n = blockIdx.y * 32 + lane;
    if (d_R) R = min(R, (int64_t)__ldg(d_R));
    const int64_t r_begin = (int64_t)blockIdx.x * slab, r_end = min(R, r_begin + slab);
    if (r_begin >= R) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (n < N) {
        int64_t r = r_begin + warp;
        for (; r + 24 < r_end; r += 32) {
            const float x0 = __ldg(X + r * ldx + n), x1 = __ldg(X + (r + 8) * ldx + n);
            const float x2 = __ldg(X + (r + 16) * ldx + n), x3 = __ldg(X + (r + 24) * ldx + n);
            s0 = fmaf(w ? __ldg(w + r) : 1.0f, x0, s0);
            s1 = fmaf(w ? __ldg(w + r + 8) : 1.0f, x1, s1);
            s2 = fmaf(w ? __ldg(w + r + 16) : 1.0f, x2, s2);
            s3 = fmaf(w ? __ldg(w + r + 24) : 1.0f, x3, s3);
        }
        for (; r < r_end; r += 8) s0 = fmaf(w ? __ldg(w + r) : 1.0f, __ldg(X + r * ldx + n), s0);
    }
    part[warp][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (warp == 0 && n < N) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += part[i][lane];
        if (slab_out) slab_out[(int64_t)blockIdx.x * N + n] = s * scale;
        else if (s != 0.0f) atomicAdd(out + (int64_t)n * out_stride, s * scale);
    }
}

// Live-cell / live-row lists.  Thread = cell (all frames in one index space).  A cell with n > 0 neighbours takes the next
// free cell slot ci and n consecutive row slots (block-wide ballot / shuffle scan, one atomicAdd per block and counter).
//   cell_list[ci] = b * cells + cell     cell_row0[ci] = first row     cell_nv[ci] = n  (float: it multiplies b3's gradient)
//   row_pt[r] = b * N + point            row_cell[r] = ci              row_cx / row_cy[r] = the cell's centre
//   row_off[j * row_cap + r], j = 0..2 = (px - cx, py - cy, pz): the three offset inputs of layer 1 for that row
// counters[0] = live cells, counters[1] = live rows (zeroed by the caller of the kernel).
// block_base != nullptr: the block's first cell / row slot is block_base[2 * block + 0 / 1] (an exclusive scan of the
// block totals, counters already hold the totals): the lists are then in grid order.
__global__ void __launch_bounds__(256) k_bwd_compact(const int32_t *__restrict__ knn, int64_t ncell, int64_t cells, int32_t W,
                                                     int32_t K, int32_t N, float x0, float y0, float dx, float dy,
                                                     int32_t *__restrict__ counters, int32_t *__restrict__ cell_list,
                                                     int32_t *__restrict__ cell_row0, float *__restrict__ cell_nv,
                                                     int32_t *__restrict__ row_pt, int32_t *__restrict__ row_cell,
                                                     float *__restrict__ row_cx, float *__restrict__ row_cy,
                                                     const float *__restrict__ points, float *__restrict__ row_off,
                                                     int64_t row_cap, const int32_t *__restrict__ block_base)
{
    __shared__ int32_t warp_cells[8], warp_rows[8], base[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x;
    int32_t nv = 0;
    if (g < ncell)
        for (int k = 0; k < K; ++k) nv += __ldg(knn + g * K + k) >= 0;
    const unsigned live = __ballot_sync(0xffffffffu, nv > 0);
    int32_t incl = nv;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) {
        warp_cells[warp] = __popc(live);
        warp_rows[warp] = incl;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t c = 0, r = 0;
        for (int i = 0; i < 8; ++i) {
            const int32_t tc = warp_cells[i], tr = warp_rows[i];
            warp_cells[i] = c;
            warp_rows[i] = r;
            c += tc;
            r += tr;
        }
        if (block_base) {
            base[0] = block_base[2 * blockIdx.x];
            base[1] = block_base[2 * blockIdx.x + 1];
        } else {
            base[0] = c ? atomicAdd(counters, c) : 0;
            base[1] = r ? atomicAdd(counters + 1, r) : 0;
        }
    }
    __syncthreads();
    if (nv == 0) return;
    const int32_t ci = base[0] + warp_cells[warp] + __popc(live & ((1u << lane) - 1u));
    int32_t r = base[1] + warp_rows[warp] + incl - nv;
    const int32_t b = (int32_t)(g / cells);
    const int64_t cell = g - (int64_t)b * cells;
    const int32_t i = (int32_t)(cell / W), j = (int32_t)(cell - (int64_t)i * W);
    const float cx = __fadd_rn(x0, __fmul_rn((float)i, dx)), cy = __fadd_rn(y0, __fmul_rn((float)j, dy));
    cell_list[ci] = (int32_t)g;
    cell_row0[ci] = r;
    cell_nv[ci] = (float)nv;
    for (int k = 0; k < K; ++k) {
        const int32_t p = __ldg(knn + g * K + k);
        if (p < 0) continue;
        row_pt[r] = b * N + p;
        row_cell[r] = ci;
        row_cx[r] = cx;
        row_cy[r] = cy;
        const float *q = points + ((size_t)b * N + p) * 3;
        row_off[r] = __fsub_rn(__ldg(q), cx);
        row_off[row_cap + r] = __fsub_rn(__ldg(q + 1), cy);
        row_off[2 * row_cap + r] = __ldg(q + 2);
        ++r;
    }
}

// G[ci, c] = gout[b, c, cell] for the live cells (32 cells x 32 channels per block through a shared-memory transpose;
// list neighbours are mostly grid neighbours, so the reads of a warp still fall into few lines).  The only reader of gout:
// a bf16 gout (CF_IO_BF16) is widened exactly here, and everything downstream is the fp32 path.
// NHWC (CF_IO_NHWC): gout already holds a cell's channels as one row, so each warp copies 32 channels of a live row
// straight into G.
template <typename MT, bool NHWC = false>
__global__ void __launch_bounds__(256) k_bwd_gather_g(const MT *__restrict__ gout, int32_t C, int64_t cells,
                                                      const int32_t *__restrict__ cell_list,
                                                      const int32_t *__restrict__ counters, float *__restrict__ G)
{
    const int32_t n = __ldg(counters);
    const int32_t t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    if (t0 >= n) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    if constexpr (NHWC) {
        const int32_t c = c0 + tx;
        for (int r = ty; r < 32 && t0 + r < n; r += 8) {
            const int64_t g = __ldg(cell_list + t0 + r);   // b * cells + cell: the row of the cell in a (B,H,W,C) map
            if (c < C) G[(size_t)(t0 + r) * C + c] = map_ldg(gout + g * C + c);
        }
        return;
    }
    __shared__ float tile[32][33];
    const int32_t ci = t0 + tx;
    int64_t src = -1;
    if (ci < n) {
        const int64_t g = __ldg(cell_list + ci);
        const int64_t b = g / cells;
        src = (b * C) * cells + (g - b * cells);
    }
    for (int r = ty; r < 32; r += 8) {
        const int32_t c = c0 + r;
        tile[r][tx] = (src >= 0 && c < C) ? map_ldg(gout + src + (int64_t)c * cells) : 0.0f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int32_t c = c0 + tx;
        if (t0 + r < n && c < C) G[(size_t)(t0 + r) * C + c] = tile[tx][r];
    }
}

// Recompute H1 rows (one warp per live row): H1[r, c] = relu(T[pt_r, c] - w1x[c] cx_r - w1y[c] cy_r)
__global__ void __launch_bounds__(256) k_bwd_h1(const float *__restrict__ T, const int32_t *__restrict__ row_pt,
                                                const float *__restrict__ row_cx, const float *__restrict__ row_cy,
                                                const int32_t *__restrict__ counters, int32_t C,
                                                const float *__restrict__ W1, int32_t Ci, float *__restrict__ H1)
{
    const int32_t rows = __ldg(counters + 1);
    const int lane = threadIdx.x & 31;
    const int32_t warps = gridDim.x * (blockDim.x >> 5);
    for (int32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
        const float cx = __ldg(row_cx + r), cy = __ldg(row_cy + r);
        const float *t = T + (size_t)__ldg(row_pt + r) * C;
        float *h = H1 + (size_t)r * C;
        for (int32_t c = lane; c < C; c += 32) {
            const float *w = W1 + (size_t)c * (Ci + 3) + Ci;
            h[c] = fmaxf(__ldg(t + c) - (__ldg(w) * cx + __ldg(w + 1) * cy), 0.0f);
        }
    }
}

// H2[r, c] = relu(Z[r, c] + b2[c]) (in place on Z; skipped when `activated`);  pooled[ci, c] = sum over the cell's rows
__global__ void __launch_bounds__(256) k_bwd_h2_pool(float *__restrict__ Z, const int32_t *__restrict__ cell_row0,
                                                     const float *__restrict__ cell_nv, const float *__restrict__ b2,
                                                     const int32_t *__restrict__ counters, int32_t C,
                                                     float *__restrict__ pooled, int activated)
{
    const int64_t total = (int64_t)__ldg(counters) * C;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ci = t / C;
        const int32_t c = (int32_t)(t - ci * C);
        const int64_t r0 = __ldg(cell_row0 + ci);
        const int32_t nv = (int32_t)__ldg(cell_nv + ci);
        const float bias = __ldg(b2 + c);
        float s = 0.0f;
        if (activated) {  // the GEMM epilogue already applied bias + ReLU
            for (int k = 0; k < nv; ++k) s += Z[(r0 + k) * C + c];
        } else {
            for (int k = 0; k < nv; ++k) {
                const float h = fmaxf(Z[(r0 + k) * C + c] + bias, 0.0f);
                Z[(r0 + k) * C + c] = h;
                s += h;
            }
        }
        pooled[t] = s;
    }
}

// dZ2[r, c] = dPooled[cell(r), c] * [H2[r, c] > 0]   (in place on H2)
__global__ void __launch_bounds__(256) k_bwd_dz2(float *__restrict__ H2, const float *__restrict__ dPooled,
                                                 const int32_t *__restrict__ row_cell,
                                                 const int32_t *__restrict__ counters, int32_t C)
{
    const int64_t total = (int64_t)__ldg(counters + 1) * C;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = t / C;
        const int32_t c = (int32_t)(t - r * C);
        H2[t] = H2[t] > 0.0f ? __ldg(dPooled + (size_t)__ldg(row_cell + r) * C + c) : 0.0f;
    }
}

// dT[pt_r, :] += dA[r, :]   (one warp per live row, float atomics)
__global__ void __launch_bounds__(256) k_bwd_scatter(const float *__restrict__ dA, const int32_t *__restrict__ row_pt,
                                                     const int32_t *__restrict__ counters, int32_t C,
                                                     float *__restrict__ dT)
{
    const int32_t rows = __ldg(counters + 1);
    const int lane = threadIdx.x & 31;
    const int32_t warps = gridDim.x * (blockDim.x >> 5);
    for (int32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
        const float *src = dA + (size_t)r * C;
        float *dst = dT + (size_t)__ldg(row_pt + r) * C;
        for (int32_t c = lane; c < C; c += 32) {
            const float v = __ldg(src + c);
            if (v != 0.0f) atomicAdd(dst + c, v);
        }
    }
}

// *(float *)g += v, g a global-space address.  The gather adjoint's gradient pointers come from the block's camera table as
// generic pointers, and atomicAdd on a generic pointer compiles to a generic atomic (with a shared-memory fallback) instead
// of a global reduction.
__device__ __forceinline__ void red_add_global(size_t g, float v) { asm volatile("red.global.add.f32 [%0], %1;" ::"l"(g), "f"(v) : "memory"); }

// d img_m[b, c, y, x] += (w_mt / n_vis) * dF[b, p, c] for the taps inside the map of every camera m that sees point p
// (adjoint of k_point_gather; with n_vis == 1 the quotient is w_mt itself).  Lane m < M resolves camera m; cams.map[m] is
// camera m's gradient, read from the block's camera table.
__global__ void __launch_bounds__(256) k_point_gather_bwd(const float *__restrict__ dF, const RigCams cams, int32_t M, int32_t Ci,
                                                          const CamSource src, const int64_t *__restrict__ num_points,
                                                          int32_t N)
{
    __shared__ CamTable ct;
    const int b = blockIdx.y;
    const int32_t n = valid_points(num_points, b, N);  // loaded before the barrier: its latency overlaps the staging
    stage_cams<float>(ct, cams, M, b);
    const int lane = threadIdx.x & 31;
    const int32_t warps = gridDim.x * (blockDim.x >> 5);
    const int cl = lane < M ? lane : 0;  // this lane's camera
    for (int32_t p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < n; p += warps) {
        float uf = 0.0f, vf = 0.0f;
        const int32_t Hf = ct.Hf[cl], Wf = ct.Wf[cl];
        const unsigned vis =
            __ballot_sync(0xffffffffu, lane < M && cam_project(src, b, N, p, lane, M, ct.sx[cl], ct.sy[cl], Hf, Wf, uf, vf));
        if (vis == 0) continue;
        const float nv = (float)__popc(vis);
        const Taps tp = bilinear_taps(uf, vf, Hf, Wf);
        const float l0 = __fdiv_rn(tp.w[0], nv), l1 = __fdiv_rn(tp.w[1], nv);
        const float l2 = __fdiv_rn(tp.w[2], nv), l3 = __fdiv_rn(tp.w[3], nv);
        const int lin = tp.in(0) | tp.in(1) << 1 | tp.in(2) << 2 | tp.in(3) << 3;
        const float *g = dF + ((size_t)b * N + p) * Ci;
        for (unsigned mk = vis; mk; mk &= mk - 1) {
            const int m = __ffs(mk) - 1;
            const int32_t ix = __shfl_sync(0xffffffffu, tp.x, m), iy = __shfl_sync(0xffffffffu, tp.y, m);
            const int in = __shfl_sync(0xffffffffu, lin, m);
            const float wt[4] = {__shfl_sync(0xffffffffu, l0, m), __shfl_sync(0xffffffffu, l1, m),
                                 __shfl_sync(0xffffffffu, l2, m), __shfl_sync(0xffffffffu, l3, m)};
            const int32_t tx[4] = {ix, ix + 1, ix, ix + 1}, ty[4] = {iy, iy, iy + 1, iy + 1};
            const size_t dst = __cvta_generic_to_global(ct.base[m]);
            const int64_t sc = ct.sc[m], sh = ct.sh[m], sw = ct.sw[m];
            for (int32_t c = lane; c < Ci; c += 32) {
                const float gval = __ldg(g + c);
                if (gval == 0.0f) continue;
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (in >> t & 1)
                        red_add_global(dst + sizeof(float) * (c * sc + ty[t] * sh + tx[t] * sw), __fmul_rn(wt[t], gval));
            }
        }
    }
}

// K-3's atomic adjoint for the M cameras of h_cams and one source, into the gradients h_gimg[m]; `fn` names the entry point
// in the error texts
static int point_gather_bwd(const char *fn, const float *d_gfeat, float *const *h_gimg, const cf_camera_map *h_cams, int32_t B,
                            int32_t M, int32_t Ci, const CamSource &src, const int64_t *d_num_points, int32_t N, void *stream)
{
    CF_TRY(require_sm100());
    CF_TRY(check_cams(fn, h_cams, M));
    CF_REQUIRE(d_gfeat && h_gimg && src.points && (src.dev || src.kind == CamSource::kHostCrt) && d_num_points, CF_ERR_ARG,
               "%s: null pointer", fn);
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && Ci > 0, CF_ERR_ARG, "%s: bad extents", fn);
    int64_t total;
    RigCams cams = rig_cams(h_cams, M, &total);
    for (int m = 0; m < M; ++m) {
        CF_REQUIRE(h_gimg[m] != nullptr, CF_ERR_ARG, "%s: null pointer (camera %d gradient)", fn, m);
        cams.map[m] = h_gimg[m];
    }
    // at most five blocks per SM and frame: each warp takes a few points, which pays for the block's camera table
    const int blocks = (int)std::min<int64_t>(ceil_div64(N, 8), 148 * 5);
    k_point_gather_bwd<<<dim3(blocks, B), 256, 0, (cudaStream_t)stream>>>(d_gfeat, cams, M, Ci, src, d_num_points, N);
    count_launches(1);
    return launch_status(fn);
}

// the B*M gradients of a (B,M,Ci,Hf,Wf) map with camera stride sm: M equal descriptors
static int point_gather_bwd_equal(const char *fn, const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sm, int64_t sc,
                                  int64_t sh, int64_t sw, int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf,
                                  const CamSource &src, const int64_t *d_num_points, int32_t N, float img_w, float img_h,
                                  void *stream)
{
    CF_REQUIRE(M >= 1 && M <= CF_MAX_CAMERAS, CF_ERR_ARG, "%s: M=%d cameras, expected 1..%d", fn, M, CF_MAX_CAMERAS);
    CF_REQUIRE(d_gimg != nullptr, CF_ERR_ARG, "%s: null pointer", fn);
    cf_camera_map cams[CF_MAX_CAMERAS];
    float *gimg[CF_MAX_CAMERAS];
    equal_cams(cams, d_gimg, sizeof(float), sb, sm, sc, sh, sw, M, Hf, Wf, img_w, img_h);
    for (int m = 0; m < M; ++m) gimg[m] = d_gimg + m * sm;
    return point_gather_bwd(fn, d_gfeat, gimg, cams, B, M, Ci, src, d_num_points, N, stream);
}

static size_t up256(size_t v) { return (v + 255) / 256 * 256; }

struct BwdWs {
    float *H1, *H2, *pooled, *G, *dPooled, *row_cx, *row_cy, *row_off, *cell_nv, *T, *dT, *W2t;
    int32_t *cell_list, *cell_row0, *row_pt, *row_cell, *counters;
    void *pW2, *pW2t, *pW3t, *pW1t;  // bf16 hi | lo operand images of the weights (tensor-core path)
    int32_t *blk;                    // deterministic mode: scanned (cells, rows) totals of the compaction blocks
    float *part;                     // deterministic mode: per-split partials of one row reduction at a time
    void *csr;                       // deterministic mode: rows of each point (det_dT)
    size_t bytes;
};

// sized for the dense upper bound (every slot of every cell holds a neighbour); the deterministic mode appends its buffers
static BwdWs carve(void *base, int32_t B, int32_t N, int32_t C, int32_t Ci, int64_t cells, int32_t K, bool det)
{
    BwdWs w;
    size_t off = 0;
    auto take = [&](size_t n_words) {
        void *p = base ? (void *)((char *)base + off) : nullptr;
        off += up256(n_words * 4);
        return p;
    };
    const size_t rows = (size_t)B * cells * K, ncell = (size_t)B * cells;
    w.H1 = (float *)take(rows * C);
    w.H2 = (float *)take(rows * C);
    w.pooled = (float *)take(ncell * C);
    w.G = (float *)take(ncell * C);
    w.dPooled = (float *)take(ncell * C);
    w.row_cx = (float *)take(rows);
    w.row_cy = (float *)take(rows);
    w.row_off = (float *)take(3 * rows);
    w.cell_nv = (float *)take(ncell);
    w.T = (float *)take((size_t)B * N * C);
    w.dT = (float *)take((size_t)B * N * C);
    w.W2t = (float *)take((size_t)C * C);
    w.cell_list = (int32_t *)take(ncell);
    w.cell_row0 = (int32_t *)take(ncell);
    w.row_pt = (int32_t *)take(rows);
    w.row_cell = (int32_t *)take(rows);
    w.counters = (int32_t *)take(2);
    w.pW2 = take(bwd_tc_packed_bytes(C, C) / 4);
    w.pW2t = take(bwd_tc_packed_bytes(C, C) / 4);
    w.pW3t = take(bwd_tc_packed_bytes(C, C) / 4);
    w.pW1t = take(bwd_tc_packed_bytes(Ci, C) / 4);
    w.blk = nullptr;
    w.part = nullptr;
    w.csr = nullptr;
    if (det) {
        // partials: at most kDetSplits splits of an (M <= C) x (n_out <= max(C, Ci) + 16) tile (the tcgen05 TN GEMM
        // halves the splits when M = C spans two 128-row tiles)
        w.blk = (int32_t *)take(2 * det_cell_blocks(ncell));
        w.part = (float *)take((size_t)kDetSplits * C * (std::max(C, Ci) + 16));
        w.csr = take(det_dT_words((int64_t)B * N, (int64_t)rows));
    }
    w.bytes = off;
    return w;
}

__global__ void __launch_bounds__(256) k_transpose_sq_b(const float *__restrict__ W, int32_t C, float *__restrict__ Wt)
{
    const int32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * C) return;
    const int32_t o = idx / C, i = idx - o * C;
    Wt[(size_t)i * C + o] = W[idx];
}

static inline unsigned blocks_for(int64_t n, int per, int64_t cap = 148 * 16)
{
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(n, per), cap));
}

}  // namespace

int point_mlp1_simt(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N,
                    int32_t Ci, int32_t C, const float *d_W1, const float *d_b1, float *d_T, cudaStream_t st);

}  // namespace cf

extern "C" size_t cf_fusion_bwd_workspace_bytes(int32_t B, int32_t N, int32_t C, int32_t Ci, int32_t H, int32_t W, int32_t K)
{
    if (B <= 0 || N <= 0 || C <= 0 || Ci <= 0 || H <= 0 || W <= 0 || K <= 0) return 0;
    return cf::carve(nullptr, B, N, C, Ci, (int64_t)H * W, K, false).bytes;
}

extern "C" size_t cf_fusion_bwd_det_workspace_bytes(int32_t B, int32_t N, int32_t C, int32_t Ci, int32_t H, int32_t W, int32_t K)
{
    if (B <= 0 || N <= 0 || C <= 0 || Ci <= 0 || H <= 0 || W <= 0 || K <= 0) return 0;
    return cf::carve(nullptr, B, N, C, Ci, (int64_t)H * W, K, true).bytes;
}

// Gradients are ACCUMULATED into d_gW1 (C,Ci+3), d_gb1, d_gW2 (C,C), d_gb2, d_gW3, d_gb3 and d_gfeat (B,N,Ci): the
// caller zero-initialises them (or passes buffers that already hold other scales' contributions).  d bev = d_gout.
// d_T: the table the forward computed with cf_point_mlp1 (nullptr: it is recomputed here).
// mode: CF_MODE_FP32_SIMT = every GEMM on CUDA cores (cross-check); otherwise the GEMMs whose operands fit run on tcgen05.
// mode | CF_BWD_DETERMINISTIC: bit-reproducible gradients (workspace: cf_fusion_bwd_det_workspace_bytes).
extern "C" int cf_fusion_bwd(const float *d_gout, const float *d_feat, const float *d_points,
                             const int64_t *d_num_points, const int32_t *d_knn_idx, int32_t B, int32_t N, int32_t C,
                             int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy,
                             const float *d_W1, const float *d_b1, int32_t Ci, const float *d_W2, const float *d_b2,
                             const float *d_W3, const float *d_T, float *d_gW1, float *d_gb1, float *d_gW2, float *d_gb2,
                             float *d_gW3, float *d_gb3, float *d_gfeat, int32_t mode, void *d_workspace, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    const bool det = (mode & CF_BWD_DETERMINISTIC) != 0;
    const bool io16 = (mode & CF_IO_BF16) != 0;   // d_gout is a bf16 map
    const bool nhwc = (mode & CF_IO_NHWC) != 0;   // d_gout is a (B,H,W,C) map
    mode = mode_base(mode);
    CF_REQUIRE(d_gout && d_feat && d_points && d_num_points && d_knn_idx && d_W1 && d_b1 && d_W2 && d_b2 && d_W3 &&
                   d_gW1 && d_gb1 && d_gW2 && d_gb2 && d_gW3 && d_gb3 && d_gfeat && d_workspace,
               CF_ERR_ARG, "cf_fusion_bwd: null pointer");
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && C > 0 && H > 0 && W > 0 && K >= 1 && K <= CF_MAX_K && Ci > 0 && Ci % 4 == 0,
               CF_ERR_ARG, "cf_fusion_bwd: bad extents");
    CF_REQUIRE(mode != CF_MODE_BF16_TABLES, CF_ERR_UNSUPPORTED, "cf_fusion_bwd: CF_MODE_BF16_TABLES is an inference mode (the backward reads fp32 tables)");
    CF_REQUIRE(mode == CF_MODE_FP32 || mode == CF_MODE_BF16 || mode == CF_MODE_FP32_SIMT, CF_ERR_ARG, "cf_fusion_bwd: unknown mode %d",
               mode);
    CF_REQUIRE(aligned16(d_workspace), CF_ERR_ALIGN, "cf_fusion_bwd: workspace must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cells = (int64_t)H * W, ncell = cells * B, rows = cells * K * B;
    CF_REQUIRE(rows < (int64_t)1 << 31 && (int64_t)B * N < (int64_t)1 << 31, CF_ERR_ARG,
               "cf_fusion_bwd: B*H*W*K and B*N must stay below 2^31");
    BwdWs w = carve(d_workspace, B, N, C, Ci, cells, K, det);
    const int32_t ldw1 = Ci + 3;
    const int32_t *n_cells = w.counters, *n_rows = w.counters + 1;
    const unsigned cchunks = (unsigned)((C + 31) / 32), ctiles = (unsigned)((C + 63) / 64);
    const bool tc = mode != CF_MODE_FP32_SIMT && aligned16(d_gfeat) && aligned16(d_feat) && (!d_T || aligned16(d_T));
    // [rows x C] x [C x C]: the weight image + one A chunk fit in shared memory up to C = 192; at C = 256 the GEMM runs as two
    // column halves (N = 128 each: 128 KB of weights + a 64 KB A chunk), every epilogue being local to its columns
    const int nsp = bwd_tc_nn_fits(C, C) ? 1 : 2;
    const int32_t Nh = C / nsp;
    const bool tc_row_nn = tc && bwd_tc_nn_fits(C, Nh);
    const bool tc_row_tn = tc && bwd_tc_tn_fits(C, C);
    const bool tc_pt_nn = tc && bwd_tc_nn_fits(C, Ci);    // dF = dT W1
    const bool tc_pt_tn = tc && bwd_tc_tn_fits(C, Ci);    // dW1 | db1 = dT^T [F | P | 1]
    const bool col2 = tc_row_tn && C + 1 <= 256;          // db2 / db3 ride in the GEMM as an extra column
    int launches = 0;
    float *part = det ? w.part : nullptr;
    // the two FFMA row reductions; deterministic mode: a fixed number of splits (shapes only), partials, ordered sum
    auto sgemm_tn = [&](const float *A, const float *Bm, int64_t ldb, float *Cm, int64_t ldc, int64_t R, int32_t M, int32_t N,
                        int64_t split, const int32_t *d_R) -> int {
        if (det) split = std::max<int64_t>(256, ceil_div64(R, kDetSplits));
        const unsigned z = (unsigned)ceil_div64(R, split);
        k_sgemm_tn<<<dim3((unsigned)((M + 63) / 64), (unsigned)((N + 63) / 64), z), 256, 0, st>>>(A, C, Bm, ldb, Cm, ldc, R, M, N,
                                                                                                 split, d_R, part);
        ++launches;
        return det ? det_reduce(part, M, N, N, (int32_t)z, R, d_R, 1, split, Cm, ldc, 1, nullptr, st) : CF_OK;
    };
    auto colsum = [&](const float *X, int64_t R, const float *wv, float *out, int64_t out_stride, const int32_t *d_R) -> int {
        const int64_t slab = det ? std::max<int64_t>(1024, ceil_div64(R, kDetSplits)) : 1024;
        const unsigned gx = (unsigned)ceil_div64(R, slab);
        k_colsum<<<dim3(gx, cchunks), 256, 0, st>>>(X, C, R, C, wv, 1.0f, out, out_stride, d_R, slab, part);
        ++launches;
        return det ? det_reduce(part, 1, C, C, (int32_t)gx, R, d_R, 1, slab, out, 0, out_stride, nullptr, st) : CF_OK;
    };

    // ---- live cells / rows, then the forward intermediates on them ----------------------------------------------------
    CF_TRY(cuda_status(cudaMemsetAsync(w.counters, 0, 2 * sizeof(int32_t), st), "cf_fusion_bwd memset"));
    if (det) CF_TRY(det_compact_bases(d_knn_idx, ncell, K, w.blk, w.counters, st));
    k_bwd_compact<<<(unsigned)ceil_div64(ncell, 256), 256, 0, st>>>(d_knn_idx, ncell, cells, W, K, N, x0, y0, dx, dy, w.counters,
                                                                   w.cell_list, w.cell_row0, w.cell_nv, w.row_pt, w.row_cell,
                                                                   w.row_cx, w.row_cy, d_points, w.row_off, rows, w.blk);
    const float *T = d_T;
    if (!T) {
        CF_TRY(point_mlp1_simt(d_feat, d_points, d_num_points, B, N, Ci, C, d_W1, d_b1, w.T, st));
        T = w.T;
    }
    k_bwd_h1<<<blocks_for(rows, 8), 256, 0, st>>>(T, w.row_pt, w.row_cx, w.row_cy, w.counters, C, d_W1, Ci, w.H1);
    launches += 2;
    if (tc_row_nn || tc_pt_nn) {  // operand images of W2, W2^T, W3^T (row side) and W1[:, :Ci]^T (dF) in one launch
        const float *Ws[4];
        int32_t lds[4], Nns[4], Kds[4];
        int trs[4], n = 0;
        void *imgs[4];
        auto job = [&](const float *Wm, int32_t ld, int32_t Nn, int32_t Kd, int tr, void *img) {
            Ws[n] = Wm; lds[n] = ld; Nns[n] = Nn; Kds[n] = Kd; trs[n] = tr; imgs[n] = img;
            ++n;
        };
        const size_t half_bytes = (size_t)2 * Nh * C * 2;   // one column half's image (hi | lo)
        auto flush = [&]() -> int {
            const int rc = n ? bwd_tc_pack4(Ws, lds, Nns, Kds, trs, imgs, n, st) : CF_OK;
            n = 0;
            return rc;
        };
        if (tc_row_nn) {
            for (int h = 0; h < nsp; ++h) {
                // B = W (n = output row): rows [h Nh, +Nh);  B = W^T (n = column): columns [h Nh, +Nh)
                job(d_W2 + (size_t)h * Nh * C, C, Nh, C, 0, (uint8_t *)w.pW2 + h * half_bytes);
                job(d_W2 + (size_t)h * Nh, C, Nh, C, 1, (uint8_t *)w.pW2t + h * half_bytes);
                job(d_W3 + (size_t)h * Nh, C, Nh, C, 1, (uint8_t *)w.pW3t + h * half_bytes);
                if (h + 1 < nsp) CF_TRY(flush());
            }
        }
        if (tc_pt_nn) job(d_W1, ldw1, Ci, C, 1, w.pW1t);
        CF_TRY(flush());
    }
    // row-side NN GEMM, one launch per column half
    auto row_nn = [&](const float *X, int64_t R, const int32_t *d_R, const void *img, float *Out, int epi, const float *aux, int64_t ldaux) -> int {
        const size_t half_bytes = (size_t)2 * Nh * C * 2;
        for (int h = 0; h < nsp; ++h)
            CF_TRY(bwd_tc_gemm_nn(X, C, R, d_R, C, Nh, (const uint8_t *)img + h * half_bytes, Out + (size_t)h * Nh, C, epi,
                                  aux ? aux + (size_t)h * Nh : nullptr, ldaux, st));
        return CF_OK;
    };
    if (tc_row_nn) {
        // H2 = relu(H1 W2^T + b2)
        CF_TRY(row_nn(w.H1, rows, n_rows, w.pW2, w.H2, EPI_BIAS_RELU, d_b2, 0));
    } else {
        k_transpose_sq_b<<<(C * C + 255) / 256, 256, 0, st>>>(d_W2, C, w.W2t);
        // Z2 = H1 W2^T  (as  H1 [rows x C] * W2t [C x C])
        k_sgemm_nn<<<dim3((unsigned)ceil_div64(rows, 64), ctiles), 256, 0, st>>>(w.H1, C, w.W2t, C, w.H2, C, rows, C, C, 0,
                                                                                nullptr, 0, n_rows);
        launches += 2;
    }
    k_bwd_h2_pool<<<blocks_for(ncell * C, 256), 256, 0, st>>>(w.H2, w.cell_row0, w.cell_nv, d_b2, w.counters, C, w.pooled,
                                                              tc_row_nn ? 1 : 0);

    // ---- layer 3 ------------------------------------------------------------------------------------------------------
    const dim3 g_grid((unsigned)ceil_div64(ncell, 32), cchunks);
    const __nv_bfloat16 *gout16 = reinterpret_cast<const __nv_bfloat16 *>(d_gout);
    if (io16 && nhwc)
        k_bwd_gather_g<__nv_bfloat16, true><<<g_grid, 256, 0, st>>>(gout16, C, cells, w.cell_list, w.counters, w.G);
    else if (io16)
        k_bwd_gather_g<<<g_grid, 256, 0, st>>>(gout16, C, cells, w.cell_list, w.counters, w.G);
    else if (nhwc)
        k_bwd_gather_g<float, true><<<g_grid, 256, 0, st>>>(d_gout, C, cells, w.cell_list, w.counters, w.G);
    else
        k_bwd_gather_g<<<g_grid, 256, 0, st>>>(d_gout, C, cells, w.cell_list, w.counters, w.G);
    launches += 2;
    if (tc_row_tn) {
        CF_TRY(bwd_tc_gemm_tn(w.G, C, C, w.pooled, C, C, nullptr, 0, 0, 0, w.cell_nv, ncell, n_cells, d_gW3, C,
                              col2 ? d_gb3 : nullptr, st, part));
    } else {
        CF_TRY(sgemm_tn(w.G, w.pooled, C, d_gW3, C, ncell, C, C, std::max<int64_t>(256, ceil_div64(ncell, 1184)), n_cells));
    }
    if (!(tc_row_tn && col2)) CF_TRY(colsum(w.G, ncell, w.cell_nv, d_gb3, 1, n_cells));
    // dPooled = G W3   (W3 is (out, in) row-major: exactly the [K=out x N=in] operand)
    if (tc_row_nn) {
        CF_TRY(row_nn(w.G, ncell, n_cells, w.pW3t, w.dPooled, EPI_STORE, nullptr, 0));
    } else {
        k_sgemm_nn<<<dim3((unsigned)ceil_div64(ncell, 64), ctiles), 256, 0, st>>>(w.G, C, d_W3, C, w.dPooled, C, ncell, C, C, 0,
                                                                                 nullptr, 0, n_cells);
        ++launches;
    }

    // ---- layer 2 ------------------------------------------------------------------------------------------------------
    // (masking each cell's dPooled row straight into the cell's rows of H2 in the GEMM epilogue was measured: the
    //  thread = cell, row-strided read-modify-write costs 4x the separate pass below)
    k_bwd_dz2<<<blocks_for(rows * C, 256), 256, 0, st>>>(w.H2, w.dPooled, w.row_cell, w.counters, C);  // H2 now holds dZ2
    ++launches;
    if (tc_row_tn) {
        CF_TRY(bwd_tc_gemm_tn(w.H2, C, C, w.H1, C, C, nullptr, 0, 0, 0, nullptr, rows, n_rows, d_gW2, C,
                              col2 ? d_gb2 : nullptr, st, part));
    } else {
        CF_TRY(sgemm_tn(w.H2, w.H1, C, d_gW2, C, rows, C, C, std::max<int64_t>(256, ceil_div64(rows, 1184)), n_rows));
    }
    if (!(tc_row_tn && col2)) CF_TRY(colsum(w.H2, rows, nullptr, d_gb2, 1, n_rows));
    // dA = (dZ2 W2) * [H1 > 0]   written over H1 (the mask is read before the overwrite, element by element)
    if (tc_row_nn) {
        CF_TRY(row_nn(w.H2, rows, n_rows, w.pW2t, w.H1, EPI_MASK, w.H1, C));
    } else {
        k_sgemm_nn<<<dim3((unsigned)ceil_div64(rows, 64), ctiles), 256, 0, st>>>(w.H2, C, d_W2, C, w.H1, C, rows, C, C, 0, w.H1,
                                                                                C, n_rows);
        ++launches;
    }

    // ---- layer 1: offset columns from the rows, scatter to points, point-side GEMMs ----------------------------------------
    // dW1[:, Ci + j] = sum_r dA_r * off_j(r) with off = (px - cx, py - cy, pz) of the row: summed as they entered the
    // forward (small numbers), not as the difference of two large point-side and cell-side sums
    if (tc_row_tn) {
        CF_TRY(bwd_tc_gemm_tn(w.H1, C, C, nullptr, 0, 0, w.row_off, 1, rows, 3, nullptr, rows, n_rows, d_gW1 + Ci, ldw1, nullptr,
                              st, part));
    } else {
        for (int j = 0; j < 3; ++j) CF_TRY(colsum(w.H1, rows, w.row_off + j * rows, d_gW1 + Ci + j, ldw1, n_rows));
    }
    const int64_t pts = (int64_t)B * N;
    if (det) {
        // dT as a gather over each point's rows in ascending row order (one writer per row of dT)
        CF_TRY(det_dT(w.H1, C, w.row_pt, n_rows, rows, pts, w.dT, w.csr, st));
    } else {
        CF_TRY(cuda_status(cudaMemsetAsync(w.dT, 0, (size_t)B * N * C * sizeof(float), st), "cf_fusion_bwd memset"));
        k_bwd_scatter<<<blocks_for(rows, 8), 256, 0, st>>>(w.H1, w.row_pt, w.counters, C, w.dT);
        ++launches;
    }
    // feat rows beyond num_points are zero and never referenced by knn, so their dT rows are zero as well
    if (tc_pt_tn) {
        CF_TRY(bwd_tc_gemm_tn(w.dT, C, C, d_feat, Ci, Ci, nullptr, 0, 0, 0, nullptr, pts, nullptr, d_gW1, ldw1, d_gb1, st, part));
    } else {
        CF_TRY(sgemm_tn(w.dT, d_feat, Ci, d_gW1, ldw1, pts, C, Ci, std::max<int64_t>(512, ceil_div64(pts, 148)), nullptr));
        CF_TRY(colsum(w.dT, pts, nullptr, d_gb1, 1, nullptr));
    }
    // dF += dT W1[:, :Ci]
    if (tc_pt_nn) {
        CF_TRY(bwd_tc_gemm_nn(w.dT, C, pts, nullptr, C, Ci, w.pW1t, d_gfeat, Ci, EPI_ACCUM, nullptr, 0, st));
    } else {
        k_sgemm_nn<<<dim3((unsigned)ceil_div64(pts, 64), (unsigned)((Ci + 63) / 64)), 256, 0, st>>>(
            w.dT, C, d_W1, ldw1, d_gfeat, Ci, pts, Ci, C, 1, nullptr, 0, nullptr);
        ++launches;
    }
    count_launches(launches);
    return launch_status("cf_fusion_bwd");
}

// adjoint of cf_point_gather: d_gimg (same logical shape / strides as the camera map) += scatter of d_gfeat (B,N,Ci)
extern "C" int cf_point_gather_bwd(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                                   int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                                   const float *d_uv, const float *h_calib, const int64_t *d_num_points, int32_t N,
                                   float img_w, float img_h, void *stream)
{
    using namespace cf;
    CF_REQUIRE((d_uv != nullptr) != (h_calib != nullptr), CF_ERR_ARG, "cf_point_gather_bwd: pass exactly one of d_uv / h_calib");
    return point_gather_bwd_equal("cf_point_gather_bwd", d_gfeat, d_gimg, sb, sb, sc, sh, sw, B, 1, Ci, Hf, Wf,
                                  camera_source(d_points, d_uv, h_calib), d_num_points, N, img_w, img_h, stream);
}

// adjoint of cf_point_gather_multi: d_gimg (the rig's logical (B,M,Ci,Hf,Wf) shape / strides) += scatter of d_gfeat (B,N,Ci)
extern "C" int cf_point_gather_multi_bwd(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sm, int64_t sc, int64_t sh,
                                         int64_t sw, int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf,
                                         const float *d_points, const float *d_calib, const int64_t *d_num_points, int32_t N,
                                         float img_w, float img_h, void *stream)
{
    using namespace cf;
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_calib) & 3u) == 0, CF_ERR_ALIGN, "cf_point_gather_multi_bwd: d_calib must be 4-byte aligned");
    return point_gather_bwd_equal("cf_point_gather_multi_bwd", d_gfeat, d_gimg, sb, sm, sc, sh, sw, B, M, Ci, Hf, Wf,
                                  rig_source(d_points, d_calib), d_num_points, N, img_w, img_h, stream);
}

// adjoint of cf_point_gather_rig: h_gimg[m] (camera m's logical (B,Ci,Hf_m,Wf_m) shape, strides of h_cams[m]) += scatter
extern "C" int cf_point_gather_rig_bwd(const float *d_gfeat, float *const *h_gimg, const cf_camera_map *h_cams, int32_t B,
                                       int32_t M, int32_t Ci, const float *d_points, const float *d_calib,
                                       const int64_t *d_num_points, int32_t N, void *stream)
{
    using namespace cf;
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_calib) & 3u) == 0, CF_ERR_ALIGN, "cf_point_gather_rig_bwd: d_calib must be 4-byte aligned");
    return point_gather_bwd("cf_point_gather_rig_bwd", d_gfeat, h_gimg, h_cams, B, M, Ci, rig_source(d_points, d_calib),
                            d_num_points, N, stream);
}
