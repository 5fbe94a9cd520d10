// cf_bwd_det.cu -- the deterministic variant of K-4b (cf_fusion_bwd with CF_BWD_DETERMINISTIC, cf_point_gather_bwd_det).
//
// The default backward (cf_bwd.cu, cf_bwd_tc.cu) places live cells and rows with one atomicAdd per block and sums rows into
// dW / db / dT / d img with float atomics, so its gradients are reproducible to rounding only.  Here every position and every
// sum has a fixed order:
//   - list positions come from device-wide exclusive scans (block totals -> one-block scan -> write), so the lists are in
//     grid order; the counts stay in device memory and nothing synchronises with the host;
//   - reductions over rows write one partial per row split into the workspace, and k_det_reduce adds the partials in split
//     order into the output, one thread per element.  The splits depend only on shapes and on the device-side counts
//     (kDetSplits is a constant, not the SM count), so a result reproduces on any B200;
//   - dT and d img are gathers over CSR lists (counting sort by point / pixel, each segment then ordered by its key), one
//     writer per output row.
#include <cstdio>

#include "cf_common.cuh"

namespace cf {

namespace {

// inclusive block-wide scan of one int per thread (blockDim.x a multiple of 32, <= 1024); `total` = the block's sum
__device__ __forceinline__ int32_t block_incl_scan(int32_t v, int32_t *warp_sums, int32_t &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    if (lane == 31) warp_sums[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int32_t s = lane < nw ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int32_t t = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += t;
        }
        if (lane < nw) warp_sums[lane] = s;
    }
    __syncthreads();
    total = warp_sums[nw - 1];
    const int32_t r = v + (warp ? warp_sums[warp - 1] : 0);
    __syncthreads();  // warp_sums may be reused by the caller's next scan
    return r;
}

// exclusive scan, in place, of n interleaved ncomp-tuples (one block of 1024 threads, tiles in order);
// totals[c] = the sum of component c
__global__ void __launch_bounds__(1024) k_det_scan_top(int32_t *__restrict__ vals, int64_t n, int ncomp,
                                                       int32_t *__restrict__ totals)
{
    __shared__ int32_t warp_sums[32];
    for (int c = 0; c < ncomp; ++c) {
        int32_t carry = 0;
        for (int64_t base = 0; base < n; base += blockDim.x) {
            const int64_t i = base + threadIdx.x;
            const int32_t v = i < n ? vals[i * ncomp + c] : 0;
            int32_t tot;
            const int32_t incl = block_incl_scan(v, warp_sums, tot);
            if (i < n) vals[i * ncomp + c] = carry + incl - v;
            carry += tot;
        }
        if (threadIdx.x == 0) totals[c] = carry;
    }
}

constexpr int kTile = 1024;  // elements per block of the tiled scan (256 threads x 4)

// sums of kTile-element tiles of in[0, n)
__global__ void __launch_bounds__(256) k_det_tile_sums(const int32_t *__restrict__ in, int64_t n, int32_t *__restrict__ sums)
{
    __shared__ int32_t warp_sums[32];
    const int64_t i0 = (int64_t)blockIdx.x * kTile + threadIdx.x * 4;
    int32_t v = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) v += i0 + j < n ? in[i0 + j] : 0;
    int32_t tot;
    block_incl_scan(v, warp_sums, tot);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

// out[i] = exclusive prefix of in at i (tile bases from k_det_scan_top)
__global__ void __launch_bounds__(256) k_det_tile_scan(const int32_t *__restrict__ in, int64_t n,
                                                       const int32_t *__restrict__ tile_base, int32_t *__restrict__ out)
{
    __shared__ int32_t warp_sums[32];
    const int64_t i0 = (int64_t)blockIdx.x * kTile + threadIdx.x * 4;
    int32_t v[4], s = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = i0 + j < n ? in[i0 + j] : 0;
        s += v[j];
    }
    int32_t tot;
    int32_t run = block_incl_scan(s, warp_sums, tot) - s + tile_base[blockIdx.x];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (i0 + j < n) out[i0 + j] = run;
        run += v[j];
    }
}

// per 256-cell block of the neighbour table: (live cells, live rows) -> blk[2 * block], blk[2 * block + 1]
__global__ void __launch_bounds__(256) k_det_cell_totals(const int32_t *__restrict__ knn, int64_t ncell, int32_t K,
                                                         int32_t *__restrict__ blk)
{
    __shared__ int32_t warp_sums[32];
    const int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x;
    int32_t nv = 0;
    if (g < ncell)
        for (int k = 0; k < K; ++k) nv += __ldg(knn + g * K + k) >= 0;
    int32_t cells, rows;
    block_incl_scan(nv > 0 ? 1 : 0, warp_sums, cells);
    block_incl_scan(nv, warp_sums, rows);
    if (threadIdx.x == 0) {
        blk[2 * blockIdx.x] = cells;
        blk[2 * blockIdx.x + 1] = rows;
    }
}

// dW[m * ldw + n * cs] (n < n_w) or db[m] (n == n_w) += sum over the active splits s, in order, of part[s][m][n]
// (part: [nsplit][M][n_out]).  A split is active when its row range is not empty: the producers skip empty ones.
// Row ranges: `per_fixed` rows per split, or (per_fixed == 0) ceil(units / nsplit) units of `unit` rows each.
__global__ void __launch_bounds__(256) k_det_reduce(const float *__restrict__ part, int32_t M, int32_t n_w, int32_t n_out,
                                                    int32_t nsplit, int64_t R, const int32_t *__restrict__ d_R, int64_t unit,
                                                    int64_t per_fixed, float *__restrict__ dW, int64_t ldw, int64_t cs,
                                                    float *__restrict__ db)
{
    const int64_t Rv = d_R ? min(R, (int64_t)__ldg(d_R)) : R;
    const int64_t units = ceil_div64(Rv, unit);
    const int64_t per = per_fixed ? per_fixed : ceil_div64(units, nsplit);
    const int64_t active = per > 0 ? min((int64_t)nsplit, ceil_div64(units, per)) : 0;
    if (active == 0) return;
    const int64_t total = (int64_t)M * n_out;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t m = idx / n_out;
        const int32_t n = (int32_t)(idx - m * n_out);
        float s = 0.0f;
        for (int64_t k = 0; k < active; ++k) s += __ldg(part + k * total + idx);
        if (n < n_w) dW[m * ldw + (int64_t)n * cs] += s;
        else db[m] += s;
    }
}

// rows per point: cnt[row_pt[r]] += 1 (integer atomics: the counts do not depend on the order)
__global__ void __launch_bounds__(256) k_det_pt_count(const int32_t *__restrict__ row_pt, const int32_t *__restrict__ n_rows,
                                                      int32_t *__restrict__ cnt)
{
    const int32_t rows = __ldg(n_rows);
    for (int32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) atomicAdd(cnt + __ldg(row_pt + r), 1);
}

// seg[off[pt] .. off[pt + 1]) = the rows of pt, in arrival order (cnt counts down to 0)
__global__ void __launch_bounds__(256) k_det_pt_fill(const int32_t *__restrict__ row_pt, const int32_t *__restrict__ n_rows,
                                                     const int32_t *__restrict__ off, int32_t *__restrict__ cnt,
                                                     int32_t *__restrict__ seg)
{
    const int32_t rows = __ldg(n_rows);
    for (int32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
        const int32_t p = __ldg(row_pt + r);
        seg[__ldg(off + p) + atomicSub(cnt + p, 1) - 1] = r;
    }
}

// one warp orders the segment [s0, s0 + L) of distinct keys ascending into `dst` (rank = number of smaller keys), carrying
// an optional float payload; any L
__device__ __forceinline__ void warp_rank_sort(const int32_t *__restrict__ key, const float *__restrict__ val, int64_t s0,
                                               int32_t L, int32_t *__restrict__ key_dst, float *__restrict__ val_dst)
{
    const int lane = threadIdx.x & 31;
    for (int32_t i = lane; i < L; i += 32) {
        const int32_t v = key[s0 + i];
        int32_t rank = 0;
        for (int32_t j = 0; j < L; ++j) rank += key[s0 + j] < v;
        key_dst[s0 + rank] = v;
        if (val) val_dst[s0 + rank] = val[s0 + i];
    }
    __syncwarp();
}

// dT[p, :] = sum of dA[r, :] over the rows r of point p in ascending r (one warp per point, lane = channel; every row of
// dT is written, zero for points without rows)
__global__ void __launch_bounds__(256) k_det_dT(const float *__restrict__ dA, int32_t C, const int32_t *__restrict__ off,
                                                const int32_t *__restrict__ seg, int32_t *__restrict__ sorted, int64_t pts,
                                                float *__restrict__ dT)
{
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < pts; p += warps) {
        const int32_t s0 = __ldg(off + p), L = __ldg(off + p + 1) - s0;
        warp_rank_sort(seg, nullptr, s0, L, sorted, nullptr);
        for (int32_t c = lane; c < C; c += 32) {
            float s = 0.0f;
            for (int32_t j = 0; j < L; ++j) s += __ldg(dA + (size_t)sorted[s0 + j] * C + c);
            dT[(size_t)p * C + c] = s;
        }
        __syncwarp();
    }
}

// ---- camera-map gradient ----------------------------------------------------------------------------------------------
// The pixel space is the concatenation over (b, m) of the camera planes Hf_m * Wf_m: frame b starts at b * total, camera m
// at cams.plane[m] within it (equal cameras: map index b * M + m).  fill == 0: cnt[pixel] += 1 per tap inside its camera's
// map;  fill == 1: place (key = 4 p + t, weight w_mt / n_vis) into the pixel's segment.  Thread = point of frame blockIdx.y;
// cameras in ascending order, the camera loops unrolled so that every camera's constants are read at a fixed index.
__global__ void __launch_bounds__(256) k_gdet_taps(const CamSource src, const int64_t *__restrict__ num_points,
                                                   const RigCams cams, int32_t M, int32_t N, int64_t total, int fill,
                                                   int32_t *__restrict__ cnt, const int32_t *__restrict__ off,
                                                   int32_t *__restrict__ key, float *__restrict__ wgt)
{
    const int b = blockIdx.y;
    const int32_t n = valid_points(num_points, b, N);
    for (int32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        // the visible set first (n_vis divides every weight), then the taps of each visible camera, projected again
        unsigned vis = 0;
        float uf, vf;
#pragma unroll
        for (int m = 0; m < CF_MAX_CAMERAS; ++m)
            if (m < M && cam_project(src, b, N, p, m, M, cams.sx[m], cams.sy[m], cams.Hf[m], cams.Wf[m], uf, vf)) vis |= 1u << m;
        const float nv = (float)__popc(vis);
#pragma unroll
        for (int m = 0; m < CF_MAX_CAMERAS; ++m) {
            if (!(vis >> m & 1u)) continue;
            const int32_t Hf = cams.Hf[m], Wf = cams.Wf[m];
            cam_project(src, b, N, p, m, M, cams.sx[m], cams.sy[m], Hf, Wf, uf, vf);
            const Taps tp = bilinear_taps(uf, vf, Hf, Wf);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (!tp.in(t)) continue;
                const int64_t px = (int64_t)b * total + cams.plane[m] + (int64_t)(tp.y + (t >> 1)) * Wf + tp.x + (t & 1);
                if (!fill) {
                    atomicAdd(cnt + px, 1);
                } else {
                    const int32_t pos = __ldg(off + px) + atomicSub(cnt + px, 1) - 1;
                    key[pos] = p * 4 + t;
                    wgt[pos] = __fdiv_rn(tp.w[t], nv);
                }
            }
        }
    }
}

// d img_m[b, c, y, x] += sum over the pixel's taps in ascending (point, tap) of w * dF[b, p, c]  (one warp per pixel of the
// pixel space; cams.map[m] is camera m's gradient)
__global__ void __launch_bounds__(256) k_gdet_sum(const float *__restrict__ dF, const RigCams cams, int32_t Ci, int32_t N,
                                                  int64_t total, int64_t npx, const int32_t *__restrict__ off,
                                                  const int32_t *__restrict__ key, const float *__restrict__ wgt,
                                                  int32_t *__restrict__ key_s, float *__restrict__ wgt_s)
{
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t px = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); px < npx; px += warps) {
        const int32_t s0 = __ldg(off + px), L = __ldg(off + px + 1) - s0;
        if (L == 0) continue;
        warp_rank_sort(key, wgt, s0, L, key_s, wgt_s);
        const int64_t b = px / total;
        const int32_t r = (int32_t)(px - b * total);  // < total <= 2^31 / B
        int m = 0;
#pragma unroll
        for (int k = 1; k < CF_MAX_CAMERAS; ++k) m += r >= cams.plane[k];  // plane[k] = INT32_MAX past the last camera
        const Cam cm = cam_get(cams, m);
        const int32_t yx = r - cm.plane, y = yx / cm.Wf, x = yx - y * cm.Wf;
        const float *src = dF + (size_t)b * N * Ci;
        float *dst = (float *)cm.map + b * cm.sb + y * cm.sh + x * cm.sw;
        for (int32_t c = lane; c < Ci; c += 32) {
            float s = 0.0f;
            for (int32_t j = 0; j < L; ++j)
                s = __fadd_rn(s, __fmul_rn(wgt_s[s0 + j], __ldg(src + (size_t)(key_s[s0 + j] >> 2) * Ci + c)));
            dst[c * cm.sc] += s;
        }
        __syncwarp();
    }
}

size_t up256(size_t v) { return (v + 255) / 256 * 256; }

// off[0, n] = exclusive prefix of cnt[0, n), off[n] = total: three launches
int scan_counts(const int32_t *cnt, int64_t n, int32_t *off, int32_t *tile_sums, cudaStream_t st)
{
    const int64_t tiles = std::max<int64_t>(1, ceil_div64(n, kTile));
    k_det_tile_sums<<<(unsigned)tiles, 256, 0, st>>>(cnt, n, tile_sums);
    k_det_scan_top<<<1, 1024, 0, st>>>(tile_sums, tiles, 1, off + n);
    k_det_tile_scan<<<(unsigned)tiles, 256, 0, st>>>(cnt, n, tile_sums, off);
    count_launches(3);
    return launch_status("deterministic scan");
}

size_t scan_tile_words(int64_t n) { return (size_t)std::max<int64_t>(1, ceil_div64(n, kTile)); }

}  // namespace

// ---- entry points for cf_bwd.cu / cf_bwd_tc.cu -------------------------------------------------------------------------
size_t det_cell_blocks(int64_t ncell) { return (size_t)ceil_div64(ncell, 256); }

// block bases (2 per 256-cell block) of k_bwd_compact and the two counts, in grid order
int det_compact_bases(const int32_t *knn, int64_t ncell, int32_t K, int32_t *blk, int32_t *counters, cudaStream_t st)
{
    const int64_t nb = ceil_div64(ncell, 256);
    k_det_cell_totals<<<(unsigned)nb, 256, 0, st>>>(knn, ncell, K, blk);
    k_det_scan_top<<<1, 1024, 0, st>>>(blk, nb, 2, counters);
    count_launches(2);
    return launch_status("cf_fusion_bwd (ordered compaction)");
}

int det_reduce(const float *part, int32_t M, int32_t n_w, int32_t n_out, int32_t nsplit, int64_t R, const int32_t *d_R,
               int64_t unit, int64_t per_fixed, float *dW, int64_t ldw, int64_t cs, float *db, cudaStream_t st)
{
    const int64_t total = (int64_t)M * n_out;
    k_det_reduce<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(total, 256), 1024)), 256, 0, st>>>(
        part, M, n_w, n_out, nsplit, R, d_R, unit, per_fixed, dW, ldw, cs, db);
    count_launches(1);
    return launch_status("cf_fusion_bwd (fixed-order reduce)");
}

// words of workspace det_dT needs for `pts` points and `rows` dense rows
size_t det_dT_words(int64_t pts, int64_t rows)
{
    return up256(4 * (size_t)pts) / 4 + up256(4 * ((size_t)pts + 1)) / 4 + 2 * (up256(4 * (size_t)rows) / 4) +
           up256(4 * scan_tile_words(pts)) / 4;
}

// dT (pts x C) = per-point sums of the rows of dA, in ascending row order
int det_dT(const float *dA, int32_t C, const int32_t *row_pt, const int32_t *n_rows, int64_t rows, int64_t pts, float *dT,
           void *ws, cudaStream_t st)
{
    int32_t *cnt = (int32_t *)ws;
    int32_t *off = cnt + up256(4 * (size_t)pts) / 4;
    int32_t *seg = off + up256(4 * ((size_t)pts + 1)) / 4;
    int32_t *sorted = seg + up256(4 * (size_t)rows) / 4;
    int32_t *tiles = sorted + up256(4 * (size_t)rows) / 4;
    CF_TRY(cuda_status(cudaMemsetAsync(cnt, 0, (size_t)pts * sizeof(int32_t), st), "cf_fusion_bwd memset"));
    const unsigned rb = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(rows, 256), 148 * 16));
    k_det_pt_count<<<rb, 256, 0, st>>>(row_pt, n_rows, cnt);
    count_launches(1);
    CF_TRY(scan_counts(cnt, pts, off, tiles, st));
    k_det_pt_fill<<<rb, 256, 0, st>>>(row_pt, n_rows, off, cnt, seg);
    k_det_dT<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(pts, 8), 148 * 16)), 256, 0, st>>>(dA, C, off, seg,
                                                                                                          sorted, pts, dT);
    count_launches(2);
    return launch_status("cf_fusion_bwd (dT)");
}

}  // namespace cf

namespace {
struct GdetWs {
    int32_t *cnt, *off, *key, *key_s, *tiles;
    float *wgt, *wgt_s;
    size_t bytes;
};

GdetWs gdet_carve(void *base, int64_t npx, int64_t taps)
{
    GdetWs w;
    size_t o = 0;
    auto take = [&](size_t words) {
        void *p = base ? (void *)((char *)base + o) : nullptr;
        o += (words * 4 + 255) / 256 * 256;
        return p;
    };
    w.cnt = (int32_t *)take(npx);
    w.off = (int32_t *)take(npx + 1);
    w.key = (int32_t *)take(taps);
    w.key_s = (int32_t *)take(taps);
    w.wgt = (float *)take(taps);
    w.wgt_s = (float *)take(taps);
    w.tiles = (int32_t *)take((npx + 1023) / 1024 + 1);
    w.bytes = o;
    return w;
}

// the pixels of the B frames' camera planes
int64_t gdet_pixels(int32_t B, int32_t M, const cf_camera_map *h_cams)
{
    int64_t per = 0;
    for (int m = 0; m < M; ++m) per += (int64_t)h_cams[m].Hf * h_cams[m].Wf;
    return (int64_t)B * per;
}

// K-3's fixed-order adjoint for the M cameras of h_cams and one source, into the gradients h_gimg[m]: CSR of the (point,
// tap) contributions by pixel of the concatenated camera planes, one thread per (pixel, channel) summing its segment in
// ascending (point, tap) order; `fn` names the entry point in the error texts
static int point_gather_bwd_det(const char *fn, const float *d_gfeat, float *const *h_gimg, const cf_camera_map *h_cams,
                                int32_t B, int32_t M, int32_t Ci, const cf::CamSource &src, const int64_t *d_num_points,
                                int32_t N, void *d_workspace, void *stream)
{
    using namespace cf;
    const char *bm = src.kind == CamSource::kRig ? "B*M" : "B";
    CF_TRY(require_sm100());
    CF_TRY(check_cams(fn, h_cams, M));
    CF_REQUIRE(d_gfeat && h_gimg && src.points && (src.dev || src.kind == CamSource::kHostCrt) && d_num_points && d_workspace,
               CF_ERR_ARG, "%s: null pointer", fn);
    CF_REQUIRE(B > 0 && B <= 65535 && N > 0 && Ci > 0, CF_ERR_ARG, "%s: bad extents", fn);
    const int64_t npx = gdet_pixels(B, M, h_cams);
    CF_REQUIRE((int64_t)4 * B * M * N < ((int64_t)1 << 31) && npx < ((int64_t)1 << 31), CF_ERR_ARG,
               "%s: 4*%s*N and B*Sum_m Hf_m*Wf_m must stay below 2^31", fn, bm);
    int64_t total;
    RigCams cams = rig_cams(h_cams, M, &total);
    for (int m = 0; m < M; ++m) {
        CF_REQUIRE(h_gimg[m] != nullptr, CF_ERR_ARG, "%s: null pointer (camera %d gradient)", fn, m);
        cams.map[m] = h_gimg[m];
    }
    cudaStream_t st = (cudaStream_t)stream;
    GdetWs w = gdet_carve(d_workspace, npx, (int64_t)4 * B * M * N);
    char what[64];
    snprintf(what, sizeof what, "%s memset", fn);
    CF_TRY(cuda_status(cudaMemsetAsync(w.cnt, 0, (size_t)npx * sizeof(int32_t), st), what));
    const dim3 tg((unsigned)std::min<int64_t>(ceil_div64(N, 256), 148 * 4), (unsigned)B);
    k_gdet_taps<<<tg, 256, 0, st>>>(src, d_num_points, cams, M, N, total, 0, w.cnt, nullptr, nullptr, nullptr);
    count_launches(1);
    CF_TRY(scan_counts(w.cnt, npx, w.off, w.tiles, st));
    k_gdet_taps<<<tg, 256, 0, st>>>(src, d_num_points, cams, M, N, total, 1, w.cnt, w.off, w.key, w.wgt);
    k_gdet_sum<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(npx, 8), 148 * 16)), 256, 0, st>>>(
        d_gfeat, cams, Ci, N, total, npx, w.off, w.key, w.wgt, w.key_s, w.wgt_s);
    count_launches(2);
    return launch_status(fn);
}

// the B*M gradients of a (B,M,Ci,Hf,Wf) map with camera stride sm: M equal descriptors
static int point_gather_bwd_det_equal(const char *fn, const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sm, int64_t sc,
                                      int64_t sh, int64_t sw, int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf,
                                      const cf::CamSource &src, const int64_t *d_num_points, int32_t N, float img_w,
                                      float img_h, void *d_workspace, void *stream)
{
    CF_REQUIRE(M >= 1 && M <= CF_MAX_CAMERAS, CF_ERR_ARG, "%s: M=%d cameras, expected 1..%d", fn, M, CF_MAX_CAMERAS);
    CF_REQUIRE(d_gimg != nullptr, CF_ERR_ARG, "%s: null pointer", fn);
    cf_camera_map cams[CF_MAX_CAMERAS];
    float *gimg[CF_MAX_CAMERAS];
    cf::equal_cams(cams, d_gimg, sizeof(float), sb, sm, sc, sh, sw, M, Hf, Wf, img_w, img_h);
    for (int m = 0; m < M; ++m) gimg[m] = d_gimg + m * sm;
    return point_gather_bwd_det(fn, d_gfeat, gimg, cams, B, M, Ci, src, d_num_points, N, d_workspace, stream);
}
}  // namespace

extern "C" size_t cf_point_gather_multi_bwd_det_workspace_bytes(int32_t B, int32_t M, int32_t N, int32_t Hf, int32_t Wf)
{
    if (B <= 0 || M <= 0 || N <= 0 || Hf <= 0 || Wf <= 0) return 0;
    return gdet_carve(nullptr, (int64_t)B * M * Hf * Wf, (int64_t)4 * B * M * N).bytes;   // B*M maps, up to 4 taps per point in each
}

extern "C" size_t cf_point_gather_bwd_det_workspace_bytes(int32_t B, int32_t N, int32_t Hf, int32_t Wf)
{
    return cf_point_gather_multi_bwd_det_workspace_bytes(B, 1, N, Hf, Wf);
}

extern "C" size_t cf_point_gather_rig_bwd_det_workspace_bytes(int32_t B, int32_t M, int32_t N, const cf_camera_map *h_cams)
{
    if (h_cams == nullptr || B <= 0 || M <= 0 || M > CF_MAX_CAMERAS || N <= 0) return 0;
    for (int m = 0; m < M; ++m)
        if (h_cams[m].Hf <= 0 || h_cams[m].Wf <= 0) return 0;
    return gdet_carve(nullptr, gdet_pixels(B, M, h_cams), (int64_t)4 * B * M * N).bytes;
}

// cf_point_gather_bwd with a fixed summation order: the rig path over B*1 maps
extern "C" int cf_point_gather_bwd_det(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                                       int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                                       const float *d_uv, const float *h_calib, const int64_t *d_num_points, int32_t N,
                                       float img_w, float img_h, void *d_workspace, void *stream)
{
    CF_REQUIRE((d_uv != nullptr) != (h_calib != nullptr), CF_ERR_ARG,
               "cf_point_gather_bwd_det: pass exactly one of d_uv / h_calib");
    return point_gather_bwd_det_equal("cf_point_gather_bwd_det", d_gfeat, d_gimg, sb, sb, sc, sh, sw, B, 1, Ci, Hf, Wf,
                                      cf::camera_source(d_points, d_uv, h_calib), d_num_points, N, img_w, img_h, d_workspace,
                                      stream);
}

// cf_point_gather_multi_bwd with a fixed summation order: the lists of cf_point_gather_bwd_det over the B*M maps
extern "C" int cf_point_gather_multi_bwd_det(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sm, int64_t sc,
                                             int64_t sh, int64_t sw, int32_t B, int32_t M, int32_t Ci, int32_t Hf, int32_t Wf,
                                             const float *d_points, const float *d_calib, const int64_t *d_num_points,
                                             int32_t N, float img_w, float img_h, void *d_workspace, void *stream)
{
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_calib) & 3u) == 0, CF_ERR_ALIGN,
               "cf_point_gather_multi_bwd_det: d_calib must be 4-byte aligned");
    return point_gather_bwd_det_equal("cf_point_gather_multi_bwd_det", d_gfeat, d_gimg, sb, sm, sc, sh, sw, B, M, Ci, Hf, Wf,
                                      cf::rig_source(d_points, d_calib), d_num_points, N, img_w, img_h, d_workspace, stream);
}

// cf_point_gather_rig_bwd with a fixed summation order: the lists over the concatenated camera planes of the B frames
extern "C" int cf_point_gather_rig_bwd_det(const float *d_gfeat, float *const *h_gimg, const cf_camera_map *h_cams, int32_t B,
                                           int32_t M, int32_t Ci, const float *d_points, const float *d_calib,
                                           const int64_t *d_num_points, int32_t N, void *d_workspace, void *stream)
{
    CF_REQUIRE((reinterpret_cast<uintptr_t>(d_calib) & 3u) == 0, CF_ERR_ALIGN,
               "cf_point_gather_rig_bwd_det: d_calib must be 4-byte aligned");
    return point_gather_bwd_det("cf_point_gather_rig_bwd_det", d_gfeat, h_gimg, h_cams, B, M, Ci,
                                cf::rig_source(d_points, d_calib), d_num_points, N, d_workspace, stream);
}
