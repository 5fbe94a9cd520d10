// cf_knn.cu -- K-2: bounded-radius top-K nearest LiDAR points per BEV cell over the bucket grid.
//
// One thread per BEV cell.  The K best candidates live in registers as 64-bit keys
// (bits(d2) << 32 | index): d2 >= 0, so the IEEE bit pattern orders like the value and one unsigned
// compare implements the total order (d2, idx) of SURVEY Appendix A5.  Buckets are visited in
// Chebyshev rings around the cell's own bucket; inside a ring every bucket-row segment is one
// contiguous slice of the sorted point array.  The search stops as soon as the K-th best distance is
// strictly below a conservative lower bound of everything not yet visited, or when the bounding
// square of the radius disc is exhausted.  Distances use __fsub_rn/__fmul_rn/__fadd_rn so no FMA
// contraction can make d2 differ from the CPU oracle (Appendix A2).
#include "cf_common.cuh"

namespace cf {

struct KnnGeom {
    float x0, y0, dx, dy;  // cell centre: x0 + i*dx, y0 + j*dy
    float radius, r2;
    int32_t H, W;
};

template <int K>
__device__ __forceinline__ void knn_insert(unsigned long long (&best)[K], unsigned long long key)
{
    // precondition: key < best[K-1]
    best[K - 1] = key;
#pragma unroll
    for (int q = K - 1; q > 0; --q) {
        const unsigned long long a = best[q - 1], b = best[q];
        const bool sw = b < a;
        best[q - 1] = sw ? b : a;
        best[q] = sw ? a : b;
    }
}

// one candidate against one cell: exact fp32 d2 (no FMA), radius / K-th distance pre-filter, ordered insertion
template <int K>
__device__ __forceinline__ void knn_test(const float4 q, float cx, float cy, float r2, float &thr,
                                         unsigned long long (&best)[K])
{
    const float ddx = __fsub_rn(q.x, cx);
    const float ddy = __fsub_rn(q.y, cy);
    const float d2 = __fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy));
    if (d2 <= thr) {  // thr = min(r2, current K-th d2): ties at the K-th distance still reach the key compare
        const unsigned long long key =
            ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)__float_as_uint(q.w);
        if (key < best[K - 1]) {
            knn_insert<K>(best, key);
            if (best[K - 1] != ~0ull) thr = fminf(r2, __uint_as_float((unsigned)(best[K - 1] >> 32)));
        }
    }
}

template <int K>
__device__ __forceinline__ void knn_scan(const float4 *__restrict__ sp, int32_t s, int32_t e, float cx, float cy,
                                         float r2, unsigned long long (&best)[K])
{
    float thr = best[K - 1] != ~0ull ? fminf(r2, __uint_as_float((unsigned)(best[K - 1] >> 32))) : r2;
    for (int32_t p = s; p < e; ++p) knn_test<K>(__ldg(sp + p), cx, cy, r2, thr, best);
}

template <int K>
__global__ void __launch_bounds__(128) k_knn_query(const int32_t *__restrict__ bucket_start,
                                                   const float4 *__restrict__ sorted, int32_t N, BucketGrid g,
                                                   KnnGeom q, int32_t *__restrict__ knn_idx)
{
    const int b = blockIdx.y;
    const int64_t cells = (int64_t)q.H * q.W;
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= cells) return;
    const int32_t i = (int32_t)(cell / q.W), j = (int32_t)(cell - (int64_t)i * q.W);
    const float cx = __fadd_rn(q.x0, __fmul_rn((float)i, q.dx));
    const float cy = __fadd_rn(q.y0, __fmul_rn((float)j, q.dy));

    const int32_t G = g.nbx * g.nby;
    const int32_t *__restrict__ bs = bucket_start + (size_t)b * (G + 1);
    const float4 *__restrict__ sp = sorted + (size_t)b * N;

    unsigned long long best[K];
#pragma unroll
    for (int k = 0; k < K; ++k) best[k] = ~0ull;

    // Conservative slack for every comparison between a bucket boundary and a distance: bucket
    // assignment and boundary coordinates carry a few ulp of fp32 error (<< 1e-4*cell for |coords| < 1e4).
    const float margin = 0.01f * g.cell;
    const float reach = q.radius + margin;
    const int32_t bxlo = bucket_coord(cx - reach, g.gx0, g.inv_cell, g.nbx);
    const int32_t bxhi = bucket_coord(cx + reach, g.gx0, g.inv_cell, g.nbx);
    const int32_t bylo = bucket_coord(cy - reach, g.gy0, g.inv_cell, g.nby);
    const int32_t byhi = bucket_coord(cy + reach, g.gy0, g.inv_cell, g.nby);
    const int32_t bcx = bucket_coord(cx, g.gx0, g.inv_cell, g.nbx);
    const int32_t bcy = bucket_coord(cy, g.gy0, g.inv_cell, g.nby);
    const int32_t rho_max = max(max(bcx - bxlo, bxhi - bcx), max(bcy - bylo, byhi - bcy));

    for (int32_t rho = 0; rho <= rho_max; ++rho) {
        const int32_t xa = bcx - rho, xb = bcx + rho;
        const int32_t ya = bcy - rho, yb = bcy + rho;
        const int32_t yac = max(ya, bylo), ybc = min(yb, byhi);
        if (yac <= ybc) {
            if (xa >= bxlo) {  // first row of the ring, full width
                const int32_t s = __ldg(bs + xa * g.nby + yac), e = __ldg(bs + xa * g.nby + ybc + 1);
                knn_scan<K>(sp, s, e, cx, cy, q.r2, best);
            }
            if (rho > 0 && xb <= bxhi) {  // last row
                const int32_t s = __ldg(bs + xb * g.nby + yac), e = __ldg(bs + xb * g.nby + ybc + 1);
                knn_scan<K>(sp, s, e, cx, cy, q.r2, best);
            }
        }
        if (rho > 0) {  // the two side columns of the rows in between
            const int32_t x_lo = max(xa + 1, bxlo), x_hi = min(xb - 1, bxhi);
            for (int32_t x = x_lo; x <= x_hi; ++x) {
                if (ya >= bylo) {
                    const int32_t s = __ldg(bs + x * g.nby + ya), e = __ldg(bs + x * g.nby + ya + 1);
                    knn_scan<K>(sp, s, e, cx, cy, q.r2, best);
                }
                if (yb <= byhi) {
                    const int32_t s = __ldg(bs + x * g.nby + yb), e = __ldg(bs + x * g.nby + yb + 1);
                    knn_scan<K>(sp, s, e, cx, cy, q.r2, best);
                }
            }
        }
        // early exit: everything not yet visited lies outside the (2rho+1)^2 block of buckets
        if (rho < rho_max && best[K - 1] != ~0ull) {
            float lb = 3.0e38f;
            if (xa > bxlo) lb = fminf(lb, cx - (g.gx0 + (float)xa * g.cell));
            if (xb < bxhi) lb = fminf(lb, (g.gx0 + (float)(xb + 1) * g.cell) - cx);
            if (ya > bylo) lb = fminf(lb, cy - (g.gy0 + (float)ya * g.cell));
            if (yb < byhi) lb = fminf(lb, (g.gy0 + (float)(yb + 1) * g.cell) - cy);
            const float lbs = lb - margin;
            const float kth = __uint_as_float((unsigned)(best[K - 1] >> 32));
            if (lbs > 0.0f && kth < lbs * lbs * 0.999999f) break;
        }
    }

    int32_t *out = knn_idx + ((size_t)b * cells + cell) * K;
#pragma unroll
    for (int k = 0; k < K; ++k) out[k] = best[k] == ~0ull ? -1 : (int32_t)(unsigned)(best[k] & 0xffffffffull);
}

// ---------------------------------------------------------------------------------------------------------------
// Patch kernel (fine scales).  One WARP owns a patch of 4 x 8 neighbouring BEV cells, one lane per cell; the 32
// cells share almost all of their candidates, so the warp gathers ONE candidate set cooperatively (coalesced loads,
// ballot compaction into shared memory) and every lane then scans it with uniform control flow.
//
// Exactness.  Let c be the patch centre, hd the half diagonal of the patch's cell centres, and U >= d_K(c) any upper
// bound of the K-th nearest distance from c (U = inf when fewer than K points are in reach).  For a cell x of the
// patch the K points nearest to c lie within U + |x - c| <= U + hd of x, hence d_K(x) <= U + hd, and every true
// neighbour p of x has |p - x| <= min(r, U + hd), i.e. |p - c| <= R := min(r, U + hd) + hd.  The candidate set
// { p : |p - c| <= R (1 + 1e-4) + 1e-4 } therefore contains the exact answer of every cell; each lane orders its
// candidates by the same (d2, idx) keys as the brute-force oracle, so the result is bit-identical.
// U is the K-th smallest distance inside the first bucket block around c that holds >= K points.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kPatchI = 4, kPatchJ = 8, kCandCap = 256;

__device__ __forceinline__ int32_t warp_sum(int32_t v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// number of points in bucket rows [xa,xb] x columns [ya,yb] (lanes split the rows)
__device__ __forceinline__ int32_t block_count(const int32_t *__restrict__ bs, int32_t nby, int32_t xa, int32_t xb,
                                               int32_t ya, int32_t yb, int lane)
{
    int32_t c = 0;
    for (int32_t x = xa + lane; x <= xb; x += 32) c += __ldg(bs + x * nby + yb + 1) - __ldg(bs + x * nby + ya);
    return warp_sum(c);
}

template <int K>
__global__ void __launch_bounds__(128) k_knn_patch(const int32_t *__restrict__ bucket_start,
                                                   const float4 *__restrict__ sorted, int32_t N, BucketGrid g,
                                                   KnnGeom q, int32_t *__restrict__ knn_idx)
{
    constexpr bool kCentreOut = K >= 8;   // candidate order of the gather (see below)
    __shared__ float4 cand_all[4][kCandCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.y;
    const int32_t pj_n = (q.W + kPatchJ - 1) / kPatchJ, pi_n = (q.H + kPatchI - 1) / kPatchI;
    const int64_t patch = (int64_t)blockIdx.x * 4 + warp;
    if (patch >= (int64_t)pj_n * pi_n) return;  // whole warp
    float4 *cand = cand_all[warp];
    const int32_t i0 = (int32_t)(patch / pj_n) * kPatchI, j0 = (int32_t)(patch % pj_n) * kPatchJ;
    const int32_t i = i0 + (lane >> 3), j = j0 + (lane & 7);
    const bool active = i < q.H && j < q.W;
    const float cx = __fadd_rn(q.x0, __fmul_rn((float)i, q.dx));
    const float cy = __fadd_rn(q.y0, __fmul_rn((float)j, q.dy));
    // patch centre / half diagonal from its corner cell centres
    const float xl = q.x0 + (float)i0 * q.dx, xh = q.x0 + (float)(i0 + kPatchI - 1) * q.dx;
    const float yl = q.y0 + (float)j0 * q.dy, yh = q.y0 + (float)(j0 + kPatchJ - 1) * q.dy;
    const float pcx = 0.5f * (xl + xh), pcy = 0.5f * (yl + yh);
    const float hx = 0.5f * fabsf(xh - xl), hy = 0.5f * fabsf(yh - yl);
    const float hd = sqrtf(hx * hx + hy * hy) * 1.0001f + 1.0e-5f;

    const int32_t G = g.nbx * g.nby;
    const int32_t *__restrict__ bs = bucket_start + (size_t)b * (G + 1);
    const float4 *__restrict__ sp = sorted + (size_t)b * N;
    const float margin = 0.01f * g.cell;

    unsigned long long best[K];
#pragma unroll
    for (int k = 0; k < K; ++k) best[k] = ~0ull;

    // ---- reach of the whole patch: anything farther than r + hd from c is irrelevant for every cell -----------------
    const float rcap = q.radius + hd + margin;
    const int32_t bxlo = bucket_coord(pcx - rcap, g.gx0, g.inv_cell, g.nbx), bxhi = bucket_coord(pcx + rcap, g.gx0, g.inv_cell, g.nbx);
    const int32_t bylo = bucket_coord(pcy - rcap, g.gy0, g.inv_cell, g.nby), byhi = bucket_coord(pcy + rcap, g.gy0, g.inv_cell, g.nby);
    const int32_t in_reach = block_count(bs, g.nby, bxlo, bxhi, bylo, byhi, lane);

    if (in_reach > 0) {
        float R = rcap;
        if (in_reach >= K) {
            // ---- U: K-th smallest distance to c inside the first bucket block around c with >= K points ---------------
            const int32_t bcx = bucket_coord(pcx, g.gx0, g.inv_cell, g.nbx), bcy = bucket_coord(pcy, g.gy0, g.inv_cell, g.nby);
            int32_t xa = bcx, xb = bcx, ya = bcy, yb = bcy;
            while (block_count(bs, g.nby, xa, xb, ya, yb, lane) < K) {  // terminates: the reach box holds >= K
                xa = max(xa - 1, bxlo); xb = min(xb + 1, bxhi);
                ya = max(ya - 1, bylo); yb = min(yb + 1, byhi);
            }
            float topk = 3.0e38f;  // lane k < K holds the k-th smallest squared distance to c
            for (int32_t x = xa; x <= xb; ++x) {
                const int32_t s = __ldg(bs + x * g.nby + ya), e = __ldg(bs + x * g.nby + yb + 1);
                for (int32_t base = s; base < e; base += 32) {
                    const int32_t pidx = base + lane;
                    float d2 = 3.0e38f;
                    if (pidx < e) {
                        const float4 pt = __ldg(sp + pidx);
                        const float ddx = pt.x - pcx, ddy = pt.y - pcy;
                        d2 = ddx * ddx + ddy * ddy;
                    }
                    unsigned m = __ballot_sync(0xffffffffu, d2 < __shfl_sync(0xffffffffu, topk, K - 1));
                    while (m) {
                        const int src = __ffs(m) - 1;
                        m &= m - 1;
                        const float v = __shfl_sync(0xffffffffu, d2, src);
                        if (v < __shfl_sync(0xffffffffu, topk, K - 1)) {  // uniform
                            float prev = __shfl_up_sync(0xffffffffu, topk, 1);
                            if (lane == 0) prev = -1.0f;
                            if (lane < K && v < topk) topk = fmaxf(v, prev);
                        }
                    }
                }
            }
            const float U = sqrtf(__shfl_sync(0xffffffffu, topk, K - 1));
            R = fminf((fminf(q.radius, U + hd) + hd) * 1.0001f + 1.0e-4f + margin, rcap);
        }
        // ---- gather { p : |p - c| <= R } in chunks of <= kCandCap and let every lane scan each chunk -----------------
        const float R2 = R * R;
        const int32_t rx0 = bucket_coord(pcx - R, g.gx0, g.inv_cell, g.nbx), rx1 = bucket_coord(pcx + R, g.gx0, g.inv_cell, g.nbx);
        const int32_t ry0 = bucket_coord(pcy - R, g.gy0, g.inv_cell, g.nby), ry1 = bucket_coord(pcy + R, g.gy0, g.inv_cell, g.nby);
        float thr = q.r2;
        int32_t count = 0;
        auto take = [&](int32_t base, int32_t e) {  // 32 sorted points from `base`, kept ones appended to the chunk
            const int32_t pidx = base + lane;
            bool keep = false;
            float4 pt = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pidx < e) {
                pt = __ldg(sp + pidx);
                const float ddx = pt.x - pcx, ddy = pt.y - pcy;
                keep = ddx * ddx + ddy * ddy <= R2;
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) cand[count + __popc(m & ((1u << lane) - 1u))] = pt;
            count += __popc(m);
            if (count > kCandCap - 32) {  // uniform: flush the chunk
                __syncwarp();
                for (int32_t t = 0; t < count; ++t) knn_test<K>(cand[t], cx, cy, q.r2, thr, best);
                __syncwarp();
                count = 0;
            }
        };
        if (kCentreOut) {
            // Order matters for speed, not for the result (the keys are a total order).  Bucket rows are visited from the
            // centre outwards and each row from the centre column outwards, so the K-th distance of every lane tightens
            // early and far candidates fail the pre-filter instead of walking the K-step insertion network (row-major
            // order feeds every cell a monotonically approaching sequence).  Measured: K = 10 at configs[2] 1.315 ->
            // 1.22 ms; K = 5 at configs[1] 0.164 -> 0.170 ms (the short network does not pay for the extra row
            // bookkeeping), hence the switch on K.
            const int32_t xc = min(max(bucket_coord(pcx, g.gx0, g.inv_cell, g.nbx), rx0), rx1);
            const int32_t yc = min(max(bucket_coord(pcy, g.gy0, g.inv_cell, g.nby), ry0), ry1);
            const int32_t span = max(xc - rx0, rx1 - xc);
            for (int32_t d = 0; d <= span; ++d) {
                for (int32_t side = 0; side < (d ? 2 : 1); ++side) {
                    const int32_t x = side ? xc - d : xc + d;
                    if (x < rx0 || x > rx1) continue;
                    const int32_t s = __ldg(bs + x * g.nby + ry0), mid = __ldg(bs + x * g.nby + yc), e = __ldg(bs + x * g.nby + ry1 + 1);
                    for (int32_t base = mid; base < e; base += 32) take(base, e);
                    for (int32_t top = mid; top > s; top -= 32) take(max(top - 32, s), top);
                }
            }
        } else {
            for (int32_t x = rx0; x <= rx1; ++x) {
                const int32_t s = __ldg(bs + x * g.nby + ry0), e = __ldg(bs + x * g.nby + ry1 + 1);
                for (int32_t base = s; base < e; base += 32) take(base, e);
            }
        }
        __syncwarp();
        for (int32_t t = 0; t < count; ++t) knn_test<K>(cand[t], cx, cy, q.r2, thr, best);
    }

    if (active) {
        int32_t *out = knn_idx + ((size_t)b * q.H * q.W + (size_t)i * q.W + j) * K;
#pragma unroll
        for (int k = 0; k < K; ++k) out[k] = best[k] == ~0ull ? -1 : (int32_t)(unsigned)(best[k] & 0xffffffffull);
    }
}

template <int K>
static void launch_knn(const int32_t *bs, const float4 *sp, int32_t B, int32_t N, const BucketGrid &g,
                       const KnnGeom &q, int32_t *out, cudaStream_t st)
{
    // fine scales (patch of 4 x 8 cells small against the radius): warp-per-patch kernel; coarse scales: thread per cell
    const float hx = 0.5f * (kPatchI - 1) * fabsf(q.dx), hy = 0.5f * (kPatchJ - 1) * fabsf(q.dy);
    const bool use_patch = sqrtf(hx * hx + hy * hy) <= 0.75f * q.radius;
    if (use_patch) {
        const int64_t patches = (int64_t)((q.H + kPatchI - 1) / kPatchI) * ((q.W + kPatchJ - 1) / kPatchJ);
        dim3 grid((unsigned)ceil_div64(patches, 4), (unsigned)B);
        k_knn_patch<K><<<grid, 128, 0, st>>>(bs, sp, N, g, q, out);
    } else {
        const int64_t cells = (int64_t)q.H * q.W;
        dim3 grid((unsigned)ceil_div64(cells, 128), (unsigned)B);
        k_knn_query<K><<<grid, 128, 0, st>>>(bs, sp, N, g, q, out);
    }
}

// coarse[b,i,j,:] = fine[b, i*step, j*step, :]
__global__ void __launch_bounds__(256) k_knn_subsample(const int32_t *__restrict__ fine, int32_t Hf, int32_t Wf,
                                                       int32_t step, int32_t *__restrict__ coarse, int32_t Hc, int32_t Wc,
                                                       int32_t K)
{
    const int b = blockIdx.y;
    const int64_t n = (int64_t)Hc * Wc * K;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int32_t k = (int32_t)(t % K);
        const int64_t cell = t / K;
        const int32_t i = (int32_t)(cell / Wc), j = (int32_t)(cell - (int64_t)i * Wc);
        coarse[(size_t)b * n + t] = __ldg(fine + (((size_t)b * Hf + (size_t)i * step) * Wf + (size_t)j * step) * K + k);
    }
}

}  // namespace cf

extern "C" int cf_knn_subsample(const int32_t *d_fine, int32_t B, int32_t Hf, int32_t Wf, int32_t step,
                                int32_t *d_coarse, int32_t Hc, int32_t Wc, int32_t K, void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_fine && d_coarse, CF_ERR_ARG, "cf_knn_subsample: null pointer");
    CF_REQUIRE(B > 0 && B <= 65535 && step >= 1 && K >= 1 && K <= CF_MAX_K && Hc > 0 && Wc > 0, CF_ERR_ARG,
               "cf_knn_subsample: bad extents");
    CF_REQUIRE((int64_t)(Hc - 1) * step < Hf && (int64_t)(Wc - 1) * step < Wf, CF_ERR_ARG,
               "cf_knn_subsample: coarse grid (%d,%d) x step %d does not fit in the fine grid (%d,%d)", Hc, Wc, step, Hf, Wf);
    const int64_t n = (int64_t)Hc * Wc * K;
    const int blocks = (int)std::min<int64_t>(ceil_div64(n, 256), 148 * 8);
    k_knn_subsample<<<dim3(blocks, B), 256, 0, (cudaStream_t)stream>>>(d_fine, Hf, Wf, step, d_coarse, Hc, Wc, K);
    count_launches(1);
    return launch_status("cf_knn_subsample");
}

extern "C" int cf_knn_query(const int32_t *d_bucket_start, const float *d_sorted, int32_t B, int32_t N, float gx0,
                            float gy0, float cell, int32_t nbx, int32_t nby, int32_t H, int32_t W, float x0,
                            float y0, float dx, float dy, float radius, int32_t K, int32_t *d_knn_idx,
                            void *stream)
{
    using namespace cf;
    CF_TRY(require_sm100());
    CF_REQUIRE(d_bucket_start && d_sorted && d_knn_idx, CF_ERR_ARG, "cf_knn_query: null pointer");
    CF_REQUIRE(B > 0 && N > 0 && H > 0 && W > 0 && nbx > 0 && nby > 0 && cell > 0.0f, CF_ERR_ARG,
               "cf_knn_query: bad extents");
    CF_REQUIRE(K >= 1 && K <= CF_MAX_K, CF_ERR_ARG, "cf_knn_query: K=%d outside [1,%d]", K, CF_MAX_K);
    CF_REQUIRE(radius > 0.0f && radius < 1.0e4f, CF_ERR_ARG, "cf_knn_query: radius=%g", (double)radius);
    CF_REQUIRE(aligned16(d_sorted), CF_ERR_ALIGN, "cf_knn_query: d_sorted must be 16-byte aligned");
    CF_REQUIRE(B <= 65535, CF_ERR_ARG, "cf_knn_query: B too large");
    cudaStream_t st = (cudaStream_t)stream;
    BucketGrid g{gx0, gy0, cell, 1.0f / cell, nbx, nby};
    KnnGeom q{x0, y0, dx, dy, radius, radius * radius, H, W};
    const float4 *sp = (const float4 *)d_sorted;
    switch (K) {
#define CF_KNN_CASE(k) \
    case k: launch_knn<k>(d_bucket_start, sp, B, N, g, q, d_knn_idx, st); break;
        CF_KNN_CASE(1) CF_KNN_CASE(2) CF_KNN_CASE(3) CF_KNN_CASE(4) CF_KNN_CASE(5) CF_KNN_CASE(6)
        CF_KNN_CASE(7) CF_KNN_CASE(8) CF_KNN_CASE(9) CF_KNN_CASE(10) CF_KNN_CASE(11) CF_KNN_CASE(12)
        CF_KNN_CASE(13) CF_KNN_CASE(14) CF_KNN_CASE(15) CF_KNN_CASE(16)
#undef CF_KNN_CASE
    }
    count_launches(1);
    return launch_status("cf_knn_query");
}
