// cf_tcgen05.cuh -- thin inline-PTX layer over the Blackwell tensor-core path used by cf_mlp_tc.cu:
// tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM), TMEM alloc / ld / st, mbarrier completion, and the
// shared-memory operand layout.
//
// Operand layout (both A and B are K-major, SWIZZLE_NONE "interleaved" canonical layout):
//   a tile of R rows x KC bf16 columns is stored as core matrices of 8 rows x 8 columns (8 x 16 B = 128 B,
//   rows 16 B apart); core matrix (r/8, k/8) lives at byte ((r/8) * (KC/8) + k/8) * 128.
//   => leading byte offset  LBO (next core matrix along K)   = 128
//      stride  byte offset  SBO (next 8-row group along M/N) = (KC/8) * 128
//   A thread that owns row r writes 16-byte units at +(r%8)*16: the 8 rows of a group fill 128 contiguous
//   bytes, so a warp's 32 unit stores take the minimum 4 shared-memory wavefronts (no bank conflicts).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace cf {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory matrix descriptor (SWIZZLE_NONE, K-major) --------------------------------------------
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);        // bits [ 0,14) start address >> 4
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;  // bits [16,30) leading byte offset >> 4
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;  // bits [32,46) stride byte offset >> 4
    d |= (uint64_t)1 << 46;                             // bits [46,48) descriptor version = 1 (sm_100)
    return d;                                           // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}

// ---- instruction descriptor: D fp32, A/B bf16, both K-major, M x N ---------------------------------------
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N)
{
    return (1u << 4)                      // c_format  = F32
           | (1u << 7)                    // a_format  = BF16
           | (1u << 10)                   // b_format  = BF16
           | ((uint32_t)(N >> 3) << 17)   // n_dim
           | ((uint32_t)(M >> 4) << 24);  // m_dim
}

__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// One lane of a CONVERGED warp (all 32 lanes must execute this).  Guarding the tcgen05.mma / commit sequence with
// `warp == w && elect_one()` instead of `tid == 0` lets ptxas keep descriptors in uniform registers and emit the UTCHMMAs
// back to back; under a plain thread-index test it wraps every UTCHMMA in an ELECT / BRA.U.ANY loop (~70 cycles per MMA,
// measured: 15 % of the tile time of a since-removed segment-tile variant of K-4 went into issuing 35 small MMAs).
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// all previously issued tcgen05 async ops of this thread arrive (count 1) on the mbarrier when complete
__device__ __forceinline__ void commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- mbarrier ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}

// ---- TMA (cp.async.bulk, cp.async.bulk.tensor), completion on an mbarrier / bulk groups ---------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar_addr, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint32_t bar_addr, uint32_t parity)
{
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(bar_addr), "r"(parity)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity)
{
    while (!mbar_test(bar_addr, parity)) {
    }
}
__device__ __forceinline__ void tma_store_3d(const void *tmap, int32_t x, int32_t y, int32_t z, uint32_t src)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(tmap), "r"(x), "r"(y), "r"(z), "r"(src)
                 : "memory");
}
// 1-D bulk copy global -> shared (TMA engine, SASS UBLKCP): `bytes` a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar_addr)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar_addr)
                 : "memory");
}
// L2 prefetch of a contiguous global range by the TMA engine (no destination in the SM): `bytes` a multiple of 16, 16-byte aligned
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- TMEM ---------------------------------------------------------------------------------------------------
// one full warp; writes the base address to *dst (shared memory).  ncols: power of two in [32, 512]
__device__ __forceinline__ void tmem_alloc(uint32_t *dst, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t addr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of warp w receives lane 32*(w%4)+t
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
        "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
        "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
        "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

template <int EW> __device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[EW]);
template <> __device__ __forceinline__ void tmem_ld<32>(uint32_t taddr, float (&v)[32]) { tmem_ld32(taddr, v); }
template <> __device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, float (&v)[16]) { tmem_ld16(taddr, v); }
template <int EW> __device__ __forceinline__ void tmem_st(uint32_t taddr, const float (&v)[EW]);
template <> __device__ __forceinline__ void tmem_st<32>(uint32_t taddr, const float (&v)[32]) { tmem_st32(taddr, v); }
template <> __device__ __forceinline__ void tmem_st<16>(uint32_t taddr, const float (&v)[16]) { tmem_st16(taddr, v); }

// ---- operand packing -------------------------------------------------------------------------------------------
// byte offset of the 16-byte unit (row r, k-unit ku) inside an R x KC tile (KC/8 units per row)
__device__ __forceinline__ uint32_t unit_offset(int r, int ku, int kc_units)
{
    return (uint32_t)(((r >> 3) * kc_units + ku) * 128 + (r & 7) * 16);
}

// split 8 fp32 into bf16 "hi" (round to nearest) and bf16 "lo" (the rounded residual): hi + lo carries ~16
// mantissa bits, so hi*hi + hi*lo + lo*hi reproduces an fp32 product to ~2^-16 relative.
// cvt.rn.bf16x2.f32 converts a pair per instruction; the bf16 -> fp32 widening is a shift / mask.
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b)
{
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);  // .x = a (low half), .y = b (high half)
    return *reinterpret_cast<const uint32_t *>(&h);
}

__device__ __forceinline__ void split_bf16x8(const float (&v)[8], uint4 &hi, uint4 &lo, bool want_lo)
{
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        h[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
        if (want_lo) {
            const float a_hi = __uint_as_float(h[i] << 16), b_hi = __uint_as_float(h[i] & 0xFFFF0000u);
            l[i] = pack_bf16x2(v[2 * i] - a_hi, v[2 * i + 1] - b_hi);
        } else {
            l[i] = 0;
        }
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}


// 256-bit read-only global load (sm_100: LDG.E.256), 32-byte aligned
__device__ __forceinline__ void ldg_nc_f32x8(const float *p, float *v)
{
    asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
        : "l"(p));
}

// 8 consecutive channels of a layer-1 table row as fp32: fp32 tables (one 256-bit load) or bf16 tables (one 128-bit load,
// bf16 -> fp32 is a shift)
__device__ __forceinline__ void ldg_row8(const float *p, float *v) { ldg_nc_f32x8(p, v); }
__device__ __forceinline__ void ldg_row8(const __nv_bfloat16 *p, float *v)
{
    uint32_t r[4];
    asm("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = __uint_as_float(r[i] << 16);
        v[2 * i + 1] = __uint_as_float(r[i] & 0xffff0000u);
    }
}

// 256-bit global store (sm_100: STG.E.256): a full 32-byte sector per lane, 32-byte aligned
__device__ __forceinline__ void stg_f32x8(float *p, const float *v)
{
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// ---- explicit shared-state-space accesses (32-bit addresses: no generic-pointer conversion in the inner loops) -----
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_f32x2(uint32_t addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u32x4(uint32_t addr, const uint4 &v)
{
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// Ampere-style asynchronous 4-byte copy global -> shared (no register staging); completion via commit / wait_all
__device__ __forceinline__ void cp_async4(uint32_t dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- packed fp32 pairs (sm_100: FFMA2 / FADD2 process two fp32 lanes per issue slot) -----------------------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c)
{
    float2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(reinterpret_cast<unsigned long long &>(d))
        : "l"(reinterpret_cast<const unsigned long long &>(a)), "l"(reinterpret_cast<const unsigned long long &>(b)),
          "l"(reinterpret_cast<const unsigned long long &>(c)));
    return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b)
{
    float2 d;
    asm("mul.rn.f32x2 %0, %1, %2;"
        : "=l"(reinterpret_cast<unsigned long long &>(d))
        : "l"(reinterpret_cast<const unsigned long long &>(a)), "l"(reinterpret_cast<const unsigned long long &>(b)));
    return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)
{
    float2 d;
    asm("add.rn.f32x2 %0, %1, %2;"
        : "=l"(reinterpret_cast<unsigned long long &>(d))
        : "l"(reinterpret_cast<const unsigned long long &>(a)), "l"(reinterpret_cast<const unsigned long long &>(b)));
    return d;
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b)
{
    float2 d;
    asm("sub.rn.f32x2 %0, %1, %2;"
        : "=l"(reinterpret_cast<unsigned long long &>(d))
        : "l"(reinterpret_cast<const unsigned long long &>(a)), "l"(reinterpret_cast<const unsigned long long &>(b)));
    return d;
}

// ReLU fused into the bf16 split of a NON-NEGATIVE-after-ReLU operand (activations):
//   hi = bf16_rz(relu(v))              one F2FP.RELU.RZ per pair; truncation keeps hi <= v, so for v >= 0 the residual
//   lo = bf16_rn(relu(v - float(hi)))  is >= 0, and for v < 0 (hi = 0) the residual v < 0 is clamped to 0 by the same
//                                      .relu: no FMNMX, no select.  |relu(v) - hi - lo| < 2^-16 |v|.
// a = element 0 (low half of the result), b = element 1 (high half).
__device__ __forceinline__ uint32_t cvt_relu_rz_bf16x2(float a, float b)
{
    uint32_t d;
    asm("cvt.rz.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ uint32_t cvt_relu_rn_bf16x2(float a, float b)
{
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ void relu_split_bf16x8(const float2 (&v)[4], uint4 &hi, uint4 &lo, bool want_lo)
{
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (want_lo) {
            h[i] = cvt_relu_rz_bf16x2(v[i].x, v[i].y);
            const float2 hf = make_float2(__uint_as_float(h[i] << 16), __uint_as_float(h[i] & 0xFFFF0000u));
            const float2 r = fsub2(v[i], hf);
            l[i] = cvt_relu_rn_bf16x2(r.x, r.y);
        } else {
            h[i] = cvt_relu_rn_bf16x2(v[i].x, v[i].y);
            l[i] = 0;
        }
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// two 32-lane x 16-column TMEM loads in flight, one wait
__device__ __forceinline__ void tmem_ld16x2(uint32_t ta, uint32_t tb, float (&a)[16], float (&b)[16])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%32];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%33];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(ta), "r"(tb)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        a[i] = __uint_as_float(r[i]);
        b[i] = __uint_as_float(r[16 + i]);
    }
}

}  // namespace tc
}  // namespace cf
