// tc_common.cuh — thin inline-PTX wrappers for the sm_100a tensor-core path (tcgen05 + TMEM + mbarrier +
// bulk async copy) and the canonical shared-memory operand layout used by the policy kernel.
//
// Operand layout (K-major, no swizzle — UMMA "INTERLEAVE"): an operand tile of R rows x K fp32 is stored as
// 8-row x 16-byte core matrices (128 contiguous bytes each):
//     byte(r, k) = (r / 8) * SBO + (k / 4) * LBO + (r % 8) * 16 + (k % 4) * 4,   LBO = 128, SBO = (K / 4) * 128
// i.e. the K/4 core matrices of an 8-row group are contiguous.  One tcgen05.mma.kind::tf32 consumes K = 8
// (two 16-byte chunks: LBO apart); the next one starts 2*LBO = 256 bytes further.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cm {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of element (r, k) inside a canonical operand tile with K columns
__device__ __forceinline__ uint32_t canon_off(int r, int k, int K)
{
    return (uint32_t)((r >> 3) * (K >> 2) * 128 + (k >> 2) * 128 + (r & 7) * 16 + (k & 3) * 4);
}

// 64-bit shared-memory matrix descriptor (SM100 UMMA): start address, LBO, SBO (all >> 4), version = 1,
// no swizzle.  kchunk selects the K = 8 slice (advances the start address by 256 bytes).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, int K, int kslice)
{
    const uint32_t start = smem_addr + (uint32_t)kslice * 256u;
    uint64_t d = 0;
    d |= (uint64_t)((start & 0x3FFFFu) >> 4);              // bits [0,14)
    d |= (uint64_t)(128u >> 4) << 16;                      // leading byte offset, bits [16,30)
    d |= (uint64_t)(((uint32_t)(K >> 2) * 128u) >> 4) << 32;  // stride byte offset, bits [32,46)
    d |= (uint64_t)1 << 46;                                // descriptor version (Blackwell)
    return d;
}

// ---- 16-bit operands (kind::f16): core matrix = 8 rows x 16 bytes = 8 elements; one MMA consumes K = 16 ----
__device__ __forceinline__ uint32_t canon_off16(int r, int k, int K)
{
    return (uint32_t)((r >> 3) * (K >> 3) * 128 + (k >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2);
}
__device__ __forceinline__ uint64_t make_smem_desc16(uint32_t smem_addr, int K, int kslice)
{
    const uint32_t start = smem_addr + (uint32_t)kslice * 256u;
    uint64_t d = 0;
    d |= (uint64_t)((start & 0x3FFFFu) >> 4);
    d |= (uint64_t)(128u >> 4) << 16;
    d |= (uint64_t)(((uint32_t)(K >> 3) * 128u) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// MN-major operand (memory [K][M or N], the M / N index contiguous) without swizzle, stored in the same chunked form as a
// K-major tile of `cols` columns written row by row:  byte(k, m) = (k / 8) * (cols / 8) * 128 + (m / 8) * 128 + (k % 8) * 16 + (m % 8) * 2.
// Measured on B200 (tests/native/mn_probe.cu): for an MN-major operand LBO is the stride between groups of 8 K rows and SBO
// the stride between 16-byte chunks (8 elements) along M / N; an instruction of K = 16 consumes two K groups.
__device__ __forceinline__ uint64_t make_smem_desc16_mn(uint32_t smem_addr, int cols)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(((uint32_t)(cols >> 3) * 128u) >> 4) << 16;   // LBO: next group of 8 K rows
    d |= (uint64_t)(128u >> 4) << 32;                             // SBO: next 8 elements along M / N
    d |= (uint64_t)1 << 46;
    return d;
}
static constexpr uint32_t kIdescAMajorMN = 1u << 15, kIdescBMajorMN = 1u << 16;   // instruction descriptor: operand is MN-major
// kind::f16 with fp16 operands (format 0), fp32 accumulate
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N)
{
    return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// The same instruction predicated on `leader` (1 in exactly one lane of a converged warp, 0 elsewhere).  Every lane
// runs the surrounding code, so descriptors and addresses stay in uniform registers and the issue loop has no
// elect / branch / reconvergence per instruction: measured 57-64 cycles per instruction (N = 64 / 128; the tensor
// floor at N = 128 is 64) against ~90 for a single-thread loop and ~190 for elect.sync around every instruction.
__device__ __forceinline__ void mma_f16_pred(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate,
                                             uint32_t leader)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
// D = A B + D 2^-12 (scale-input-d, an immediate of kind::f16 / kind::tf32): the accumulator that holds the low-order cross
// terms — computed with the remainders scaled by 2^12 — takes the high-order product on top, so hi*hi + 2^-12 (hi*lo + lo*hi)
// needs ONE accumulator block instead of two.  The scaling by a power of two is exact.
__device__ __forceinline__ void mma_f16_scale12_pred(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t leader)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "setp.ne.b32 q, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 12;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void mma_commit_pred(uint64_t *bar, uint32_t leader)
{
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}\n" ::"r"(smem_u32(bar)), "r"(leader)
        : "memory");
}

// 32-bit instruction descriptor, kind::tf32, fp32 accumulate, A and B K-major, M x N tile
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst, uint32_t ncols)   // one full warp
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols)       // the same warp
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void fence_before_thread_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_thread_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tensor core / bulk copies)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// one lane of a converged warp (warp-uniform code keeps descriptors in uniform registers; the elected lane issues)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void mma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// bounded wait (never hangs the GPU): returns false when the phase did not complete within `spins` polls
__device__ __forceinline__ bool mbar_wait(uint64_t *bar, uint32_t parity, uint32_t spins = 1u << 22)
{
    const uint32_t addr = smem_u32(bar);
#pragma unroll 1
    for (uint32_t i = 0; i < spins; ++i) {
        uint32_t ok;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
        if (ok) return true;
    }
    return false;
}

// 1-D bulk async copy global -> shared, completion counted in bytes on an mbarrier (TMA engine, no tensor map)
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 8 consecutive fp32 columns starting at column `col`
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8])
{
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// TMEM -> registers for an M = 64 accumulator, whose rows sit in lanes 0..15 of each lane quadrant: the 16 lanes from `taddr`
// (the lane field of taddr selects them) x 32 consecutive columns, split between the two half-warps so that every thread
// carries data — thread t holds lane t % 16, columns col + 16 (t / 16) .. + 15 (shape 16x32bx2, half split offset 16)
__device__ __forceinline__ void tmem_ld16x32(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.16x32bx2.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16], 16;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM: this warp's 32 lanes x NC (1, 2, 4 or 8) consecutive fp32 columns starting at column `col`.
// Tensor memory doubles as a per-row scratch pad: a lane (= tile row) is private to the row, and every warp of the
// row's lane quadrant can read it back, so row-private exchanges between those warps need no shared memory.
template <int NC>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const float *v)
{
    static_assert(NC == 1 || NC == 2 || NC == 4 || NC == 8, "tmem_st width");
    if constexpr (NC == 1)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(__float_as_uint(v[0])) : "memory");
    else if constexpr (NC == 2)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                     "r"(__float_as_uint(v[1]))
                     : "memory");
    else if constexpr (NC == 4)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                     "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3]))
                     : "memory");
    else
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                     "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                     "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                     : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Error-compensated TF32 split: hi = x rounded to nearest TF32 (low 13 bits zero), lo = the exact remainder
// x - hi, itself rounded to nearest TF32.  Rounding to NEAREST (cvt.rna) instead of letting the tensor core
// truncate keeps the representation errors unbiased, so they accumulate like a random walk over K instead of
// coherently.
__device__ __forceinline__ float tf32_rna(float a)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(a));
    return __uint_as_float(r);
}
__device__ __forceinline__ float tf32_hi(float a) { return tf32_rna(a); }
__device__ __forceinline__ float tf32_lo(float a, float hi) { return tf32_rna(a - hi); }

}  // namespace tc
}  // namespace cm
