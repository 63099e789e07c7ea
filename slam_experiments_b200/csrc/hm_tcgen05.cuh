// Thin inline-PTX wrappers for the sm_100a features the tensor-core variant uses:
// mbarrier, 1-D bulk async copy (UBLKCP), TMEM allocation, tcgen05.mma kind::i8 / kind::mxf4,
// tcgen05.commit, tcgen05.ld.  No CUTLASS: the bit layouts of the shared-memory
// matrix descriptor and the instruction descriptor are spelled out here.
#pragma once

#include <stdint.h>

namespace hm {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one()
{
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xFFFFFFFF;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// non-blocking probe (never suspends the thread)
// the same on a precomputed shared-memory address
__device__ __forceinline__ bool mbar_try_wait_addr(uint32_t bar_addr, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar_addr), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_arrive_addr(uint32_t bar_addr)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar_addr) : "memory");
}
// A shared-memory word read back through a volatile load: the value is opaque to ptxas, so addresses derived from it
// stay in a register instead of being recomputed (S2R + address arithmetic) inside a hot loop.
__device__ __forceinline__ uint32_t lds_volatile_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---- bulk async copy global -> shared (completes on an mbarrier) ----------------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// same, delivered to the same CTA-relative offset (data and mbarrier signal) of every CTA in cta_mask
__device__ __forceinline__ void bulk_g2s_multicast(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                                   uint64_t* bar, uint16_t cta_mask)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;\n" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}

// ---- thread-block cluster ------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync()   // all threads of all CTAs of the cluster
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

// ---- tensor memory ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols)   // whole warp
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_dst)),
                 "r"(cols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish()
{
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)     // whole warp
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// all previously issued tcgen05.mma of this thread arrive on `bar` when complete
__device__ __forceinline__ void tc_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
                 : "memory");
}

// same, arriving on the barrier at this CTA-relative offset in every CTA of cta_mask
__device__ __forceinline__ void tc_commit_multicast(uint64_t* bar, uint16_t cta_mask)
{
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
            smem_u32(bar)),
        "h"(cta_mask)
        : "memory");
}

// D[tmem] (+)= A[smem] * B[smem], int8 x int8 -> int32, issued by ONE thread
__device__ __forceinline__ void mma_i8_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D[tmem] (+)= A[smem] * B[smem], block-scaled e2m1 x e2m1 -> fp32 (K = 64 per instruction, one ue8m0
// scale per 32 elements, read from TMEM at tmem_sfa / tmem_sfb), issued by ONE thread
__device__ __forceinline__ void mma_mxf4_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t tmem_sfa, uint32_t tmem_sfb, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(tmem_sfa), "r"(tmem_sfb)
        : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns, registers -> TMEM (scale-factor fill)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns: thread `lane` gets columns [col, col+32) of its TMEM lane
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
          "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// 32 lanes x 64 consecutive 32-bit columns in ONE instruction (the two x32 halves cannot be separated
// by the scheduler, so the accumulator unit is released as early as possible)
__device__ __forceinline__ void tmem_ld_32x64(uint32_t taddr, uint32_t (&r)[64])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr)
        : "memory");
}

// ---- descriptors ----------------------------------------------------------------------------
// Shared-memory matrix descriptor, K-major operand stored as rows of 128 bytes with the
// 128-byte swizzle (16-byte chunk index XOR (row % 8)), 8-row groups 1024 bytes apart:
//   [ 0,14) start address >> 4      [16,30) leading byte offset >> 4 (unused: one atom along K)
//   [32,46) stride byte offset >> 4 = 1024 >> 4   [46,48) version = 1 (sm_100)
//   [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// The same descriptor from its start-address field (smem_addr >> 4, fits 14 bits for any shared-memory
// address): advancing the operand by `bytes` is `lo + (bytes >> 4)` -- one add, no shift / mask per MMA.
constexpr uint32_t kKmajorSw128DescHi = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t kmajor_sw128_desc_from_lo(uint32_t lo)
{
    return ((uint64_t)kKmajorSw128DescHi << 32) | lo;
}

// Instruction descriptor for kind::i8, dense, no saturate:
//   [4,6) D format = 2 (S32)   [7,10) A format = 1 (signed 8-bit)   [10,13) B format = 1
//   bit 15 / 16: A / B major = 0 (K-major)   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_i8_idesc(int m, int n)
{
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// Instruction descriptor for kind::mxf4 (block-scaled), dense, K = 64:
//   [4,6) B scale-factor id = 0   [7,10) A format = 1 (e2m1)   [10,13) B format = 1   bit 15 / 16: K-major
//   [17,23) N >> 3   bit 23 scale format = 1 (ue8m0)   [24,29) M >> 4   [29,31) A scale-factor id = 0
__host__ __device__ constexpr uint32_t make_mxf4_idesc(int m, int n)
{
    return (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | (1u << 23) | ((uint32_t)(m >> 4) << 24);
}

}  // namespace ptx
}  // namespace hm
