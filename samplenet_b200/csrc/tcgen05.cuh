// tcgen05.cuh -- the 5th-generation tensor-core (tcgen05) wrappers shared by the per-layer kernel (encoder_tc.cu) and the persistent
// conv-stack kernel (conv_stack.cu).  The encodings are validated against fp64 in tests/test_gpu_parity.py::test_tc_gemm_3xtf32.
#pragma once
#include "common.cuh"

namespace snb {

// ---- tensor-memory allocation (one warp) and ordering around thread synchronisation
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- MMA issue (one thread) and completion
// A from shared memory: D[tmem] (+)= A[smem descriptor] . B[smem descriptor]
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A from tensor memory: D[tmem] (+)= A[tmem, 128 lanes x 8 columns] . B[smem descriptor]
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier when every MMA this thread issued so far has completed
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- tensor memory <-> registers, 32x32b shape: thread t of the warp gets lane (lane base + t), one column per register
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// columns taddr .. taddr+7; the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t *r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
// columns taddr .. taddr+31, waited for
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v)
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr)
        : "memory");
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
// columns taddr .. taddr+7; the store is complete after tmem_st_wait()
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// ---- descriptors
// Instruction descriptor, kind::tf32, fp32 accumulate, A and B K-major (cute/arch/mma_sm100_desc.hpp InstrDescriptor):
//   [4,6) c_format = 1 (F32) | [7,10) a_format = 2 (TF32) | [10,13) b_format = 2 | bit 15/16 a/b major = 0 (K) |
//   [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// Shared-memory matrix descriptor, K-major SWIZZLE_128B (SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) = 1 |
// SBO>>4 [32,46) = 64 (8 rows x 128 B) | version [46,48) = 1 | layout_type [61,64) = 2
constexpr unsigned kDescHiSw128 = (64u) | (1u << 14) | (2u << 29);  // bits [32,64) of the descriptor
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr, unsigned desc_hi)
{
    return (uint64_t)((smem_addr >> 4) & 0x3fffu) | (1ull << 16) | ((uint64_t)desc_hi << 32);
}

}  // namespace snb
