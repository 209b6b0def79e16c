// tcgen05_util.cuh - hand-written sm_100a building blocks for the fused policy kernels: shared-memory operand
// layout + UMMA descriptors, tcgen05.mma issue / commit, TMEM allocation and loads, mbarrier waits.
//
// Operand layout (K-major, no swizzle - "interleaved" canonical layout of the UMMA shared-memory descriptor):
// a [rows x K] bf16 tile is stored as 8x8 "core matrices" of 128 contiguous bytes (8 rows x 16 B); core matrices that
// are adjacent along K are contiguous (LBO = 128 B) and 8-row groups are SBO = K/8 * 128 B apart:
//     offset(r, k) = (r / 8) * (K * 16) + (k / 8) * 128 + (r % 8) * 16 + (k % 8) * 2      [bytes]
// One tcgen05.mma.kind::f16 consumes K = 16 (two core matrices along K); k-step j starts at +j * 256 B.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of element (r, k) of a K-major canonical tile with row length K (elements)
__device__ __forceinline__ uint32_t canon_off(int r, int k, int K) {
    return (uint32_t)((r >> 3) * (K * 16) + (k >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2);
}

// UMMA shared-memory descriptor (cute/arch/mma_sm100_desc.hpp: SmemDescriptor): start address, leading (K) and
// stride (M/N) byte offsets in 16 B units, version 1 (Blackwell), no swizzle
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// the same for a 128-byte-swizzled tile (what a TMA tensor load with CU_TENSOR_MAP_SWIZZLE_128B writes): layout type 2
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return smem_desc(saddr, lbo_bytes, sbo_bytes) | ((uint64_t)2 << 61);
}

// UMMA instruction descriptor for kind::f16 (InstrDescriptor): D = f32, A = B = bf16, both K-major, M x N
__host__ __device__ constexpr uint32_t instr_desc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// the same with both operands MN-major (bits 15 / 16): the contraction runs over the ROWS of the shared-memory tiles.
// A K-major canonical tile [rows x W] read this way is an MN-major operand with MN = the W columns and K = the rows:
// its core matrices (8 rows x 16 B) are the same, only the roles of the two strides swap - the 8-column groups
// (128 B apart) become the stride dimension (SBO) and the 8-row groups (W * 16 B apart) the leading dimension (LBO).
__host__ __device__ constexpr uint32_t instr_desc_bf16_mn(int M, int N) { return instr_desc_bf16(M, N) | (1u << 15) | (1u << 16); }

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// all MMAs issued so far by this thread arrive on the mbarrier when they have completed
__device__ __forceinline__ void mma_commit(uint64_t *mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(mbar)) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t *mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *mbar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smem_u32(mbar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// TMEM: 512 columns x 128 lanes x 32 bit per SM.  One warp allocates / frees; the address lands in shared memory.
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_result, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_result)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(cols) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane (lane = 32 * (warp % 4) + laneid): v[0..31]
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 1-D bulk TMA copy global -> shared (UBLKCP) of `bytes` (multiple of 16, both sides 16 B aligned); completion is
// signalled on the mbarrier as a transaction count.  Issued by ONE thread, which also posts the expected bytes.
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *mbar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(mbar)) : "memory");
}

// the copy alone (the caller has posted the bytes of all the copies of this phase with ONE mbar_expect_tx)
__device__ __forceinline__ void bulk_copy(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(mbar)) : "memory");
}

// 2-D TMA tensor load (UTMALDG) of one box at element coordinates (c0 = innermost, c1) of the tensor map; completion is
// signalled on the mbarrier as a transaction count (post the expected bytes with mbar_expect_tx first).  ONE thread.
__device__ __forceinline__ void mbar_expect_tx(uint64_t *mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const void *tensor_map, int c0, int c1, uint64_t *mbar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
                     smem_u32(smem_dst)), "l"(tensor_map), "r"(c0), "r"(c1), "r"(smem_u32(mbar)) : "memory");
}

// cooperative copy of a row-major bf16 matrix [rows x K] (global, row stride ld elements) into a canonical tile; rows >=
// valid_rows are zero-filled (self-test / ragged activations)
__device__ __forceinline__ void load_canon(unsigned char *smem_tile, const __nv_bfloat16 *g, int rows, int K, int64_t ld,
                                           int valid_rows, int tid, int nthreads) {
    const int chunks_per_row = K >> 3;              // 16 B chunks
    for (int i = tid; i < rows * chunks_per_row; i += nthreads) {
        const int r = i / chunks_per_row, c = i % chunks_per_row;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (r < valid_rows) v = *reinterpret_cast<const uint4 *>(g + (int64_t)r * ld + c * 8);
        *reinterpret_cast<uint4 *>(smem_tile + canon_off(r, c * 8, K)) = v;
    }
}

}  // namespace tc
