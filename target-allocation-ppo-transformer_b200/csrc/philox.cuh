// philox.cuh - Philox4x32-10 (Salmon et al. SC'11), the counter RNG of both libraries: the env's scenes and random
// actions (uavenv_kernels.cuh) and the policy's action samples (policy_forward.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

__device__ __forceinline__ uint4 philox4x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2,
                                            uint32_t c3) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
