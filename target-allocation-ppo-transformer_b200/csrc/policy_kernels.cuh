// policy_kernels.cuh - device helpers that more than one translation unit of the policy library uses: bf16 pack /
// unpack, xor-shuffle sums and the second head layers (head_out).  It holds no kernel: every kernel is defined in the
// file that launches it.  Internal linkage.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "policy_weights.cuh"

namespace {
using namespace uavp;

// ---- bf16 <-> fp32: 4 values (8 B), 8 values (16 B), 16 values (32 B) -----------------------------------------------
__device__ __forceinline__ void unpack4f(const uint2 w, float *o) {
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162 *>(&w.x), b = *reinterpret_cast<const __nv_bfloat162 *>(&w.y);
    o[0] = __low2float(a); o[1] = __high2float(a); o[2] = __low2float(b); o[3] = __high2float(b);
}
__device__ __forceinline__ uint2 pack4f(const float *v) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 w;
    w.x = *reinterpret_cast<const uint32_t *>(&a); w.y = *reinterpret_cast<const uint32_t *>(&b);
    return w;
}
__device__ __forceinline__ void unpack8(const uint4 &q, float *o) {   // bf16 -> fp32 is a 16-bit shift
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        o[2 * i] = __uint_as_float(w[i] << 16); o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ uint4 pack8(const float *v) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t *>(&t);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void load16(const __nv_bfloat16 *p, float *out) {
    const uint4 a = reinterpret_cast<const uint4 *>(p)[0], b = reinterpret_cast<const uint4 *>(p)[1];
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162 *>(&w[i]);
        out[2 * i] = __low2float(v); out[2 * i + 1] = __high2float(v);
    }
}
__device__ __forceinline__ void store16(__nv_bfloat16 *p, const float *v) {
    reinterpret_cast<uint4 *>(p)[0] = pack8(v);
    reinterpret_cast<uint4 *>(p)[1] = pack8(v + 8);
}

// sum of v over the lanes reached by the given xor offsets, exchanged in the order given: xor_sum<16, 8, 4, 2, 1> is a
// whole warp.  The order fixes the grouping of the fp32 additions, so a reduction keeps its offsets where results have
// to stay bit-identical.
template <int... kOffsets>
__device__ __forceinline__ float xor_sum(float v) {
    ((v += __shfl_xor_sync(0xffffffffu, v, kOffsets)), ...);
    return v;
}

// second head layers (transformer_net.py:78-91; the first layers 128 -> 64 + ReLU ran before) of sample b = the thread's
// index in the grid: logits (l0, l1) = W2a ha + b2a from the bf16 hidden row Ha[b], and with kValue also the value
// v = W2c hc + b2c from Hc[b].  The CTA stages W2 in shared memory first, so every thread calls this; it returns false
// for the threads past B.
template <bool kValue>
__device__ __forceinline__ bool head_out(const __nv_bfloat16 *Ha, const __nv_bfloat16 *Hc, const float *w2a, const float *b2a,
                                         const float *w2c, const float *b2c, int B, int &b, float &l0, float &l1, float &v) {
    __shared__ float s_w[kValue ? 3 : 2][HID];
    for (int i = threadIdx.x; i < HID; i += blockDim.x) {
        s_w[0][i] = w2a[i]; s_w[1][i] = w2a[HID + i];
        if constexpr (kValue) s_w[2][i] = w2c[i];
    }
    __syncthreads();
    b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return false;
    l0 = b2a[0]; l1 = b2a[1];
    if constexpr (kValue) v = b2c[0];
#pragma unroll
    for (int c = 0; c < HID / DH; ++c) {
        float xa[DH], xc[DH];
        load16(Ha + (size_t)b * HID + c * DH, xa);
        if constexpr (kValue) load16(Hc + (size_t)b * HID + c * DH, xc);
#pragma unroll
        for (int e = 0; e < DH; ++e) {
            l0 = fmaf(s_w[0][c * DH + e], xa[e], l0);
            l1 = fmaf(s_w[1][c * DH + e], xa[e], l1);
            if constexpr (kValue) v = fmaf(s_w[2][c * DH + e], xc[e], v);
        }
    }
    return true;
}

}  // namespace
