// ppo_attn.cu - fused multi-head self-attention over the 5-token observation window, forward and backward, for the
// PPO update (agents/ppo.py:126 -> networks/transformer_net.py:63: nn.TransformerEncoderLayer self-attention with a
// key-padding mask; 8 heads x 16 dims).  The library path spends two thirds of an update in batched 5x16x5 matrix
// products, softmax and mask kernels; here one thread owns one (sample, head, token): scores, masked softmax and the
// weighted sum - or, backward, the softmax Jacobian and all three gradients - stay in registers.  fp32 throughout.
// NQ = 5: every token is a query (inner encoder layers).  NQ = 1: only the newest token is (last layer).
#include "uavenv_b200.h"

#include <cstdint>
#include <cuda_runtime.h>

#include "handle.cuh"

namespace {
constexpr int S = 5, H = 8, DH = 16;

struct AttnArgs {
    const float *q, *k, *v;        // q: [n, NQ, H*DH] rows of stride q_stride; k, v: [n, S, H*DH] rows of stride kv_stride
    int64_t q_stride, kv_stride;
    const uint8_t *pad;            // [n, S] 1 = key is padding
    int64_t n;
};

__device__ __forceinline__ void load16(const float *p, float *o) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 t = reinterpret_cast<const float4 *>(p)[i];
        o[4 * i] = t.x; o[4 * i + 1] = t.y; o[4 * i + 2] = t.z; o[4 * i + 3] = t.w;
    }
}
__device__ __forceinline__ void store16(float *p, const float *o) {
#pragma unroll
    for (int i = 0; i < 4; ++i) reinterpret_cast<float4 *>(p)[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
}

// probabilities of query row `qrow` (already loaded) over the 5 keys of (sample b, head h)
__device__ __forceinline__ void softmax_row(const AttnArgs &a, int64_t b, int h, const float *q, float *p) {
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float kk[DH], s = 0.0f;
        load16(a.k + (b * S + j) * a.kv_stride + h * DH, kk);
#pragma unroll
        for (int e = 0; e < DH; ++e) s = fmaf(q[e], kk[e], s);
        p[j] = a.pad[b * S + j] ? -INFINITY : s * 0.25f;      // 1/sqrt(16)
        mx = fmaxf(mx, p[j]);
    }
    float den = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) { p[j] = expf(p[j] - mx); den += p[j]; }
    const float inv = 1.0f / den;
#pragma unroll
    for (int j = 0; j < S; ++j) p[j] *= inv;
}

template <int NQ>
__global__ void __launch_bounds__(256) attn5_forward_kernel(AttnArgs a, float *__restrict__ out /* [n, NQ, H*DH] dense */) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.n * H * NQ) return;
    const int64_t b = idx / (H * NQ);
    const int h = (int)((idx / NQ) % H), i = (int)(idx % NQ);
    float q[DH], p[S], o[DH];
    load16(a.q + (b * NQ + i) * a.q_stride + h * DH, q);
    softmax_row(a, b, h, q, p);
#pragma unroll
    for (int e = 0; e < DH; ++e) o[e] = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float vv[DH];
        load16(a.v + (b * S + j) * a.kv_stride + h * DH, vv);
#pragma unroll
        for (int e = 0; e < DH; ++e) o[e] = fmaf(p[j], vv[e], o[e]);
    }
    store16(out + (b * NQ + i) * (H * DH) + h * DH, o);
}

// thread (sample, head, token t): gradient of key / value t, and of query t when t < NQ
template <int NQ>
__global__ void __launch_bounds__(256) attn5_backward_kernel(AttnArgs a, const float *__restrict__ gout /* [n,NQ,128] dense */,
                                                             float *__restrict__ gq, float *__restrict__ gk, float *__restrict__ gv) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.n * H * S) return;
    const int64_t b = idx / (H * S);
    const int h = (int)((idx / S) % H), t = (int)(idx % S);
    float dk[DH], dv[DH], dq[DH];
#pragma unroll
    for (int e = 0; e < DH; ++e) { dk[e] = 0.0f; dv[e] = 0.0f; dq[e] = 0.0f; }
#pragma unroll 1
    for (int i = 0; i < NQ; ++i) {
        float q[DH], go[DH], p[S], dp[S];
        load16(a.q + (b * NQ + i) * a.q_stride + h * DH, q);
        load16(gout + (b * NQ + i) * (H * DH) + h * DH, go);
        softmax_row(a, b, h, q, p);
        float dot = 0.0f;                                   // sum_j p_ij * dP_ij
#pragma unroll
        for (int j = 0; j < S; ++j) {
            float vv[DH], s = 0.0f;
            load16(a.v + (b * S + j) * a.kv_stride + h * DH, vv);
#pragma unroll
            for (int e = 0; e < DH; ++e) s = fmaf(go[e], vv[e], s);
            dp[j] = s;
            dot = fmaf(p[j], s, dot);
        }
        const float ds_t = p[t] * (dp[t] - dot) * 0.25f;     // dL/d(score_it) incl. the 1/sqrt(dh) scale
#pragma unroll
        for (int e = 0; e < DH; ++e) { dk[e] = fmaf(ds_t, q[e], dk[e]); dv[e] = fmaf(p[t], go[e], dv[e]); }
        if (i == (NQ == S ? t : 0) && (NQ == S || t == 0)) { // this thread also owns query i's gradient
#pragma unroll
            for (int j = 0; j < S; ++j) {
                float kk[DH];
                load16(a.k + (b * S + j) * a.kv_stride + h * DH, kk);
                const float ds = p[j] * (dp[j] - dot) * 0.25f;
#pragma unroll
                for (int e = 0; e < DH; ++e) dq[e] = fmaf(ds, kk[e], dq[e]);
            }
        }
    }
    store16(gk + (b * S + t) * a.kv_stride + h * DH, dk);
    store16(gv + (b * S + t) * a.kv_stride + h * DH, dv);
    if (NQ == S) store16(gq + (b * S + t) * a.q_stride + h * DH, dq);
    else if (t == 0) store16(gq + b * a.q_stride + h * DH, dq);
}

// the checks forward and backward make on the window geometry
int check_shape(const char *fn, int64_t n, int32_t num_queries, int64_t q_stride, int64_t kv_stride) {
    if (n <= 0) return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: n must be > 0 (got %lld)", fn, (long long)n);
    if (num_queries != 1 && num_queries != 5)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: num_queries %d is neither 1 nor 5", fn, num_queries);
    if ((q_stride | kv_stride) % 4)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: q_stride %lld and kv_stride %lld must be multiples of 4", fn,
                                  (long long)q_stride, (long long)kv_stride);
    return UAVENV_OK;
}
}  // namespace

extern "C" int ppo_attn5_forward(const float *d_q, int64_t q_stride, const float *d_k, const float *d_v, int64_t kv_stride,
                                 const uint8_t *d_pad, int64_t n, int32_t num_queries, float *d_out, int32_t device, void *stream) {
    if (!d_q || !d_k || !d_v || !d_pad || !d_out)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: q / k / v / pad / out must be non-NULL", __func__);
    if (int rc = check_shape(__func__, n, num_queries, q_stride, kv_stride)) return rc;
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    AttnArgs a{d_q, d_k, d_v, q_stride, kv_stride, d_pad, n};
    const int64_t threads = n * H * num_queries;
    const unsigned grid = (unsigned)((threads + 255) / 256);
    if (num_queries == 5) attn5_forward_kernel<5><<<grid, 256, 0, (cudaStream_t)stream>>>(a, d_out);
    else attn5_forward_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(a, d_out);
    return capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "attn5_forward_kernel launch");
}

extern "C" int ppo_attn5_backward(const float *d_q, int64_t q_stride, const float *d_k, const float *d_v, int64_t kv_stride,
                                  const uint8_t *d_pad, int64_t n, int32_t num_queries, const float *d_grad_out, float *d_grad_q,
                                  float *d_grad_k, float *d_grad_v, int32_t device, void *stream) {
    if (!d_q || !d_k || !d_v || !d_pad || !d_grad_out || !d_grad_q || !d_grad_k || !d_grad_v)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: q / k / v / pad / grad_out / grad_q / grad_k / grad_v must be "
                                  "non-NULL", __func__);
    if (int rc = check_shape(__func__, n, num_queries, q_stride, kv_stride)) return rc;
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    AttnArgs a{d_q, d_k, d_v, q_stride, kv_stride, d_pad, n};
    const unsigned grid = (unsigned)((n * H * S + 255) / 256);
    if (num_queries == 5) attn5_backward_kernel<5><<<grid, 256, 0, (cudaStream_t)stream>>>(a, d_grad_out, d_grad_q, d_grad_k, d_grad_v);
    else attn5_backward_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(a, d_grad_out, d_grad_q, d_grad_k, d_grad_v);
    return capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "attn5_backward_kernel launch");
}
