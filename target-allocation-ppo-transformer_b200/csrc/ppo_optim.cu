// ppo_optim.cu - the post-backward chain of one PPO minibatch step on flat fp32 buffers (sm_100a):
//   grad /= world (after the NCCL sum)  ->  global-norm clip (agents/ppo.py:160, torch clip_grad_norm_)  ->
//   Adam with per-group learning rates (agents/ppo.py:17-22: actor 2e-4, critic 1e-3)  ->  parameters in place.
// Two launches: (1) block-wise sums of squares, one partial per CTA written in place (no atomics: the result is
// bit-identical on every rank, so data-parallel replicas never drift apart); (2) every CTA re-reduces the partials
// in the same fixed order, then updates its slice.  The step counter lives on the device (CUDA-graph replays).
#include "uavenv_b200.h"

#include <algorithm>
#include <cstdint>
#include <cuda_runtime.h>

#include "handle.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxParts = 296;  // CTAs of the norm pass (2 per SM)

struct Segs {
    int32_t n;
    int64_t end[PPO_OPTIM_MAX_GROUPS];  // exclusive end offset of each learning-rate segment (ascending)
    float lr[PPO_OPTIM_MAX_GROUPS];
};

__device__ __forceinline__ double block_sum(double v, double *sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double s = 0.0;
    if (warp == 0) {
        s = lane < kThreads / 32 ? sh[lane] : 0.0;
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    }
    return s;  // valid in warp 0
}

// partial[blockIdx] = sum over this CTA's contiguous chunk of (grad * grad_scale)^2 ; block 0 also advances the step
__global__ void __launch_bounds__(kThreads) sumsq_kernel(const float *__restrict__ grad, int64_t n, float grad_scale,
                                                          double *__restrict__ partial, int64_t *__restrict__ step) {
    __shared__ double sh[kThreads / 32];
    const int64_t per = (n + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * per, hi = min(n, lo + per);
    double acc = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
        const float g = grad[i] * grad_scale;
        acc += (double)g * (double)g;
    }
    const double s = block_sum(acc, sh);
    if (threadIdx.x == 0) {
        partial[blockIdx.x] = s;
        if (blockIdx.x == 0) step[0] += 1;   // Adam's t of THIS update (read by adam_kernel, which runs after)
    }
}

__global__ void __launch_bounds__(kThreads) adam_kernel(float *__restrict__ param, float *__restrict__ grad,
                                                         float *__restrict__ exp_avg, float *__restrict__ exp_avg_sq,
                                                         int64_t n, const Segs segs, float grad_scale, float max_norm,
                                                         float beta1, float beta2, float eps,
                                                         const double *__restrict__ partial, int nparts,
                                                         const int64_t *__restrict__ step, float *__restrict__ norm_out) {
    __shared__ double sh[kThreads / 32];
    __shared__ float s_clip;
    // every CTA reduces the same partials in the same order: identical clip coefficient everywhere
    double acc = 0.0;
    for (int i = threadIdx.x; i < nparts; i += kThreads) acc += partial[i];
    const double tot = block_sum(acc, sh);
    if (threadIdx.x == 0) {
        const float norm = (float)sqrt(tot);
        const float coef = max_norm / (norm + 1e-6f);                 // torch.nn.utils.clip_grad_norm_
        s_clip = max_norm > 0.f ? fminf(coef, 1.0f) : 1.0f;
        if (blockIdx.x == 0 && norm_out) norm_out[0] = norm;
    }
    __syncthreads();
    const float scale = grad_scale * s_clip;
    const double t = (double)step[0];
    const float bc1 = (float)(1.0 - pow((double)beta1, t));
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, t));
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
        float lr = segs.lr[segs.n - 1];
#pragma unroll
        for (int s = PPO_OPTIM_MAX_GROUPS - 1; s >= 0; --s)
            if (s < segs.n && i < segs.end[s]) lr = segs.lr[s];
        const float g = grad[i] * scale;
        grad[i] = g;                                                   // the clipped gradient stays observable
        const float m = exp_avg[i] + (g - exp_avg[i]) * (1.0f - beta1);   // exp_avg.lerp_(grad, 1 - beta1)
        const float v = exp_avg_sq[i] * beta2 + (1.0f - beta2) * g * g;
        exp_avg[i] = m;
        exp_avg_sq[i] = v;
        const float denom = sqrtf(v) / bc2_sqrt + eps;
        param[i] -= (lr / bc1) * (m / denom);
    }
}

}  // namespace

extern "C" int ppo_clip_adam_step(float *d_params, float *d_grad, float *d_exp_avg, float *d_exp_avg_sq, int64_t n,
                                  const int64_t *seg_end, const float *seg_lr, int32_t num_segments, float grad_scale,
                                  float max_norm, float beta1, float beta2, float eps, int64_t *d_step,
                                  double *d_partials, float *d_norm_out, int32_t device, void *stream) {
    if (!d_params || !d_grad || !d_exp_avg || !d_exp_avg_sq || !seg_end || !seg_lr || !d_step || !d_partials)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: params / grad / exp_avg / exp_avg_sq / seg_end / seg_lr / step / "
                                  "partials must be non-NULL", __func__);
    if (n <= 0) return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: n must be > 0 (got %lld)", __func__, (long long)n);
    if (num_segments < 1 || num_segments > PPO_OPTIM_MAX_GROUPS)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: num_segments %d outside [1, %d]", __func__, num_segments,
                                  PPO_OPTIM_MAX_GROUPS);
    Segs segs;
    segs.n = num_segments;
    for (int i = 0; i < PPO_OPTIM_MAX_GROUPS; ++i) {
        segs.end[i] = i < num_segments ? seg_end[i] : n;
        segs.lr[i] = i < num_segments ? seg_lr[i] : 0.f;
        if (i > 0 && i < num_segments && seg_end[i] < seg_end[i - 1])
            return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: seg_end decreases at segment %d", __func__, i);
    }
    if (segs.end[num_segments - 1] != n)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: the last seg_end (%lld) is not n (%lld)", __func__,
                                  (long long)segs.end[num_segments - 1], (long long)n);
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const int nparts = (int)std::min<int64_t>(kMaxParts, (n + 4 * kThreads - 1) / (4 * kThreads));
    sumsq_kernel<<<nparts, kThreads, 0, s>>>(d_grad, n, grad_scale, d_partials, d_step);
    const int grid = (int)std::min<int64_t>((n + kThreads - 1) / kThreads, 148 * 8);
    adam_kernel<<<grid, kThreads, 0, s>>>(d_params, d_grad, d_exp_avg, d_exp_avg_sq, n, segs, grad_scale, max_norm, beta1,
                                          beta2, eps, d_partials, nparts, d_step, d_norm_out);
    return capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "sumsq_kernel / adam_kernel launch");
}

extern "C" int ppo_optim_partials(void) { return kMaxParts; }
