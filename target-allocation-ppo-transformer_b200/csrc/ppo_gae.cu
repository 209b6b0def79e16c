// ppo_gae.cu - GAE(gamma, lambda) + advantage normalisation over a [T,B] rollout (sm_100a).
//
// Reference: agents/ppo.py:77-94.  The reversed Python loop there is the first-order linear
// recurrence  gae_t = delta_t + c_t * gae_{t+1},  c_t = gamma*lambda*(1-done_t),
// delta_t = r_t + gamma*V_{t+1}*(1-done_t) - V_t  (V_T = bootstrap value, 0 in the reference).
// Affine maps compose associatively, so the time axis is cut into chunks:
//   pass 1  every warp folds its chunk into one map (A,B) for 32 env columns at once
//           (lane = column => 128 B coalesced rows of the time-major layout),
//   scan    a warp-shuffle suffix scan over the chunk maps of each column yields the carry-in,
//   pass 2  the chunk is replayed with its carry-in, writing returns / advantages and
//           accumulating {sum, sum of squares} for the normalisation in fp64.
// All recurrences are evaluated in fp64 and rounded once.
#include "uavenv_b200.h"

#include <algorithm>
#include <cstdint>
#include <cuda_runtime.h>

#include "handle.cuh"

namespace {

constexpr int kCols = 32;       // env columns per CTA (one per lane)
constexpr int kMaxChunks = 32;  // warps per CTA = time chunks (scan width is one warp)

__global__ void __launch_bounds__(kCols * kMaxChunks)
gae_kernel(const float *__restrict__ rewards, const float *__restrict__ values, const uint8_t *__restrict__ dones,
           const float *__restrict__ last_value, int T, int B, int chunk_len, double gamma, double lam,
           float *__restrict__ returns, float *__restrict__ adv, double *__restrict__ stats) {
    __shared__ double s_A[kMaxChunks][kCols + 1], s_B[kMaxChunks][kCols + 1], s_carry[kMaxChunks][kCols + 1];
    __shared__ double s_sum[kMaxChunks], s_sq[kMaxChunks];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, W = blockDim.x >> 5;
    const int b = blockIdx.x * kCols + lane;
    const bool live = b < B;
    const int t0 = w * chunk_len, t1 = min(T, t0 + chunk_len);

    // pass 1: fold the chunk [t0,t1) backwards into gae_{t0} = Bc + Ac * gae_{t1}
    double Ac = 1.0, Bc = 0.0;
    if (live) {
        double v_next = (t1 < T) ? (double)values[(size_t)t1 * B + b] : (last_value ? (double)last_value[b] : 0.0);
        for (int t = t1 - 1; t >= t0; --t) {
            const size_t i = (size_t)t * B + b;
            const double nd = dones[i] ? 0.0 : 1.0;
            const double v = (double)values[i];
            const double delta = (double)rewards[i] + gamma * v_next * nd - v;   // ppo.py:86
            const double c = gamma * lam * nd;                                  // ppo.py:87
            Bc = delta + c * Bc;
            Ac = c * Ac;
            v_next = v;
        }
    }
    s_A[w][lane] = Ac; s_B[w][lane] = Bc;
    __syncthreads();

    // warp-shuffle suffix scan over the chunk maps: warp j serves columns j, j+W, ...; lane = chunk
    for (int col = w; col < kCols; col += W) {
        double a = lane < W ? s_A[lane][col] : 1.0;
        double bb = lane < W ? s_B[lane][col] : 0.0;
#pragma unroll
        for (int o = 1; o < kMaxChunks; o <<= 1) {
            const double a2 = __shfl_down_sync(0xffffffffu, a, o);
            const double b2 = __shfl_down_sync(0xffffffffu, bb, o);
            if (lane + o < kMaxChunks) { bb = bb + a * b2; a = a * a2; }   // (later chunks) then (this one)
        }
        // bb = gae at the first step of chunk `lane`; the carry-in of chunk `lane` is the next chunk's
        const double carry = __shfl_down_sync(0xffffffffu, bb, 1);
        if (lane < W) s_carry[lane][col] = (lane + 1 < W) ? carry : 0.0;
    }
    __syncthreads();

    // pass 2: replay with the carry-in, write outputs, accumulate normalisation statistics
    double sum = 0.0, sq = 0.0;
    if (live) {
        double gae = s_carry[w][lane];
        double v_next = (t1 < T) ? (double)values[(size_t)t1 * B + b] : (last_value ? (double)last_value[b] : 0.0);
        for (int t = t1 - 1; t >= t0; --t) {
            const size_t i = (size_t)t * B + b;
            const double nd = dones[i] ? 0.0 : 1.0;
            const double v = (double)values[i];
            const double delta = (double)rewards[i] + gamma * v_next * nd - v;
            gae = delta + gamma * lam * nd * gae;
            const float ret = (float)(gae + v);                                  // ppo.py:89
            const float a = ret - (float)v;                                      // ppo.py:92 (f32 subtraction)
            returns[i] = ret;
            adv[i] = a;
            sum += (double)a; sq += (double)a * (double)a;
            v_next = v;
        }
    }
    if (stats) {
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sq += __shfl_xor_sync(0xffffffffu, sq, o);
        }
        if (lane == 0) { s_sum[w] = sum; s_sq[w] = sq; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double S = 0.0, Q = 0.0;
            for (int i = 0; i < W; ++i) { S += s_sum[i]; Q += s_sq[i]; }
            atomicAdd(&stats[1], S);
            atomicAdd(&stats[2], Q);
            if (blockIdx.x == 0) stats[0] = (double)T * (double)B;
        }
    }
}

// advantages = (adv - mean) / (std_unbiased + 1e-7)          agents/ppo.py:94
__global__ void normalize_kernel(float *__restrict__ adv, int64_t n, const double *__restrict__ stats) {
    const double cnt = stats[0], S = stats[1], Q = stats[2];
    const double mean = S / cnt;
    double var = cnt > 1.0 ? (Q - S * S / cnt) / (cnt - 1.0) : 0.0;
    if (var < 0.0) var = 0.0;
    const float fmean = (float)mean;
    const float inv = (float)(1.0 / (sqrt(var) + 1e-7));
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) adv[i] = (adv[i] - fmean) * inv;
}

}  // namespace

extern "C" int ppo_normalize_advantages(float *d_advantages, int64_t n, const double *d_adv_stats, int32_t device,
                                        void *stream) {
    if (!d_advantages || !d_adv_stats)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: advantages / adv_stats must be non-NULL", __func__);
    if (n <= 0) return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: n must be > 0 (got %lld)", __func__, (long long)n);
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    normalize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_advantages, n, d_adv_stats);
    return capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "normalize_kernel launch");
}

extern "C" int ppo_gae_advantages(const float *d_rewards, const float *d_values, const uint8_t *d_dones,
                                  const float *d_last_value, int32_t T, int32_t B, float gamma, float lam,
                                  float *d_returns, float *d_advantages, int32_t normalize, double *d_adv_stats,
                                  int32_t device, void *stream) {
    if (!d_rewards || !d_values || !d_dones || !d_returns || !d_advantages)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: rewards / values / dones / returns / advantages must be non-NULL",
                                  __func__);
    if (T <= 0 || B <= 0)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: need T > 0 and B > 0 (got %d, %d)", __func__, T, B);
    if (normalize && !d_adv_stats)  // the statistics buffer is caller-owned (no hidden allocation)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: normalize needs adv_stats", __func__);
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    // chunks: as many warps as keep every chunk >= 4 steps, at most 32
    int W = std::max(1, std::min(kMaxChunks, T / 4));
    const int chunk_len = (T + W - 1) / W;
    W = (T + chunk_len - 1) / chunk_len;
    if (d_adv_stats) {
        const cudaError_t e = cudaMemsetAsync(d_adv_stats, 0, 3 * sizeof(double), s);
        if (int rc = capi::check_cuda<uavenv>(e, __func__, "cudaMemsetAsync")) return rc;
    }
    const int grid = (B + kCols - 1) / kCols;
    gae_kernel<<<grid, kCols * W, 0, s>>>(d_rewards, d_values, d_dones, d_last_value, T, B, chunk_len, (double)gamma,
                                          (double)lam, d_returns, d_advantages, d_adv_stats);
    if (int rc = capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "gae_kernel launch")) return rc;
    if (normalize) return ppo_normalize_advantages(d_advantages, (int64_t)T * B, d_adv_stats, device, stream);
    return UAVENV_OK;
}
