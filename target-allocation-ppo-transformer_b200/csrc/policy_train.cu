// policy_train.cu - forward + backward of the two transformer trunks for the PPO update (agents/ppo.py:126-160:
// policy.evaluate(...) and loss.backward() of networks/transformer_net.py:47-65) on sm_100a.
//
// Same formulation as the rollout forward (policy_forward.cu): the last encoder layer of a block computes K/V for all
// five tokens but everything else for the newest token only.  Activations are bf16 and are KEPT for the backward;
// LayerNorm statistics, softmax, all reductions and every parameter gradient are fp32.
//   activation-gradient GEMMs  dX = dY W     -> uavp::gemm_bias_act on pre-transposed bf16 weights (tcgen05)
//   weight-gradient GEMMs      dW += dY^T X  -> uavp::wgrad (policy_wgrad.cu: split-K, TMA ring, accumulator resident in TMEM)
//   ReLU backward of the FFN                 -> fused into the epilogue of the activation-gradient GEMM (uavp::gemm_drelu)
//   everything else (LayerNorm / attention / embedding backward, LayerNorm parameter gradients, heads, PPO loss) is
//   hand-written below; bias gradients come from the LayerNorm backward where a bias feeds a LayerNorm, and from the
//   weight-gradient kernel (as dY^T 1 on the tensor cores) everywhere else.
// Three entry levels: uavtrain_forward / _backward stop at the trunks' last-token features ([n,2,128] out, their gradient
// in); uavtrain_forward_heads / _backward_heads also run the two MLP heads (logits [n,2] + value [n] out, their
// gradients in); uavtrain_ppo_loss turns the heads' outputs into the PPO loss statistics and those gradients.
#include "uavpolicy_b200.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "policy_gemm.cuh"
#include "handle.cuh"
#include "policy_kernels.cuh"
#include "policy_weights.cuh"

namespace uavp {
int wgrad_prepare();
int wgrad(const __nv_bfloat16 *dY, int64_t ld_dy, const __nv_bfloat16 *X, int64_t ld_x, int rows, int Nout, int Kin, float *dW,
          int nout_valid, float *dbias, int num_sms, cudaStream_t stream, int out_ld, int kin_valid);
}  // namespace uavp

namespace {
using bf16 = __nv_bfloat16;

// ---------------------------------------------------------------------------------------------- forward kernels

// embedding of both nets: E = relu(obs W^T + b) + pos (transformer_net.py:24-30,57-59) and the key-padding mask
// (rows that are all zero, newest row never: :52-54).  One CTA = 64 tokens; thread = (net, feature pair), so a warp
// stores 128 contiguous bytes per token.
constexpr int kEmbTok = 60;                                   // whole windows per CTA: token i sits at position i % 5
// packed fp32x2 arithmetic (FFMA2): both features of a thread advance with one instruction per observation column
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
constexpr int kEmbThreads = 64;                               // warp 0: actor, warp 1: critic; lane = 4 features
__global__ void __launch_bounds__(kEmbThreads) embed_kernel(const float *__restrict__ obs, int R, BlockW a, BlockW c,
                                                            __nv_bfloat16 *__restrict__ Ea, __nv_bfloat16 *__restrict__ Ec,
                                                            uint8_t *__restrict__ pad, __nv_bfloat16 *__restrict__ obs16 = nullptr,
                                                            uint32_t *__restrict__ relu_mask = nullptr) {
    // obs16 / relu_mask (training only): a bf16 copy of the observation rows zero-padded to 64 columns (the B operand of
    // the embedding's weight-gradient product) and the ReLU activity bits of both networks, [R][net][4 words]:
    // word k, bit l  <->  feature 4 l + k
    // (the update always passes both; without the null checks below nvcc schedules this kernel about 11 us slower per
    // 131072-window minibatch on a B200, measured)
    __shared__ __align__(16) float2 s_obs[kEmbTok][F];            // every value twice: the (x, x) operand of the packed FMA
    const int t0 = blockIdx.x * kEmbTok;
    {   // the CTA's 60 x 14 floats are contiguous and 16-byte aligned: all loads of a thread go out before any is used
        constexpr int kVec = kEmbTok * F / 4, kPer = (kVec + kEmbThreads - 1) / kEmbThreads;
        const float4 *src = reinterpret_cast<const float4 *>(obs + (size_t)t0 * F);
        const int nvec = min(kVec, (int)(((size_t)(R - t0) * F) / 4));        // R % 5 == 0 and 5 * 14 % 4 != 0: see tail below
        float4 v[kPer];
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int i = threadIdx.x + k * kEmbThreads;
            v[k] = i < nvec ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int i = threadIdx.x + k * kEmbThreads;
            if (i < kVec) {
                float2 *dst = &s_obs[0][0] + i * 4;
                dst[0] = make_float2(v[k].x, v[k].x); dst[1] = make_float2(v[k].y, v[k].y);
                dst[2] = make_float2(v[k].z, v[k].z); dst[3] = make_float2(v[k].w, v[k].w);
            }
        }
        const int done = nvec * 4, total = min(kEmbTok, R - t0) * F;          // at most 3 trailing floats of the last CTA
        for (int i = done + threadIdx.x; i < total; i += kEmbThreads) { const float x = obs[(size_t)t0 * F + i]; (&s_obs[0][0])[i] = make_float2(x, x); }
    }
    __syncthreads();
    if (threadIdx.x < kEmbTok && t0 + threadIdx.x < R) {
        float sum = 0.0f;
        for (int j = 0; j < F; ++j) sum += fabsf(s_obs[threadIdx.x][j].x);
        pad[t0 + threadIdx.x] = (sum == 0.0f && (t0 + threadIdx.x) % S != S - 1) ? 1 : 0;
    }
    if (obs16) {
        for (int i = threadIdx.x; i < kEmbTok * 32; i += kEmbThreads) {
            const int tok = i >> 5, c2 = (i & 31) * 2;
            if (t0 + tok < R)
                *reinterpret_cast<__nv_bfloat162 *>(obs16 + (size_t)(t0 + tok) * 64 + c2) =
                    __floats2bfloat162_rn(c2 < F ? s_obs[tok][c2].x : 0.0f, c2 + 1 < F ? s_obs[tok][c2 + 1].x : 0.0f);
        }
    }
    const bool critic = threadIdx.x >= 32;
    const int d = (threadIdx.x & 31) * 4;                          // features d .. d+3
    const BlockW &w = critic ? c : a;
    __nv_bfloat16 *E = critic ? Ec : Ea;
    uint64_t wa[F], wb[F];                                         // (w[d], w[d+1]) and (w[d+2], w[d+3]) per observation column
#pragma unroll
    for (int j = 0; j < F; ++j) {
        wa[j] = pack_f32x2(w.emb_w[d * F + j], w.emb_w[(d + 1) * F + j]);
        wb[j] = pack_f32x2(w.emb_w[(d + 2) * F + j], w.emb_w[(d + 3) * F + j]);
    }
    const uint64_t ba = pack_f32x2(w.emb_b[d], w.emb_b[d + 1]), bb = pack_f32x2(w.emb_b[d + 2], w.emb_b[d + 3]);
    float pos[S][4];
#pragma unroll
    for (int p = 0; p < S; ++p)
#pragma unroll
        for (int k = 0; k < 4; ++k) pos[p][k] = w.pos[p * D + d + k];
    uint32_t *const mask_dst = relu_mask ? relu_mask + (critic ? 4 : 0) : nullptr;
    for (int win = 0; win < kEmbTok / S; ++win) {                 // R is a multiple of 5: windows are never split
        if (t0 + win * S >= R) break;
#pragma unroll
        for (int p = 0; p < S; ++p) {                              // p = position of the token in its window (static)
            const int i = win * S + p, t = t0 + i;
            uint64_t xa = ba, xb = bb;
#pragma unroll
            for (int j = 0; j < F; ++j) {
                const uint64_t oo = *reinterpret_cast<const uint64_t *>(&s_obs[i][j]);     // (o_j, o_j)
                xa = fma_f32x2(wa[j], oo, xa);
                xb = fma_f32x2(wb[j], oo, xb);
            }
            float x[4];
            unpack_f32x2(xa, x[0], x[1]);
            unpack_f32x2(xb, x[2], x[3]);
            if (mask_dst) {
                unsigned m[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) m[k] = __ballot_sync(0xffffffffu, x[k] > 0.0f);
                if ((threadIdx.x & 31) == 0) *reinterpret_cast<uint4 *>(mask_dst + (size_t)t * 8) = make_uint4(m[0], m[1], m[2], m[3]);
            }
            const __nv_bfloat162 e0 = __floats2bfloat162_rn(fmaxf(x[0], 0.0f) + pos[p][0], fmaxf(x[1], 0.0f) + pos[p][1]);
            const __nv_bfloat162 e1 = __floats2bfloat162_rn(fmaxf(x[2], 0.0f) + pos[p][2], fmaxf(x[3], 0.0f) + pos[p][3]);
            uint2 ev;
            ev.x = *reinterpret_cast<const uint32_t *>(&e0); ev.y = *reinterpret_cast<const uint32_t *>(&e1);
            *reinterpret_cast<uint2 *>(E + (size_t)t * D + d) = ev;
        }
    }
}

// ---- attention of an inner encoder layer (all five queries), warp = sample --------------------------------------------
// Lane l owns 4 of the 128 feature dimensions: head h = l / 4, dimensions h*16 + (l % 4)*4 ..+4.  A token row of Q, K, V
// or of the output is then ONE fully coalesced 256-byte warp access (8 B per lane), every element of Q / K / V is loaded
// exactly once per sample, and the 5 x 5 score block of a head is a folded reduction: each lane forms its 4-dimension
// partial of all 25 dot products, two xor-shuffles (lanes l^1, l^2) complete them inside the head's 4 lanes.
// (The first version had a thread per (sample, head, query) holding 16-dimension vectors: every K / V row was re-loaded
// five times and the register footprint capped the occupancy - 0.37-0.69 of the traffic floor.)
struct Rows4 { uint2 t[S]; };                     // 5 token rows x this lane's 4 bf16 features, packed
// block[i][j] = a_i . b_j over the head's 16 dimensions (every lane of the head ends with all 25 values)
__device__ __forceinline__ void head_dots(const Rows4 &A, const Rows4 &Bm, float (*blk)[S]) {
    float bf[S][4];
#pragma unroll
    for (int j = 0; j < S; ++j) unpack4f(Bm.t[j], bf[j]);
#pragma unroll
    for (int i = 0; i < S; ++i) {
        float af[4];
        unpack4f(A.t[i], af);
#pragma unroll
        for (int j = 0; j < S; ++j)
            blk[i][j] = xor_sum<1, 2>(fmaf(af[0], bf[j][0], fmaf(af[1], bf[j][1], fmaf(af[2], bf[j][2], af[3] * bf[j][3]))));
    }
}
// softmax over the keys of every query row, scores scaled by 1/sqrt(16), padded keys masked (transformer_net.py:52-54,63)
__device__ __forceinline__ void head_softmax(float (*p)[S], const uint8_t *pad) {
    bool pd[S];
#pragma unroll
    for (int j = 0; j < S; ++j) pd[j] = pad[j] != 0;
#pragma unroll
    for (int i = 0; i < S; ++i) {
        float mx = -INFINITY, den = 0.0f;
#pragma unroll
        for (int j = 0; j < S; ++j) { p[i][j] = pd[j] ? -INFINITY : p[i][j] * 0.25f; mx = fmaxf(mx, p[i][j]); }
#pragma unroll
        for (int j = 0; j < S; ++j) { p[i][j] = __expf(p[i][j] - mx); den += p[i][j]; }
        const float inv = 1.0f / den;
#pragma unroll
        for (int j = 0; j < S; ++j) p[i][j] *= inv;
    }
}

// QKV [R,384] -> ATT [R,128]
__global__ void __launch_bounds__(256) attn_full_kernel(const __nv_bfloat16 *__restrict__ QKV, const uint8_t *__restrict__ pad, int B,
                                                        __nv_bfloat16 *__restrict__ ATT) {
    const int lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += nwarps) {
        const __nv_bfloat16 *base = QKV + (size_t)b * S * 3 * D + lane * 4;
        Rows4 q, k, v;
#pragma unroll
        for (int t = 0; t < S; ++t) {
            q.t[t] = *reinterpret_cast<const uint2 *>(base + (size_t)t * 3 * D);
            k.t[t] = *reinterpret_cast<const uint2 *>(base + (size_t)t * 3 * D + D);
            v.t[t] = *reinterpret_cast<const uint2 *>(base + (size_t)t * 3 * D + 2 * D);
        }
        float p[S][S];
        head_dots(q, k, p);
        head_softmax(p, pad + (size_t)b * S);
        float vf[S][4];
#pragma unroll
        for (int j = 0; j < S; ++j) unpack4f(v.t[j], vf[j]);
#pragma unroll
        for (int i = 0; i < S; ++i) {
            float o[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int j = 0; j < S; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) o[e] = fmaf(p[i][j], vf[j][e], o[e]);
            *reinterpret_cast<uint2 *>(ATT + ((size_t)b * S + i) * D + lane * 4) = pack4f(o);
        }
    }
}

// ---- attention of the last encoder layer (newest query only), thread = (sample, head) ----------------------------------
// normalised softmax(q k^T / sqrt(16), key padding mask) of one (sample, head) over its 5 keys (rows k0 + j * stride).
// The backward (attn_row_grads) recomputes exactly these probabilities by calling this too.
__device__ __forceinline__ void softmax_row(const float *q, const __nv_bfloat16 *k0, int64_t stride, const uint8_t *pad, float *p) {
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float kk[DH], s = 0.0f;
        load16(k0 + j * stride, kk);
#pragma unroll
        for (int e = 0; e < DH; ++e) s = fmaf(q[e], kk[e], s);
        p[j] = pad[j] ? -INFINITY : s * 0.25f;
        mx = fmaxf(mx, p[j]);
    }
    float den = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) { p[j] = __expf(p[j] - mx); den += p[j]; }
    const float inv = 1.0f / den;
#pragma unroll
    for (int j = 0; j < S; ++j) p[j] *= inv;
}

// softmax(q k^T / sqrt(16), key padding mask) v for one (sample, head, query): q, and 5 keys / values of 16 dims
__device__ __forceinline__ void attend(const float *q, const __nv_bfloat16 *k0, const __nv_bfloat16 *v0, int64_t stride,
                                       const uint8_t *pad, float *out) {
    float p[S];
    softmax_row(q, k0, stride, pad, p);
#pragma unroll
    for (int e = 0; e < DH; ++e) out[e] = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float vv[DH];
        load16(v0 + j * stride, vv);
#pragma unroll
        for (int e = 0; e < DH; ++e) out[e] = fmaf(p[j], vv[e], out[e]);
    }
}

// Q [B,128], KV [R,256] -> ATT [B,128]
__global__ void attn_last_kernel(const __nv_bfloat16 *__restrict__ Q, const __nv_bfloat16 *__restrict__ KV,
                                 const uint8_t *__restrict__ pad, int B, __nv_bfloat16 *__restrict__ ATT) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * H) return;
    const int b = idx / H, h = idx % H;
    float q[DH], o[DH];
    load16(Q + (size_t)b * D + h * DH, q);
    const __nv_bfloat16 *base = KV + (size_t)b * S * 2 * D + h * DH;
    attend(q, base, base + D, 2 * D, pad + b * S, o);
    store16(ATT + (size_t)b * D + h * DH, o);
}

// out = LayerNorm(x + y) * g + beta, keeping what the backward needs: the normalised row x^ (bf16) and 1/sigma.
// Half a warp per row, 8 features (16 bytes) per lane.  out16 (bf16, dense) and out32 (fp32, row stride out32_stride)
// are both optional.
__global__ void __launch_bounds__(256) add_ln_train_kernel(const bf16 *__restrict__ x, int64_t x_stride, const bf16 *__restrict__ y,
                                                           const float *__restrict__ g, const float *__restrict__ beta, int rows,
                                                           bf16 *__restrict__ out16, float *__restrict__ out32, int64_t out32_stride,
                                                           bf16 *__restrict__ xhat, float *__restrict__ rstd_out) {
    const int hl = threadIdx.x & 15;
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool live = r < rows;
    const int rc = live ? r : rows - 1;                               // (idle tail lanes still take part in the shuffles)
    float a[8], b[8], v[8];
    unpack8(*reinterpret_cast<const uint4 *>(x + (size_t)rc * x_stride + hl * 8), a);
    unpack8(*reinterpret_cast<const uint4 *>(y + (size_t)rc * D + hl * 8), b);
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i] = a[i] + b[i]; s += v[i]; }
    const float mean = xor_sum<8, 4, 2, 1>(s) * (1.0f / D);       // over the 16 lanes that share a row
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i] -= mean; q = fmaf(v[i], v[i], q); }
    const float rstd = rsqrtf(xor_sum<8, 4, 2, 1>(q) * (1.0f / D) + 1e-5f);
    if (!live) return;
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i] *= rstd; o[i] = v[i] * g[hl * 8 + i] + beta[hl * 8 + i]; }
    *reinterpret_cast<uint4 *>(xhat + (size_t)r * D + hl * 8) = pack8(v);
    if (hl == 0) rstd_out[r] = rstd;
    if (out16) *reinterpret_cast<uint4 *>(out16 + (size_t)r * D + hl * 8) = pack8(o);
    if (out32) {
        float4 *dst = reinterpret_cast<float4 *>(out32 + (size_t)r * out32_stride + hl * 8);
        dst[0] = make_float4(o[0], o[1], o[2], o[3]); dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
}

// fp32 row-major [N,K] -> bf16 copy and / or bf16 transposed copy [K,N]; one launch converts every GEMM weight
struct PrepJob { const float *src; bf16 *dst, *dst_t; int N, K; };
constexpr int kMaxPrepJobs = 24;
struct PrepJobs { PrepJob job[kMaxPrepJobs]; };
__global__ void prep_weights_kernel(const __grid_constant__ PrepJobs jobs) {
    const PrepJob &j = jobs.job[blockIdx.y];
    const int n = j.N * j.K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const bf16 v = __float2bfloat16(j.src[i]);
        if (j.dst) j.dst[i] = v;
        if (j.dst_t) j.dst_t[(size_t)(i % j.K) * j.N + i / j.K] = v;
    }
}

// ---------------------------------------------------------------------------------------------- backward kernels

// block-level reduction of per-lane column partial sums: part[NV] of every warp (lane owns columns col(lane, i)) ->
// one atomicAdd per column per CTA.  s_red: [warps][C] floats.
template <int NV, int C, typename ColFn>
__device__ __forceinline__ void block_colsum_flush(const float *part, float *s_red, float *dst, ColFn col) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) s_red[warp * C + col(lane, i)] = part[i];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float s = 0.0f;
        for (int w = 0; w < nwarps; ++w) s += s_red[w * C + c];
        atomicAdd(dst + c, s);
    }
    __syncthreads();
}

// LayerNorm backward over 128 features.  dy = (DY32 ? fp32 rows of stride dy_stride : bf16 dense) [+ add (bf16 dense)];
//   dz = rstd * (g*dy - mean(g*dy) - x^ * mean(g*dy*x^))       -> bf16 dense (gradient of the pre-norm sum: it flows
//   into the residual branch and into the GEMM branch alike)
//   g_gamma += sum_r dy*x^,  g_beta += sum_r dy,  g_bias += sum_r dz (bias of the linear layer that fed the sum)
// A warp walks `rows_per_warp` consecutive rows with its lanes on fixed columns, so the three column sums stay in
// registers until the end.
template <bool DY32>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const void *__restrict__ dy_, int64_t dy_stride, const bf16 *__restrict__ add,
                                                     const bf16 *__restrict__ xhat, const float *__restrict__ rstd,
                                                     const float *__restrict__ gamma, int rows, int rows_per_warp,
                                                     bf16 *__restrict__ dz, float *__restrict__ g_gamma,
                                                     float *__restrict__ g_beta, float *__restrict__ g_bias) {
    __shared__ float s_red[8 * D];
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int r0 = gw * rows_per_warp, r1 = min(rows, r0 + rows_per_warp);
    float gm[4], ag[4] = {0, 0, 0, 0}, ab[4] = {0, 0, 0, 0}, az[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 4; ++i) gm[i] = gamma[lane * 4 + i];
    for (int r = r0; r < r1; ++r) {
        float dy[4], xh[4];
        if (DY32) {
            const float4 t = *reinterpret_cast<const float4 *>(static_cast<const float *>(dy_) + (size_t)r * dy_stride + lane * 4);
            dy[0] = t.x; dy[1] = t.y; dy[2] = t.z; dy[3] = t.w;
        } else {
            unpack4f(*reinterpret_cast<const uint2 *>(static_cast<const bf16 *>(dy_) + (size_t)r * D + lane * 4), dy);
        }
        if (add) {
            float t[4];
            unpack4f(*reinterpret_cast<const uint2 *>(add + (size_t)r * D + lane * 4), t);
#pragma unroll
            for (int i = 0; i < 4; ++i) dy[i] += t[i];
        }
        unpack4f(*reinterpret_cast<const uint2 *>(xhat + (size_t)r * D + lane * 4), xh);
        const float rs = rstd[r];
        float s1 = 0.0f, s2 = 0.0f, gd[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { gd[i] = gm[i] * dy[i]; s1 += gd[i]; s2 = fmaf(gd[i], xh[i], s2); }
        for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
        s1 *= (1.0f / D); s2 *= (1.0f / D);
        float z[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            z[i] = rs * (gd[i] - s1 - xh[i] * s2);
            ag[i] = fmaf(dy[i], xh[i], ag[i]); ab[i] += dy[i]; az[i] += z[i];
        }
        *reinterpret_cast<uint2 *>(dz + (size_t)r * D + lane * 4) = pack4f(z);
    }
    auto col = [](int l, int i) { return l * 4 + i; };
    block_colsum_flush<4, D>(ag, s_red, g_gamma, col);
    block_colsum_flush<4, D>(ab, s_red, g_beta, col);
    block_colsum_flush<4, D>(az, s_red, g_bias, col);
}

// attention backward.  dS_ij = p_ij (dO_i.v_j - sum_l p_il dO_i.v_l) / 4;  dQ_i = sum_j dS_ij k_j;  dK_j = sum_i dS_ij q_i;
// dV_j = sum_i p_ij dO_i.  The softmax rows are recomputed from Q / K (nothing but Q, K, V was kept by the forward).
struct AttnBwdArgs {
    const bf16 *q, *k, *v, *gout;      // q rows: (b*NQ+i)*q_stride; k/v rows: (b*S+j)*kv_stride; gout rows dense 128
    bf16 *gq, *gk, *gv;                // same strides as q / k / v
    int64_t q_stride, kv_stride;
    const uint8_t *pad;
    int n;
};

// softmax row of one query over the 5 keys of (sample b, head h) (the forward's softmax_row), and dS for that query
__device__ __forceinline__ void attn_row_grads(const AttnBwdArgs &a, int64_t b, int h, const float *q, const float *go, float *p, float *ds) {
    softmax_row(q, a.k + b * S * a.kv_stride + h * DH, a.kv_stride, a.pad + b * S, p);
    float dot = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float vv[DH], s = 0.0f;
        load16(a.v + (b * S + j) * a.kv_stride + h * DH, vv);
#pragma unroll
        for (int e = 0; e < DH; ++e) s = fmaf(go[e], vv[e], s);
        ds[j] = s;
        dot = fmaf(p[j], s, dot);
    }
#pragma unroll
    for (int j = 0; j < S; ++j) ds[j] = p[j] * (ds[j] - dot) * 0.25f;
}

// last layer (one query per sample): thread = (sample, head) owns dQ and all five dK / dV rows of its head
__global__ void __launch_bounds__(256) attn_bwd_last_kernel(const AttnBwdArgs a) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)a.n * H) return;
    const int64_t b = idx / H;
    const int h = (int)(idx % H);
    float q[DH], go[DH], p[S], ds[S], dq[DH];
    load16(a.q + b * a.q_stride + h * DH, q);
    load16(a.gout + b * D + h * DH, go);
    attn_row_grads(a, b, h, q, go, p, ds);
#pragma unroll
    for (int e = 0; e < DH; ++e) dq[e] = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float kk[DH], dk[DH], dv[DH];
        load16(a.k + (b * S + j) * a.kv_stride + h * DH, kk);
#pragma unroll
        for (int e = 0; e < DH; ++e) { dq[e] = fmaf(ds[j], kk[e], dq[e]); dk[e] = ds[j] * q[e]; dv[e] = p[j] * go[e]; }
        store16(a.gk + (b * S + j) * a.kv_stride + h * DH, dk);
        store16(a.gv + (b * S + j) * a.kv_stride + h * DH, dv);
    }
    store16(a.gq + b * a.q_stride + h * DH, dq);
}

// inner layer (five queries): warp = sample, lane = 4 feature dimensions of a head (as in attn_full_kernel above).
// P is recomputed from Q, K; dP = dO V^T is a second folded 5 x 5 reduction; dS = P o (dP - rowsum(P o dP)) / 4; then
// dQ = dS K, dK = dS^T Q, dV = P^T dO are plain 4-dimension FMAs per lane.  Every input row is loaded once (coalesced
// 256 B per warp access) and every gradient row stored once.
__global__ void __launch_bounds__(256, 2) attn_bwd_full_kernel(const AttnBwdArgs a) {
    const int lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int64_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < a.n; b += nwarps) {
        Rows4 q, k, v, go;
#pragma unroll
        for (int t = 0; t < S; ++t) {
            q.t[t] = *reinterpret_cast<const uint2 *>(a.q + (b * S + t) * a.q_stride + lane * 4);
            k.t[t] = *reinterpret_cast<const uint2 *>(a.k + (b * S + t) * a.kv_stride + lane * 4);
            v.t[t] = *reinterpret_cast<const uint2 *>(a.v + (b * S + t) * a.kv_stride + lane * 4);
            go.t[t] = *reinterpret_cast<const uint2 *>(a.gout + (b * S + t) * D + lane * 4);
        }
        float p[S][S], ds[S][S];
        head_dots(q, k, p);
        head_softmax(p, a.pad + b * S);
        head_dots(go, v, ds);                                  // dP_ij = dO_i . v_j
#pragma unroll
        for (int i = 0; i < S; ++i) {
            float dot = 0.0f;
#pragma unroll
            for (int j = 0; j < S; ++j) dot = fmaf(p[i][j], ds[i][j], dot);
#pragma unroll
            for (int j = 0; j < S; ++j) ds[i][j] = p[i][j] * (ds[i][j] - dot) * 0.25f;
        }
        {   // dQ_i = sum_j dS_ij k_j
            float kf[S][4];
#pragma unroll
            for (int j = 0; j < S; ++j) unpack4f(k.t[j], kf[j]);
#pragma unroll
            for (int i = 0; i < S; ++i) {
                float o[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int j = 0; j < S; ++j)
#pragma unroll
                    for (int e = 0; e < 4; ++e) o[e] = fmaf(ds[i][j], kf[j][e], o[e]);
                *reinterpret_cast<uint2 *>(a.gq + (b * S + i) * a.q_stride + lane * 4) = pack4f(o);
            }
        }
        {   // dK_j = sum_i dS_ij q_i ;  dV_j = sum_i p_ij dO_i
            float qf[S][4], gf[S][4];
#pragma unroll
            for (int i = 0; i < S; ++i) { unpack4f(q.t[i], qf[i]); unpack4f(go.t[i], gf[i]); }
#pragma unroll
            for (int j = 0; j < S; ++j) {
                float dk[4] = {0.0f, 0.0f, 0.0f, 0.0f}, dv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int i = 0; i < S; ++i)
#pragma unroll
                    for (int e = 0; e < 4; ++e) { dk[e] = fmaf(ds[i][j], qf[i][e], dk[e]); dv[e] = fmaf(p[i][j], gf[i][e], dv[e]); }
                *reinterpret_cast<uint2 *>(a.gk + (b * S + j) * a.kv_stride + lane * 4) = pack4f(dk);
                *reinterpret_cast<uint2 *>(a.gv + (b * S + j) * a.kv_stride + lane * 4) = pack4f(dv);
            }
        }
    }
}

// dX[b*5+4] += t[b] + u[b]  (last layer: the newest token's row also receives the Q-projection and residual gradients)
__global__ void scatter_add_last_kernel(bf16 *__restrict__ dX, const bf16 *__restrict__ t, const bf16 *__restrict__ u, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;       // one thread = 4 features
    if (i >= n * (D / 4)) return;
    const int b = i / (D / 4), c = (i % (D / 4)) * 4;
    float x[4], y[4], z[4];
    bf16 *dst = dX + ((size_t)b * S + S - 1) * D + c;
    unpack4f(*reinterpret_cast<const uint2 *>(dst), x);
    unpack4f(*reinterpret_cast<const uint2 *>(t + (size_t)b * D + c), y);
    unpack4f(*reinterpret_cast<const uint2 *>(u + (size_t)b * D + c), z);
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] += y[k] + z[k];
    *reinterpret_cast<uint2 *>(dst) = pack4f(x);
}

// embedding backward: E = relu(obs W^T + b) + pos.  The forward left the ReLU activity bits (embed_kernel) and a bf16
// copy of the observations padded to 64 columns, so what remains here is elementwise:
// dPre = (g1 [+ g2]) masked -> bf16 rows, dpos = per-position column sums of the unmasked gradient (registers, lane = 4
// features).  dW = dPre^T obs16 and db = dPre^T 1 then come from the tensor-core weight-gradient kernel (Kin = 64).
__global__ void __launch_bounds__(256) embed_mask_kernel(const bf16 *__restrict__ g1, const bf16 *__restrict__ g2,
                                                         const uint32_t *__restrict__ mask /* this net's 4 words of row 0; row stride 8 */,
                                                         int n, int samples_per_warp, bf16 *__restrict__ dpre, float *__restrict__ g_pos) {
    __shared__ float s_red[S][D];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < S * D; i += blockDim.x) (&s_red[0][0])[i] = 0.0f;
    __syncthreads();
    const int gw = blockIdx.x * 8 + warp;
    const int b0 = gw * samples_per_warp, b1 = min(n, b0 + samples_per_warp);
    float dpos[S][4];
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
        for (int f = 0; f < 4; ++f) dpos[s][f] = 0.0f;
    for (int b = b0; b < b1; ++b) {
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const size_t row = (size_t)b * S + s, off = row * D + lane * 4;
            float g[4];
            unpack4f(*reinterpret_cast<const uint2 *>(g1 + off), g);
            if (g2) {
                float t[4];
                unpack4f(*reinterpret_cast<const uint2 *>(g2 + off), t);
#pragma unroll
                for (int f = 0; f < 4; ++f) g[f] += t[f];
            }
            const uint4 m = *reinterpret_cast<const uint4 *>(mask + row * 8);             // word f, bit lane <-> feature 4 lane + f
            const unsigned mw[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                dpos[s][f] += g[f];
                g[f] = ((mw[f] >> lane) & 1u) ? g[f] : 0.0f;
            }
            *reinterpret_cast<uint2 *>(dpre + off) = pack4f(g);
        }
    }
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
        for (int f = 0; f < 4; ++f) atomicAdd(&s_red[s][lane * 4 + f], dpos[s][f]);
    __syncthreads();
    for (int i = threadIdx.x; i < S * D; i += blockDim.x) atomicAdd(g_pos + i, (&s_red[0][0])[i]);
}

// second layers of the two heads (transformer_net.py:78-91): logits = W2a ha + b2a, value = W2c hc + b2c; one thread per sample
__global__ void __launch_bounds__(256) head_out_kernel(const bf16 *__restrict__ Ha, const bf16 *__restrict__ Hc, const float *__restrict__ w2a,
                                                       const float *__restrict__ b2a, const float *__restrict__ w2c,
                                                       const float *__restrict__ b2c, int n, float *__restrict__ logits,
                                                       float *__restrict__ value) {
    int b;
    float l0, l1, vv;
    if (!head_out<true>(Ha, Hc, w2a, b2a, w2c, b2c, n, b, l0, l1, vv)) return;
    logits[2 * b] = l0; logits[2 * b + 1] = l1;
    value[b] = vv;
}

// backward of both second head layers and of the ReLU in front of them.  A warp walks a run of samples, lane = 2 of
// the 64 hidden units: dH = (W2^T dout) * (h > 0) goes out as bf16 rows of 128 (columns 64.. stay zero: the weight-
// gradient kernel consumes 128-column blocks); dW2, db2 and db1 (column sums of dH) are reduced in registers.
__global__ void __launch_bounds__(256) head_bwd_kernel(const bf16 *__restrict__ Ha, const bf16 *__restrict__ Hc, const float *__restrict__ w2a,
                                                       const float *__restrict__ w2c, const float *__restrict__ dlogits,
                                                       const float *__restrict__ dvalue, int n, int samples_per_warp,
                                                       bf16 *__restrict__ dHa, bf16 *__restrict__ dHc, float *__restrict__ g_w2a,
                                                       float *__restrict__ g_b2a, float *__restrict__ g_b1a, float *__restrict__ g_w2c,
                                                       float *__restrict__ g_b2c, float *__restrict__ g_b1c) {
    constexpr int kAcc = 10;                               // per lane: 2 x {dW2a row 0, dW2a row 1, dW2c, db1a, db1c}
    __shared__ float s_red[kAcc / 2][HID];
    __shared__ float s_b2[3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (kAcc / 2) * HID; i += blockDim.x) (&s_red[0][0])[i] = 0.0f;
    if (threadIdx.x < 3) s_b2[threadIdx.x] = 0.0f;
    __syncthreads();
    const int gw = blockIdx.x * 8 + warp;
    const int b0 = gw * samples_per_warp, b1 = min(n, b0 + samples_per_warp);
    const int j = lane * 2;
    const float wa0[2] = {w2a[j], w2a[j + 1]}, wa1[2] = {w2a[HID + j], w2a[HID + j + 1]}, wc[2] = {w2c[j], w2c[j + 1]};
    float acc[5][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}, sb[3] = {0, 0, 0};
    for (int b = b0; b < b1; ++b) {
        const float dl0 = dlogits[2 * b], dl1 = dlogits[2 * b + 1], dv = dvalue[b];
        const __nv_bfloat162 ha2 = *reinterpret_cast<const __nv_bfloat162 *>(Ha + (size_t)b * HID + j);
        const __nv_bfloat162 hc2 = *reinterpret_cast<const __nv_bfloat162 *>(Hc + (size_t)b * HID + j);
        const float ha[2] = {__low2float(ha2), __high2float(ha2)}, hc[2] = {__low2float(hc2), __high2float(hc2)};
        float da[2], dc[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            da[k] = ha[k] > 0.0f ? dl0 * wa0[k] + dl1 * wa1[k] : 0.0f;
            dc[k] = hc[k] > 0.0f ? dv * wc[k] : 0.0f;
            acc[0][k] = fmaf(dl0, ha[k], acc[0][k]); acc[1][k] = fmaf(dl1, ha[k], acc[1][k]); acc[2][k] = fmaf(dv, hc[k], acc[2][k]);
            acc[3][k] += da[k]; acc[4][k] += dc[k];
        }
        sb[0] += dl0; sb[1] += dl1; sb[2] += dv;
        *reinterpret_cast<__nv_bfloat162 *>(dHa + (size_t)b * D + j) = __floats2bfloat162_rn(da[0], da[1]);
        *reinterpret_cast<__nv_bfloat162 *>(dHc + (size_t)b * D + j) = __floats2bfloat162_rn(dc[0], dc[1]);
    }
#pragma unroll
    for (int a = 0; a < 5; ++a) { atomicAdd(&s_red[a][j], acc[a][0]); atomicAdd(&s_red[a][j + 1], acc[a][1]); }
    if (lane == 0) { atomicAdd(&s_b2[0], sb[0]); atomicAdd(&s_b2[1], sb[1]); atomicAdd(&s_b2[2], sb[2]); }
    __syncthreads();
    for (int i = threadIdx.x; i < 5 * HID; i += blockDim.x) {
        const int a = i / HID, c = i % HID;
        float *dst = a == 0 ? g_w2a + c : a == 1 ? g_w2a + HID + c : a == 2 ? g_w2c + c : a == 3 ? g_b1a + c : g_b1c + c;
        atomicAdd(dst, s_red[a][c]);
    }
    if (threadIdx.x == 0) { atomicAdd(g_b2a, s_b2[0]); atomicAdd(g_b2a + 1, s_b2[1]); atomicAdd(g_b2c, s_b2[2]); }
}

// PPO loss (agents/ppo.py:126-153) on the heads' outputs, forward and backward in two passes over the minibatch:
//   L = -mean(min(r A, clip(r, 1-eps, 1+eps) A)) + c_v max(mean((v - R)^2), mean((v_clip - R)^2)) - c_e mean(entropy)
// pass 1 accumulates the four sums; pass 2 (which needs the means to pick the value-loss branch torch.max picks)
// writes dL/dlogits and dL/dvalue.  acc: [0] sum -surrogate, [1] sum (v-R)^2, [2] sum (v_clip-R)^2, [3] sum entropy.
struct PpoLossArgs {
    const float *logits, *value, *old_logp, *adv, *ret, *old_value;
    const int64_t *action;
    int n;
    float eps, c_value, c_entropy;
};
__device__ __forceinline__ void ppo_sample(const PpoLossArgs &a, int b, float &lp0, float &lp1, float &ratio, float &adv, float &surr1,
                                           float &surr2, float &ent, float &v, float &vclip, float &ret) {
    const float l0 = a.logits[2 * b], l1 = a.logits[2 * b + 1];
    const float m = fmaxf(l0, l1), lse = m + logf(expf(l0 - m) + expf(l1 - m));
    lp0 = l0 - lse; lp1 = l1 - lse;
    const float p0 = expf(lp0), p1 = expf(lp1);
    ent = -(p0 * lp0 + p1 * lp1);
    const float logp = a.action[b] == 1 ? lp1 : lp0;
    ratio = expf(logp - a.old_logp[b]);
    adv = a.adv[b];
    surr1 = ratio * adv;
    surr2 = fminf(fmaxf(ratio, 1.0f - a.eps), 1.0f + a.eps) * adv;
    v = a.value[b]; ret = a.ret[b];
    const float ov = a.old_value[b];
    vclip = ov + fminf(fmaxf(v - ov, -a.eps), a.eps);
}
__global__ void __launch_bounds__(256) ppo_loss_sums_kernel(const PpoLossArgs a, float *__restrict__ acc) {
    __shared__ float s_red[4][8];
    float s[4] = {0, 0, 0, 0};
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.n; b += gridDim.x * blockDim.x) {
        float lp0, lp1, ratio, adv, s1, s2, ent, v, vc, r;
        ppo_sample(a, b, lp0, lp1, ratio, adv, s1, s2, ent, v, vc, r);
        s[0] -= fminf(s1, s2); s[1] += (v - r) * (v - r); s[2] += (vc - r) * (vc - r); s[3] += ent;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        s[k] = xor_sum<16, 8, 4, 2, 1>(s[k]);
        if ((threadIdx.x & 31) == 0) s_red[k][threadIdx.x >> 5] = s[k];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        float t = 0.0f;
        for (int w = 0; w < 8; ++w) t += s_red[threadIdx.x][w];
        atomicAdd(acc + threadIdx.x, t);
    }
}
__global__ void __launch_bounds__(256) ppo_loss_grad_kernel(const PpoLossArgs a, const float *__restrict__ acc, float *__restrict__ dlogits,
                                                            float *__restrict__ dvalue, float *__restrict__ stats) {
    const float inv_n = 1.0f / (float)a.n;
    const bool clipped_branch = acc[2] > acc[1];          // torch.max(mean1, mean2): the larger mean carries the gradient
    if (blockIdx.x == 0 && threadIdx.x == 0 && stats) {   // the three numbers the reference logs (ppo.py:162-168)
        stats[0] = acc[0] * inv_n; stats[1] = fmaxf(acc[1], acc[2]) * inv_n; stats[2] = acc[3] * inv_n;
    }
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.n) return;
    float lp0, lp1, ratio, adv, s1, s2, ent, v, vc, r;
    ppo_sample(a, b, lp0, lp1, ratio, adv, s1, s2, ent, v, vc, r);
    // d(-min(s1, s2))/d ratio: A where the unclipped term is the minimum or the clamp is inactive, else 0
    const bool inside = ratio >= 1.0f - a.eps && ratio <= 1.0f + a.eps;
    const float dlogp = (s1 < s2 || inside) ? -adv * ratio * inv_n : 0.0f;
    const float p0 = expf(lp0), p1 = expf(lp1);
    const bool a1 = a.action[b] == 1;
    const float ce = a.c_entropy * inv_n;                 // -c_e mean(H):  dH/dz_k = -p_k (log p_k + H)
    dlogits[2 * b] = dlogp * ((a1 ? 0.0f : 1.0f) - p0) + ce * p0 * (lp0 + ent);
    dlogits[2 * b + 1] = dlogp * ((a1 ? 1.0f : 0.0f) - p1) + ce * p1 * (lp1 + ent);
    const float ov = a.old_value[b];
    float dv;
    if (!clipped_branch) dv = 2.0f * (v - r);
    else dv = (v - ov >= -a.eps && v - ov <= a.eps) ? 2.0f * (vc - r) : 0.0f;
    dvalue[b] = a.c_value * dv * inv_n;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------- host side

namespace {
struct LayerT { const bf16 *in_t, *in_q_t, *in_kv_t, *out_t, *l1_t, *l2_t; };          // transposed bf16 GEMM weights
// bf16 forms of one GEMM weight: row-major copy, transpose, and for an in_w the transposes of its Q rows and K / V rows
struct Gemm16 { bf16 *w, *t, *q_t, *kv_t; };
static_assert(kNumGemmW + 2 * 3 <= kMaxPrepJobs, "a conversion job per GEMM weight and two more per in_w (3 layers)");
struct FullAct { bf16 *QKV, *ATT, *XH1, *Y1, *Hf, *XH2, *Xout; float *rstd1, *rstd2; };   // inner layer, R rows
struct LastAct { bf16 *KV, *Q, *AL, *XH1, *Y1, *Hs, *XH2; float *rstd1, *rstd2; };        // last layer
struct HeadT { bf16 *w1, *w1_t; bf16 *Z, *Hh, *dHh; };                                     // bf16 weights, feature / hidden / gradient rows
}  // namespace

struct uavtrain : capi::Handle {
    int max_samples = 0, sms = 0, n = 0;
    bf16 *arena = nullptr;                       // bf16 GEMM weights: row-major copies and transposes
    Gemm16 g16[uavp::kNumGemmW];                 // their slices of the arena, in kGemmW order
    uavp::BlockW actor, critic;                  // fp32 members point into the caller's flat parameter buffer (set per forward)
    uavp::HeadW actor_head, critic_head;         // likewise
    LayerT actor_t[1], critic_t[2];
    HeadT ahead, chead;
    bool with_heads = false;                     // the last forward also ran the heads
    bf16 *Ea, *Ec;
    LastAct la, lc;
    FullAct fc;
    bf16 *T, *T2;                                // forward scratch (GEMM outputs feeding add+LN)
    bf16 *dS1, *dS2, *dH, *dQKV, *dXa, *dXb, *dQ, *tmp;   // backward scratch
    float *zeros = nullptr, *loss_acc = nullptr;
    bf16 *obs16 = nullptr;                       // [R,64] bf16 observations (zero-padded): B operand of the embedding weight gradient
    uint32_t *relu_mask = nullptr;               // [R][2 nets][4 words] ReLU activity bits of the two embeddings
    uint8_t *pad = nullptr;
};

namespace {
struct TCtx { uavtrain *p; cudaStream_t s; int rc; };

void gemm(TCtx &c, const bf16 *A, int64_t lda, const bf16 *W, const float *bias, bf16 *Dst, int M, int N, int K, int relu) {
    if (c.rc) return;
    const int r = uavp::gemm_bias_act(A, lda, W, bias ? bias : c.p->zeros, Dst, M, N, K, relu, c.s);
    if (r) c.rc = fail(c.p, -2, "tcgen05 GEMM (M=%d N=%d K=%d) failed with %d", M, N, K, r);
}
// out = LayerNorm(x + A W^T + bias) fused into the dense kernel's epilogue (policy_dense.cu), keeping x^ and 1/sigma
void gemm_ln(TCtx &c, const bf16 *A, int64_t lda, const bf16 *W, const float *bias, const bf16 *x, int64_t xs, const float *g,
             const float *b, int rows, int K, bf16 *out16, bf16 *xhat, float *rstd) {
    if (c.rc) return;
    const int r = uavp::gemm_add_ln(A, lda, W, bias, x, xs, g, b, out16, xhat, rstd, rows, K, c.s);
    if (r) c.rc = fail(c.p, -2, "tcgen05 GEMM + LayerNorm (M=%d K=%d) failed with %d", rows, K, r);
}
void wgrad(TCtx &c, const bf16 *dY, int64_t ld_dy, const bf16 *X, int64_t ld_x, int rows, int Nout, int Kin, float *dW,
           int nout_valid = -1, float *dbias = nullptr, int out_ld = 0, int kin_valid = 0) {
    if (c.rc) return;
    const int r = uavp::wgrad(dY, ld_dy, X, ld_x, rows, Nout, Kin, dW, nout_valid < 0 ? Nout : nout_valid, dbias, c.p->sms, c.s, out_ld,
                              kin_valid);
    if (r) c.rc = fail(c.p, -2, "weight-gradient kernel (rows=%d Nout=%d Kin=%d) failed with %d", rows, Nout, Kin, r);
}
void add_ln(TCtx &c, const bf16 *x, int64_t xs, const bf16 *y, const float *g, const float *b, int rows, bf16 *out16, float *out32,
            int64_t out32_stride, bf16 *xhat, float *rstd) {
    if (c.rc) return;
    add_ln_train_kernel<<<(rows * 16 + 255) / 256, 256, 0, c.s>>>(x, xs, y, g, b, rows, out16, out32, out32_stride, xhat, rstd);
}
// launch geometry of the "a warp walks consecutive rows" kernels: about 8 CTAs of 8 warps per SM
inline void row_grid(const uavtrain *p, int rows, int &grid, int &rpw) {
    const int warps = p->sms * 8 * 8;
    rpw = (rows + warps - 1) / warps;
    if (rpw < 4) rpw = 4;
    grid = ((rows + rpw - 1) / rpw + 7) / 8;
}
void ln_bwd(TCtx &c, const float *dy32, int64_t dy_stride, const bf16 *dy16, const bf16 *add, const bf16 *xhat, const float *rstd,
            const float *gamma, int rows, bf16 *dz, float *g_gamma, float *g_beta, float *g_bias) {
    if (c.rc) return;
    int grid, rpw;
    row_grid(c.p, rows, grid, rpw);
    if (dy32) ln_bwd_kernel<true><<<grid, 256, 0, c.s>>>(dy32, dy_stride, add, xhat, rstd, gamma, rows, rpw, dz, g_gamma, g_beta, g_bias);
    else ln_bwd_kernel<false><<<grid, 256, 0, c.s>>>(dy16, D, add, xhat, rstd, gamma, rows, rpw, dz, g_gamma, g_beta, g_bias);
}

// ---- forward -----------------------------------------------------------------------------------------------
void last_layer_fwd(TCtx &c, const uavp::LayerW &L, const bf16 *X, int n, LastAct &A, float *feat, int64_t feat_stride, bf16 *feat16) {
    uavtrain *p = c.p;
    const int R = n * S;
    const bf16 *Xl = X + (S - 1) * D;
    gemm(c, X, D, L.in_w + D * D, L.in_b + D, A.KV, R, 2 * D, D, 0);
    gemm(c, Xl, (int64_t)S * D, L.in_w, L.in_b, A.Q, n, D, D, 0);
    if (!c.rc) attn_last_kernel<<<(n * H + 255) / 256, 256, 0, c.s>>>(A.Q, A.KV, p->pad, n, A.AL);
    gemm_ln(c, A.AL, D, L.out_w, L.out_b, Xl, (int64_t)S * D, L.n1_w, L.n1_b, n, D, A.Y1, A.XH1, A.rstd1);
    gemm(c, A.Y1, D, L.l1_w, L.l1_b, A.Hs, n, FF, D, 1);
    gemm(c, A.Hs, FF, L.l2_w, L.l2_b, p->T2, n, D, FF, 0);
    add_ln(c, A.Y1, D, p->T2, L.n2_w, L.n2_b, n, feat16, feat, feat_stride, A.XH2, A.rstd2);
}
void full_layer_fwd(TCtx &c, const uavp::LayerW &L, const bf16 *X, int n, FullAct &A) {
    uavtrain *p = c.p;
    const int R = n * S;
    gemm(c, X, D, L.in_w, L.in_b, A.QKV, R, 3 * D, D, 0);
    if (!c.rc) attn_full_kernel<<<std::min((n + 7) / 8, p->sms * 16), 256, 0, c.s>>>(A.QKV, p->pad, n, A.ATT);
    gemm_ln(c, A.ATT, D, L.out_w, L.out_b, X, D, L.n1_w, L.n1_b, R, D, A.Y1, A.XH1, A.rstd1);
    gemm(c, A.Y1, D, L.l1_w, L.l1_b, A.Hf, R, FF, D, 1);
    gemm_ln(c, A.Hf, FF, L.l2_w, L.l2_b, A.Y1, D, L.n2_w, L.n2_b, R, FF, A.Xout, A.XH2, A.rstd2);
}

// ---- backward ----------------------------------------------------------------------------------------------
// shared tail of both layer kinds: from the gradient of the layer output down to dS1 (gradient of x + attn-proj)
void ffn_ln_bwd(TCtx &c, const uavp::LayerW &L, const LayerT &T, const uavp::LayerOff &o, float *g, int rows, const float *dz32,
                int64_t dz_stride, const bf16 *dz16, const bf16 *XH2, const float *rstd2, const bf16 *Hact, const bf16 *Y1,
                const bf16 *XH1, const float *rstd1) {
    uavtrain *p = c.p;
    ln_bwd(c, dz32, dz_stride, dz16, nullptr, XH2, rstd2, L.n2_w, rows, p->dS2, g + o.n2_w, g + o.n2_b, g + o.l2_b);
    wgrad(c, p->dS2, D, Hact, FF, rows, D, FF, g + o.l2_w);
    if (!c.rc) {                                              // dH = (dS2 W2) masked by the forward's ReLU, in one GEMM
        const int r = uavp::gemm_drelu(p->dS2, D, T.l2_t, Hact, FF, p->dH, rows, FF, D, c.s);
        if (r) c.rc = fail(p, -2, "tcgen05 GEMM with ReLU-backward epilogue (M=%d) failed with %d", rows, r);
    }
    wgrad(c, p->dH, FF, Y1, D, rows, FF, D, g + o.l1_w, -1, g + o.l1_b);                  // + bias gradient dH^T 1
    gemm(c, p->dH, FF, T.l1_t, nullptr, p->tmp, rows, D, FF, 0);
    ln_bwd(c, nullptr, 0, p->tmp, p->dS2, XH1, rstd1, L.n1_w, rows, p->dS1, g + o.n1_w, g + o.n1_b, g + o.out_b);
}
// dX [R,128] <- gradient w.r.t. the layer input (all five tokens)
void last_layer_bwd(TCtx &c, const uavp::LayerW &L, const LayerT &T, const uavp::LayerOff &o, float *g, const bf16 *X, int n, LastAct &A,
                    const float *dfeat, int64_t dfeat_stride, const bf16 *dfeat16, bf16 *dX) {
    uavtrain *p = c.p;
    const int R = n * S;
    ffn_ln_bwd(c, L, T, o, g, n, dfeat, dfeat_stride, dfeat16, A.XH2, A.rstd2, A.Hs, A.Y1, A.XH1, A.rstd1);
    wgrad(c, p->dS1, D, A.AL, D, n, D, D, g + o.out_w);
    gemm(c, p->dS1, D, T.out_t, nullptr, p->tmp, n, D, D, 0);                       // dAL
    if (!c.rc) {
        AttnBwdArgs a{A.Q, A.KV, A.KV + D, p->tmp, p->dQ, p->dQKV, p->dQKV + D, D, 2 * D, p->pad, n};
        attn_bwd_last_kernel<<<(n * H + 255) / 256, 256, 0, c.s>>>(a);
    }
    wgrad(c, p->dQ, D, X + (S - 1) * D, (int64_t)S * D, n, D, D, g + o.in_w, -1, g + o.in_b);          // + bias gradients
    wgrad(c, p->dQKV, 2 * D, X, D, R, 2 * D, D, g + o.in_w + D * D, -1, g + o.in_b + D);
    gemm(c, p->dQKV, 2 * D, T.in_kv_t, nullptr, dX, R, D, 2 * D, 0);
    gemm(c, p->dQ, D, T.in_q_t, nullptr, p->tmp, n, D, D, 0);
    if (!c.rc) scatter_add_last_kernel<<<(n * (D / 4) + 255) / 256, 256, 0, c.s>>>(dX, p->tmp, p->dS1, n);
}
// returns the two addends of the gradient w.r.t. the layer input: dXg (GEMM branch) and p->dS1 (residual branch)
void full_layer_bwd(TCtx &c, const uavp::LayerW &L, const LayerT &T, const uavp::LayerOff &o, float *g, const bf16 *X, int n, FullAct &A,
                    const bf16 *dY, bf16 *dXg) {
    uavtrain *p = c.p;
    const int R = n * S;
    ffn_ln_bwd(c, L, T, o, g, R, nullptr, 0, dY, A.XH2, A.rstd2, A.Hf, A.Y1, A.XH1, A.rstd1);
    wgrad(c, p->dS1, D, A.ATT, D, R, D, D, g + o.out_w);
    gemm(c, p->dS1, D, T.out_t, nullptr, p->tmp, R, D, D, 0);                       // dATT
    if (!c.rc) {
        AttnBwdArgs a{A.QKV, A.QKV + D, A.QKV + 2 * D, p->tmp, p->dQKV, p->dQKV + D, p->dQKV + 2 * D, 3 * D, 3 * D, p->pad, n};
        attn_bwd_full_kernel<<<std::min((n + 7) / 8, p->sms * 16), 256, 0, c.s>>>(a);
    }
    wgrad(c, p->dQKV, 3 * D, X, D, R, 3 * D, D, g + o.in_w, -1, g + o.in_b);                           // + bias gradient
    gemm(c, p->dQKV, 3 * D, T.in_t, nullptr, dXg, R, D, 3 * D, 0);
}
void embed_bwd(TCtx &c, const uavp::NetOff &o, int net, float *g, int n, const bf16 *g1, const bf16 *g2) {
    if (c.rc) return;
    uavtrain *p = c.p;
    int grid, rpw;
    row_grid(p, n, grid, rpw);                                  // (here a "row" is a window of 5 token rows)
    embed_mask_kernel<<<grid, 256, 0, c.s>>>(g1, g2, p->relu_mask + net * 4, n, rpw, p->tmp, g + o.pos);
    wgrad(c, p->tmp, D, p->obs16, 64, n * S, D, 64, g + o.emb_w, -1, g + o.emb_b, F, F);
}
}  // namespace

extern "C" const char *uavtrain_last_error(const uavtrain_t *p) { return capi::last_error(p); }

extern "C" int uavtrain_create(int32_t device, int32_t max_samples, uavtrain_t **out) {
    uavtrain *p;
    if (const int rc = capi::check_create_args("uavtrain_create", "max_samples", max_samples, out)) return rc;
    if (const int rc = capi::new_handle("uavtrain_create", device, p)) return rc;
    p->max_samples = max_samples;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
    const size_t n = (size_t)max_samples, R = n * S;
    if (e == cudaSuccess) e = alloc(p, &p->arena, (size_t)3 * (2 * 3 * D * D + 3 * D * D + 2 * D * D + 4 * FF * D) + 4 * HID * D + 64 * 64);
    bf16 **rowsR128[] = {&p->Ea, &p->Ec, &p->fc.ATT, &p->fc.XH1, &p->fc.Y1, &p->fc.XH2, &p->fc.Xout, &p->T, &p->dS1, &p->dS2, &p->dXa, &p->dXb, &p->tmp};
    for (auto b : rowsR128) if (e == cudaSuccess) e = alloc(p, b, R * D);
    bf16 **rowsR256[] = {&p->la.KV, &p->lc.KV, &p->fc.Hf, &p->dH};
    for (auto b : rowsR256) if (e == cudaSuccess) e = alloc(p, b, R * FF);
    bf16 **rowsR384[] = {&p->fc.QKV, &p->dQKV};
    for (auto b : rowsR384) if (e == cudaSuccess) e = alloc(p, b, R * 3 * D);
    for (LastAct *A : {&p->la, &p->lc}) {
        bf16 **rowsN128[] = {&A->Q, &A->AL, &A->XH1, &A->Y1, &A->XH2};
        for (auto b : rowsN128) if (e == cudaSuccess) e = alloc(p, b, n * D);
        if (e == cudaSuccess) e = alloc(p, &A->Hs, n * FF);
        if (e == cudaSuccess) e = alloc(p, &A->rstd1, n);
        if (e == cudaSuccess) e = alloc(p, &A->rstd2, n);
    }
    for (HeadT *Hd : {&p->ahead, &p->chead}) {
        if (e == cudaSuccess) e = alloc(p, &Hd->Z, n * D);
        if (e == cudaSuccess) e = alloc(p, &Hd->Hh, n * HID);
        if (e == cudaSuccess) e = alloc(p, &Hd->dHh, n * D);
        if (e == cudaSuccess) e = cudaMemset(Hd->dHh, 0, n * D * sizeof(bf16));      // columns 64.. are never written again
    }
    if (e == cudaSuccess) e = alloc(p, &p->T2, n * D);
    if (e == cudaSuccess) e = alloc(p, &p->dQ, n * D);
    if (e == cudaSuccess) e = alloc(p, &p->fc.rstd1, R);
    if (e == cudaSuccess) e = alloc(p, &p->fc.rstd2, R);
    if (e == cudaSuccess) e = alloc(p, &p->pad, R);
    if (e == cudaSuccess) e = alloc(p, &p->loss_acc, (size_t)4);
    if (e == cudaSuccess) e = alloc(p, &p->obs16, R * 64);
    if (e == cudaSuccess) e = alloc(p, &p->relu_mask, R * 8);
    if (e == cudaSuccess) e = alloc(p, &p->zeros, (size_t)3 * D);
    if (e == cudaSuccess) e = cudaMemset(p->zeros, 0, 3 * D * sizeof(float));
    if (e != cudaSuccess) return capi::abandon_handle(p, fail(p, -2, "uavtrain_create: %s", cudaGetErrorString(e)));
    if (uavp::wgrad_prepare() != 0)
        return capi::abandon_handle(p, fail(p, -2, "uavtrain_create: cannot reserve shared memory for the weight-gradient kernel"));
    size_t a = 0;                                               // slices 64-element aligned: TMA tensor maps are built on them
    auto take = [&](size_t elems) { bf16 *q = p->arena + a; a += (elems + 63) / 64 * 64; return q; };
    for (int i = 0; i < kNumGemmW; ++i) {
        const GemmW &g = kGemmW.w[i];
        Gemm16 &G = p->g16[i];
        G.w = take((size_t)g.N * g.K); G.t = take((size_t)g.N * g.K);
        if (g.N == 3 * D) { G.q_t = take(D * D); G.kv_t = take(2 * D * D); }
    }
    auto forms = [&](size_t off) -> const Gemm16 & { int i = 0; while (kGemmW.w[i].off != off) ++i; return p->g16[i]; };
    const NetOff *offs[2] = {&kActorOff, &kCriticOff};
    BlockW *blocks[2] = {&p->actor, &p->critic};
    LayerT *lts[2] = {p->actor_t, p->critic_t};
    HeadT *heads[2] = {&p->ahead, &p->chead};
    for (int k = 0; k < 2; ++k) {
        for (int l = 0; l < offs[k]->layers; ++l) {
            const LayerOff &o = offs[k]->layer[l];
            const Gemm16 &in = forms(o.in_w), &out = forms(o.out_w), &l1 = forms(o.l1_w), &l2 = forms(o.l2_w);
            LayerW &L = blocks[k]->layer[l];
            L.in_w = in.w; L.out_w = out.w; L.l1_w = l1.w; L.l2_w = l2.w;
            lts[k][l] = LayerT{in.t, in.q_t, in.kv_t, out.t, l1.t, l2.t};
        }
        heads[k]->w1 = forms(offs[k]->head.w1).w;
        heads[k]->w1_t = forms(offs[k]->head.w1).t;
    }
    *out = p;
    return 0;
}

extern "C" int uavtrain_destroy(uavtrain_t *p) { return capi::destroy_handle(p); }

namespace {
int forward_impl(uavtrain *p, const float *w, const float *d_obs, int n, float *d_feat, float *d_logits, float *d_value, void *stream) {
    if (n <= 0 || n > p->max_samples) return fail(p, -1, "uavtrain_forward: n=%d outside (0, %d]", n, p->max_samples);
    CU_TRY(p, cudaSetDevice(p->device));
    TCtx c{p, (cudaStream_t)stream, 0};
    const bool heads = d_logits != nullptr;
    p->n = 0;
    bind_fp32(p->actor, p->actor_head, kActorOff, w);
    bind_fp32(p->critic, p->critic_head, kCriticOff, w);
    PrepJobs jobs{};
    int n_jobs = 0;
    for (int i = 0; i < kNumGemmW; ++i) {
        const GemmW &g = kGemmW.w[i];
        const Gemm16 &G = p->g16[i];
        jobs.job[n_jobs++] = PrepJob{w + g.off, G.w, G.t, g.N, g.K};
        if (G.q_t) {
            jobs.job[n_jobs++] = PrepJob{w + g.off, nullptr, G.q_t, D, D};
            jobs.job[n_jobs++] = PrepJob{w + g.off + D * D, nullptr, G.kv_t, 2 * D, D};
        }
    }
    prep_weights_kernel<<<dim3(24, n_jobs), 256, 0, c.s>>>(jobs);
    const int R = n * S;
    embed_kernel<<<(R + kEmbTok - 1) / kEmbTok, kEmbThreads, 0, c.s>>>(d_obs, R, p->actor, p->critic, p->Ea, p->Ec, p->pad, p->obs16, p->relu_mask);
    last_layer_fwd(c, p->actor.layer[0], p->Ea, n, p->la, d_feat, 2 * D, heads ? p->ahead.Z : nullptr);
    full_layer_fwd(c, p->critic.layer[0], p->Ec, n, p->fc);
    last_layer_fwd(c, p->critic.layer[1], p->fc.Xout, n, p->lc, d_feat ? d_feat + D : nullptr, 2 * D, heads ? p->chead.Z : nullptr);
    if (heads) {
        const HeadW &ha = p->actor_head, &hc = p->critic_head;
        gemm(c, p->ahead.Z, D, p->ahead.w1, ha.b1, p->ahead.Hh, n, HID, D, 1);
        gemm(c, p->chead.Z, D, p->chead.w1, hc.b1, p->chead.Hh, n, HID, D, 1);
        if (!c.rc)
            head_out_kernel<<<(n + 255) / 256, 256, 0, c.s>>>(p->ahead.Hh, p->chead.Hh, ha.w2, ha.b2, hc.w2, hc.b2, n, d_logits, d_value);
    }
    if (c.rc) return c.rc;
    CU_TRY(p, cudaGetLastError());
    p->n = n;
    p->with_heads = heads;
    return 0;
}

int backward_impl(uavtrain *p, const float *d_dfeat, const float *d_dlogits, const float *d_dvalue, float *g, void *stream) {
    CU_TRY(p, cudaSetDevice(p->device));
    TCtx c{p, (cudaStream_t)stream, 0};
    const int n = p->n;
    const bool heads = d_dlogits != nullptr;
    CU_TRY(p, cudaMemsetAsync(g, 0, (size_t)UAVPOLICY_NUM_PARAMS * sizeof(float), c.s));
    if (heads) {
        const HeadOff &ao = kActorOff.head, &co = kCriticOff.head;
        const int warps = p->sms * 8 * 4, spw = max(1, (n + warps - 1) / warps);
        head_bwd_kernel<<<((n + spw - 1) / spw + 7) / 8, 256, 0, c.s>>>(
            p->ahead.Hh, p->chead.Hh, p->actor_head.w2, p->critic_head.w2, d_dlogits, d_dvalue, n, spw, p->ahead.dHh, p->chead.dHh,
            g + ao.w2, g + ao.b2, g + ao.b1, g + co.w2, g + co.b2, g + co.b1);
        wgrad(c, p->ahead.dHh, D, p->ahead.Z, D, n, D, D, g + ao.w1, HID);
        wgrad(c, p->chead.dHh, D, p->chead.Z, D, n, D, D, g + co.w1, HID);
        gemm(c, p->ahead.dHh, D, p->ahead.w1_t, nullptr, p->ahead.Z, n, D, HID, 0);      // dZ overwrites Z (no longer needed)
        gemm(c, p->chead.dHh, D, p->chead.w1_t, nullptr, p->chead.Z, n, D, HID, 0);
    }
    // actor: one (last) layer on the embedding
    last_layer_bwd(c, p->actor.layer[0], p->actor_t[0], kActorOff.layer[0], g, p->Ea, n, p->la, heads ? nullptr : d_dfeat, 2 * D,
                   heads ? p->ahead.Z : nullptr, p->dXa);
    embed_bwd(c, kActorOff, 0, g, n, p->dXa, nullptr);
    // critic: last layer, inner layer, embedding
    last_layer_bwd(c, p->critic.layer[1], p->critic_t[1], kCriticOff.layer[1], g, p->fc.Xout, n, p->lc,
                   heads ? nullptr : d_dfeat + D, 2 * D, heads ? p->chead.Z : nullptr, p->dXa);
    full_layer_bwd(c, p->critic.layer[0], p->critic_t[0], kCriticOff.layer[0], g, p->Ec, n, p->fc, p->dXa, p->dXb);
    embed_bwd(c, kCriticOff, 1, g, n, p->dXb, p->dS1);
    if (c.rc) return c.rc;
    CU_TRY(p, cudaGetLastError());
    return 0;
}
}  // namespace

extern "C" int uavtrain_forward(uavtrain_t *p, const float *d_flat_params, const float *d_obs, int32_t n, float *d_feat, void *stream) {
    if (!p) return -1;
    if (!d_flat_params || !d_obs || !d_feat) return fail(p, -1, "uavtrain_forward: NULL argument");
    return forward_impl(p, d_flat_params, d_obs, n, d_feat, nullptr, nullptr, stream);
}

extern "C" int uavtrain_backward(uavtrain_t *p, const float *d_dfeat, float *d_flat_grad, void *stream) {
    if (!p) return -1;
    if (!d_dfeat || !d_flat_grad) return fail(p, -1, "uavtrain_backward: NULL argument");
    if (p->n <= 0 || p->with_heads) return fail(p, -4, "uavtrain_backward without a preceding uavtrain_forward");
    return backward_impl(p, d_dfeat, nullptr, nullptr, d_flat_grad, stream);
}

extern "C" int uavtrain_forward_heads(uavtrain_t *p, const float *d_flat_params, const float *d_obs, int32_t n, float *d_logits,
                                      float *d_value, void *stream) {
    if (!p) return -1;
    if (!d_flat_params || !d_obs || !d_logits || !d_value) return fail(p, -1, "uavtrain_forward_heads: NULL argument");
    return forward_impl(p, d_flat_params, d_obs, n, nullptr, d_logits, d_value, stream);
}

extern "C" int uavtrain_backward_heads(uavtrain_t *p, const float *d_dlogits, const float *d_dvalue, float *d_flat_grad, void *stream) {
    if (!p) return -1;
    if (!d_dlogits || !d_dvalue || !d_flat_grad) return fail(p, -1, "uavtrain_backward_heads: NULL argument");
    if (p->n <= 0 || !p->with_heads) return fail(p, -4, "uavtrain_backward_heads without a preceding uavtrain_forward_heads");
    return backward_impl(p, nullptr, d_dlogits, d_dvalue, d_flat_grad, stream);
}

extern "C" int uavtrain_ppo_loss(uavtrain_t *p, const float *d_logits, const float *d_value, const int64_t *d_action, const float *d_old_logp,
                                 const float *d_adv, const float *d_ret, const float *d_old_value, int32_t n, float eps_clip, float c_value,
                                 float c_entropy, float *d_dlogits, float *d_dvalue, float *d_stats, void *stream) {
    if (!p) return -1;
    if (!d_logits || !d_value || !d_action || !d_old_logp || !d_adv || !d_ret || !d_old_value || !d_dlogits || !d_dvalue || n <= 0)
        return fail(p, -1, "uavtrain_ppo_loss: NULL argument or n <= 0");
    CU_TRY(p, cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    PpoLossArgs a{d_logits, d_value, d_old_logp, d_adv, d_ret, d_old_value, d_action, n, eps_clip, c_value, c_entropy};
    CU_TRY(p, cudaMemsetAsync(p->loss_acc, 0, 4 * sizeof(float), s));
    ppo_loss_sums_kernel<<<min((n + 255) / 256, p->sms * 4), 256, 0, s>>>(a, p->loss_acc);
    ppo_loss_grad_kernel<<<(n + 255) / 256, 256, 0, s>>>(a, p->loss_acc, d_dlogits, d_dvalue, d_stats);
    CU_TRY(p, cudaGetLastError());
    return 0;
}
