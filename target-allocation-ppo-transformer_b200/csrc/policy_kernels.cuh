// policy_kernels.cuh - the hand-written (non-GEMM) kernels of the policy network outside the fused blocks: the weight
// packing of the rollout forward (policy_forward.cu), and the embedding + positions + padding mask and the attention over
// the 5-token window of the PPO update (policy_train.cu).  Internal linkage: each translation unit gets its own copy.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "policy_weights.cuh"

namespace {
using namespace uavp;

// element offset of (row n, column k) in the UMMA canonical K-major order (tcgen05_util.cuh: 8x8 core matrices)
__device__ __forceinline__ int canon_elem(int n, int k, int K) { return (n >> 3) * (K * 8) + (k >> 3) * 64 + (n & 7) * 8 + (k & 7); }

// [128 x 14] fp32 embedding weight -> [128 x 32] bf16, canonical order, the 14 columns duplicated at 0.. and 16..
// columns 14 / 15: the embedding bias as bf16 + rounding remainder (the A operand carries ones in these two columns)
__global__ void emb_w2_kernel(const float *__restrict__ w, const float *__restrict__ b, __nv_bfloat16 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D * 32) return;
    const int d = i / 32, c = i % 32, j = c % 16;
    float v = j < F ? w[d * F + j] : 0.0f;
    if (c == 14) v = b[d];
    if (c == 15) v = b[d] - __bfloat162float(__float2bfloat16(b[d]));
    out[canon_elem(d, c, 32)] = __float2bfloat16(v);
}

// bias [N] fp32 -> [N x 16] bf16 B-operand in canonical order: column 0 = bf16(b), column 1 = b - bf16(b), rest zero
__global__ void pack_bias_kernel(const float *__restrict__ b, __nv_bfloat16 *__restrict__ out, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * 16) return;
    const int n = i / 16, c = i % 16;
    const float hi = __bfloat162float(__float2bfloat16(b[n]));
    out[canon_elem(n, c, 16)] = __float2bfloat16(c == 0 ? hi : (c == 1 ? b[n] - hi : 0.0f));
}

// row-major fp32 [N x K] -> bf16 in canonical order (one bulk TMA copy then stages a whole B operand)
__global__ void pack_canon_kernel(const float *__restrict__ w, __nv_bfloat16 *__restrict__ out, int N, int K) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * K) return;
    out[canon_elem(i / K, i % K, K)] = __float2bfloat16(w[i]);
}

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

__device__ __forceinline__ void load16(const __nv_bfloat16 *p, float *out) {  // 16 bf16 = 32 B
    const uint4 a = reinterpret_cast<const uint4 *>(p)[0], b = reinterpret_cast<const uint4 *>(p)[1];
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162 *>(&w[i]);
        out[2 * i] = __low2float(v); out[2 * i + 1] = __high2float(v);
    }
}
__device__ __forceinline__ void store16(__nv_bfloat16 *p, const float *v) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t *>(&t);
    }
    reinterpret_cast<uint4 *>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
    reinterpret_cast<uint4 *>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
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

// softmax(q k^T / sqrt(16), key padding mask) v for one (sample, head, query): q, and 5 keys / values of 16 dims
__device__ __forceinline__ void attend(const float *q, const __nv_bfloat16 *k0, const __nv_bfloat16 *v0, size_t stride,
                                       const uint8_t *pad, float *out) {
    float sc[S], mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float kk[DH], s = 0.0f;
        load16(k0 + j * stride, kk);
#pragma unroll
        for (int e = 0; e < DH; ++e) s = fmaf(q[e], kk[e], s);
        sc[j] = pad[j] ? -INFINITY : s * 0.25f;
        mx = fmaxf(mx, sc[j]);
    }
    float den = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) { sc[j] = __expf(sc[j] - mx); den += sc[j]; }
    const float inv = 1.0f / den;
#pragma unroll
    for (int e = 0; e < DH; ++e) out[e] = 0.0f;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        float vv[DH];
        load16(v0 + j * stride, vv);
        const float p = sc[j] * inv;
#pragma unroll
        for (int e = 0; e < DH; ++e) out[e] = fmaf(p, vv[e], out[e]);
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
__device__ __forceinline__ float head_sum(float v) {   // sum over the 4 lanes of a head
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}
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
            blk[i][j] = head_sum(fmaf(af[0], bf[j][0], fmaf(af[1], bf[j][1], fmaf(af[2], bf[j][2], af[3] * bf[j][3]))));
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

// last query only (the last encoder layer): Q [B,128], KV [R,256] -> ATT [B,128]; thread = (sample, head)
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

}  // namespace
