// policy_fused.cu - hand-written tcgen05 kernels of the policy forward (sm_100a).  See tcgen05_util.cuh.
#include "uavpolicy_b200.h"

#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "policy_kernels.cuh"
#include "policy_weights.cuh"
#include "tcgen05_util.cuh"

namespace {
using namespace tc;
using namespace uavp;

// ------------------------------------------------------------------------------------------------------------
// Fused encoder blocks, two kernels (fused_body below).  One CTA (16 warps) owns a tile of 128 rows at a time: 25 samples =
// 125 token rows (3 rows of padding make the M = 128 of tcgen05.mma) in the first kernel, the newest-token rows of 128
// samples in the second.  Activations never leave the SM inside a kernel: the layer input X lives in shared memory as a
// UMMA A-operand (canonical K-major tile), each GEMM accumulates in TMEM, the epilogue threads (FOUR per row: TMEM lane =
// row, each thread a quarter of the columns - a warp can only read the 32 TMEM lanes of its quadrant, so the way to
// put more threads on an epilogue is more warps per quadrant) apply ReLU / residual + LayerNorm and write the
// next A-operand back to shared memory.  Weights stream L2 -> shared memory by bulk TMA behind the running epilogue.
//
//   shared memory (215 KB):  sX 32 KB | sQ sK sV 3 x 32 KB (attention output overwrites Q; the FFN hidden tile
//                            [128 x 256] later aliases sQ+sK) | sW 64 KB (one weight matrix at a time; the QKV projection
//                            arrives as Wq|Wk, then Wv) | sB 8 KB + 4 KB: the bias of that matrix as a [N x 16] B operand and
//                            a constant A operand of ones - ONE more k-step per GEMM adds the bias on the tensor core
//                            (bf16 value + rounding remainder in two columns), so no epilogue loads or adds a bias |
//                            11 KB: the LayerNorm / position vectors of both networks, staged once per CTA (warp-uniform
//                            operands of the epilogues: as global loads they kept missing the little L1 that is left)
//   TMEM: 512 columns; Q|K uses [0,256), V [256,384), the other GEMMs [0,256) / [0,128) / [0,64).  TMEM reads are
//   64 B per cycle per SM, so reading a [128 x N] fp32 accumulator costs 8 N cycles - more than its MMAs (4.2 N): wherever
//   a GEMM has independent column blocks (Q|K vs V, the two halves of the FFN hidden layer) the second block's MMAs run
//   under the first block's epilogue.
constexpr int kTileSamples = 25;                                   // 125 valid token rows of the 128
constexpr int kFusedThreads = 512, kColParts = kFusedThreads / 128;   // column parts per row
constexpr uint32_t kTileBytes = 128 * D * 2;                       // a [128 x 128] bf16 canonical tile
// parameter vectors in shared memory (float offsets).  per network: pos | per layer: LayerNorm gamma / beta x 2
// (position rows are kPosStride floats apart: the lanes of a quarter-warp read up to 5 different position rows at the same
// column, and rows a multiple of 128 B apart would put them on the same banks - a 5-way conflict on every 16-byte load)
constexpr int kPosStride = D + 4;
constexpr int kPPos = 0, kPLayer = S * kPosStride, kPLayerSize = 4 * D;
constexpr int kPN1W = 0, kPN1B = D, kPN2W = 2 * D, kPN2B = 3 * D;
constexpr int kPActor = 0, kPActorSize = kPLayer + 1 * kPLayerSize, kPCritic = kPActorSize, kPCriticSize = kPLayer + 2 * kPLayerSize;
static_assert(kPActorSize % 4 == 0 && kPLayer % 4 == 0 && kPLayerSize % 4 == 0, "16-byte loads of the staged vectors");
constexpr uint32_t kWBytes = 64 * 1024;                            // sW: the largest block staged at once (Wq|Wk, W1, W2)
constexpr uint32_t kBBytes = 2 * D * kBiasK * 2;                   // sB: its bias operand, [<= 256 x 16] bf16 (8 KB)
constexpr uint32_t kOnesBytes = 128 * kBiasK * 2;                  // the A operand of the bias k-step: ones in columns 0, 1
constexpr size_t kFusedSmem = 4 * (size_t)kTileBytes + kWBytes + kBBytes + kOnesBytes + (size_t)(kPActorSize + kPCriticSize) * 4;

// issue D[tmem cols 0..N) = A[128 x K] * W[N x K]^T (+ 1 * bias^T) as K/16 (+ 1) k-steps, N <= 256; thread 0 only.
// sBias: the [N x 16] bias operand (or NULL), sOnes: the [128 x 16] A operand with ones in columns 0 and 1
__device__ __forceinline__ void issue_gemm(uint32_t tmem, const unsigned char *sA, const unsigned char *sWt, int N, int K,
                                           uint64_t *mbar, const unsigned char *sBias = nullptr, const unsigned char *sOnes = nullptr) {
    const uint32_t sbo = (uint32_t)K * 16, idesc = instr_desc_bf16(128, N);
    for (int j = 0; j < K / 16; ++j)
        mma_bf16(tmem, smem_desc(smem_u32(sA) + j * 256, 128, sbo), smem_desc(smem_u32(sWt) + j * 256, 128, sbo), idesc, j > 0);
    if (sBias) mma_bf16(tmem, smem_desc(smem_u32(sOnes), 128, kBiasK * 16), smem_desc(smem_u32(sBias), 128, kBiasK * 16), idesc, 1);
    mma_commit(mbar);
}

// a weight matrix and its bias operand land on ONE mbarrier phase (one arrival, the sum of the bytes)
__device__ __forceinline__ void bulk_load2(void *s0, const void *g0, uint32_t b0, void *s1, const void *g1, uint32_t b1, uint64_t *mbar) {
    mbar_expect_tx(mbar, b0 + b1);
    bulk_copy(s0, g0, b0, mbar);
    bulk_copy(s1, g1, b1, mbar);
}

// Epilogues run on all 16 warps: warp w reads TMEM lanes 32*(w%4).. (its rows) and the column quarter w/4.


// Column parameters (gamma, beta, positions) are the same for every row: warp-uniform (broadcast) loads from the staged copy
// in shared memory, issued BEFORE the TMEM load (or the barrier) an epilogue has to wait for anyway; packed fp32x2 arithmetic.
// The biases are already in the accumulators (bias k-step of issue_gemm).
__device__ __forceinline__ void load_cols32(const float *p, float2 *o) {   // p: shared memory, 16 B aligned
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 q = reinterpret_cast<const float4 *>(p)[i];
        o[2 * i] = make_float2(q.x, q.y); o[2 * i + 1] = make_float2(q.z, q.w);
    }
}

// plain layer: out = act(acc) -> bf16; column c goes to tile (c / tile_cols) of dst, canonical row length Kout
__device__ __forceinline__ void epilogue_act(uint32_t tmem_lane, int row, int c_begin, int c_end, bool relu, unsigned char *dst,
                                             int Kout, int tile_cols) {
    for (int c0 = c_begin; c0 < c_end; c0 += 32) {
        float v[32];
        tmem_ld32(tmem_lane + c0, v);
        if (relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
        }
        unsigned char *tile = dst + (c0 / tile_cols) * kTileBytes;
#pragma unroll
        for (int g = 0; g < 4; ++g)
            *reinterpret_cast<uint4 *>(tile + canon_off(row, (c0 % tile_cols) + g * 8, Kout)) = pack8(v + g * 8);
    }
}

// residual layer: X[row] <- LayerNorm(X[row] + acc) * g + beta (post-LN, eps 1e-5), in place.  The four column
// quarters of a row exchange their partial sums through shared memory (all threads call: contains a CTA barrier).
__device__ __forceinline__ void epilogue_residual_ln(uint32_t tmem_lane, int row, int part, const float *g, const float *beta,
                                                     unsigned char *sX, float2 (*s_part)[128]) {
    constexpr int W = D / kColParts;              // 32 columns per thread
    static_assert(W == 32, "one tcgen05.ld of 32 columns per thread");
    const int c0 = part * W;
    uint4 xr[4];
#pragma unroll
    for (int gch = 0; gch < 4; ++gch) xr[gch] = *reinterpret_cast<const uint4 *>(sX + canon_off(row, c0 + gch * 8, D));
    float t[W];
    tmem_ld32(tmem_lane + c0, t);
    float2 s2 = make_float2(0.0f, 0.0f), q2 = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int gch = 0; gch < 4; ++gch) {
        float x[8];
        unpack8(xr[gch], x);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = gch * 8 + 2 * i;
            const float2 u = __fadd2_rn(make_float2(t[c], t[c + 1]), make_float2(x[2 * i], x[2 * i + 1]));
            t[c] = u.x; t[c + 1] = u.y;
            s2 = __fadd2_rn(s2, u); q2 = __ffma2_rn(u, u, q2);
        }
    }
    s_part[part][row] = make_float2(s2.x + s2.y, q2.x + q2.y);
    float2 p[16];
    load_cols32(g + c0, p);                        // gamma arrives while the CTA meets at the barrier
    __syncthreads();
    float sum = 0.0f, sq = 0.0f;
#pragma unroll
    for (int q = 0; q < kColParts; ++q) { const float2 p2 = s_part[q][row]; sum += p2.x; sq += p2.y; }
    const float mean = sum * (1.0f / D);
    const float rstd = rsqrtf(fmaxf(sq * (1.0f / D) - mean * mean, 0.0f) + 1e-5f);
    const float2 a2 = make_float2(rstd, rstd), m2 = make_float2(-mean * rstd, -mean * rstd);
#pragma unroll
    for (int i = 0; i < 16; ++i) p[i] = __fmul2_rn(__ffma2_rn(make_float2(t[2 * i], t[2 * i + 1]), a2, m2), p[i]);   // x^ * gamma
    float2 be[16];
    load_cols32(beta + c0, be);
#pragma unroll
    for (int gch = 0; gch < 4; ++gch) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 u = __fadd2_rn(p[gch * 4 + i], be[gch * 4 + i]);
            o[2 * i] = u.x; o[2 * i + 1] = u.y;
        }
        *reinterpret_cast<uint4 *>(sX + canon_off(row, c0 + gch * 8, D)) = pack8(o);
    }
}

// one observation row (a token) of tile row r, zero beyond the batch
__device__ __forceinline__ void load_obs_row(const float *__restrict__ obs, int s0, int nrows, int r, float *o) {
    const bool valid = r < nrows;
#pragma unroll
    for (int j = 0; j < 16; ++j) o[j] = (valid && j < F) ? __ldg(obs + ((size_t)s0 * S + r) * F + j) : 0.0f;
}

__device__ __forceinline__ void stage_vec(float *dst, const float *__restrict__ src, int n, int tid) {
    for (int i = tid; i < n; i += kFusedThreads) dst[i] = __ldg(src + i);
}
__device__ __forceinline__ void stage_params(float *dst, const BlockW &w, int tid) {
    for (int i = tid; i < S * D; i += kFusedThreads) dst[kPPos + (i / D) * kPosStride + i % D] = __ldg(w.pos + i);
    for (int l = 0; l < w.layers; ++l) {
        float *d = dst + kPLayer + l * kPLayerSize;
        const LayerW &L = w.layer[l];
        stage_vec(d + kPN1W, L.n1_w, D, tid); stage_vec(d + kPN1B, L.n1_b, D, tid);
        stage_vec(d + kPN2W, L.n2_w, D, tid); stage_vec(d + kPN2B, L.n2_b, D, tid);
    }
}

constexpr int kGroupRows = 128;   // samples per work item of the second kernel (one full M = 128 tile of newest-token rows)

// Both kernels of the forward share this body (kPhase picks the work loop):
//   phase 0 (fused_tiles_kernel)  work item = (network, tile of 25 samples = 125 token rows): embedding, the critic's inner
//            layer, and of the LAST layer the QKV projection and the attention of the newest token of each sample - all that
//            is consumed of it (transformer_net.py:106).  The 25 newest-token rows (attention output, and the layer input =
//            residual) go to a compact [samples x 128] bf16 scratch in canonical tile order (L2-resident).
//   phase 1 (fused_heads_kernel)  work item = (network, 128 samples): the rest of the last layer - out-proj, LayerNorm1, FFN,
//            LayerNorm2 - and the head's first layer, on FULL M = 128 tiles of those rows, bulk-copied from the scratch.
// So the four fifths of a last layer that a tile-at-a-time kernel spends on rows nobody reads are not computed, every
// product of phase 1 runs on a full tile, and its weights stream once per 128 samples instead of once per 25.
template <int kPhase>
__device__ __forceinline__ void fused_body(const float *__restrict__ obs, int B, const BlockW &w_actor, const HeadW &head_actor,
                                           __nv_bfloat16 *__restrict__ hh_actor, const BlockW &w_critic, const HeadW &head_critic,
                                           __nv_bfloat16 *__restrict__ hh_critic, int *__restrict__ work_counter,
                                           unsigned char *__restrict__ scratch) {
    extern __shared__ __align__(1024) unsigned char smem[];
    // MMA completion (two in flight) / weight staging by bulk TMA (wbar: the matrix in sW; ebar: the embedding operand in sK
    // resp. the compact tiles of phase 1, in flight together with the first matrix)
    __shared__ uint64_t mbar, mbar2, wbar, ebar;
    __shared__ uint32_t tmem_base_s;
    __shared__ int s_item[2];                             // this work item / the next one (fetched a whole item ahead)
    __shared__ uint8_t s_pad[128];
    unsigned char *sX = smem, *sQ = smem + kTileBytes, *sK = sQ + kTileBytes, *sV = sK + kTileBytes;
    unsigned char *sH = sQ;                               // [128 x 256] canonical, aliases sQ + sK after attention
    unsigned char *sW = smem + 4 * kTileBytes;
    unsigned char *sB = sW + kWBytes, *sOnes = sB + kBBytes;
    float *const sP = reinterpret_cast<float *>(sOnes + kOnesBytes);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // LayerNorm partial sums {sum, sum of squares} per (column part, row): 4 KB at the start of sV, which is idle in both
    // residual epilogues (after the attention has consumed V; before the next V epilogue rewrites it)
    float2 (*s_part)[128] = reinterpret_cast<float2 (*)[128]>(sV);
    const int row = tid & 127, part = warp >> 2;          // thread = (row, column quarter); TMEM lane = row
    const int num_tiles = (B + kTileSamples - 1) / kTileSamples, num_groups = (B + kGroupRows - 1) / kGroupRows;
    const int num_items = 2 * (kPhase == 0 ? num_tiles : num_groups);
    // compact scratch: per network the attention outputs, then the residual rows, of every 128 samples as one canonical tile
    unsigned char *const scr_critic = scratch, *const scr_actor = scratch + (size_t)2 * num_groups * kTileBytes;
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        mbar_init(&mbar, 1); mbar_init(&mbar2, 1); mbar_init(&wbar, 1); mbar_init(&ebar, 1); fence_mbar_init();
        s_item[0] = atomicAdd(work_counter, 1);
    }
    stage_params(sP + kPActor, w_actor, tid);
    stage_params(sP + kPCritic, w_critic, tid);
    if (tid < 256) {   // the ones operand, canonical [128 x 16]: 16-byte chunk = (8-row group, k half, row); 1.0 at k = 0, 1
        const int kh = (tid >> 3) & 1;
        *reinterpret_cast<uint4 *>(sOnes + (tid >> 4) * 256 + kh * 128 + (tid & 7) * 16) = make_uint4(kh ? 0u : 0x3F803F80u, 0u, 0u, 0u);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const uint32_t tmem_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    // programmatic dependent launch: the second kernel's CTAs may start (on SMs the first kernel has left) and run the
    // prologue above while the first kernel's last work items are still running; they wait HERE for its completion and the
    // visibility of its scratch writes
    if constexpr (kPhase == 0) asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    else asm volatile("griddepcontrol.wait;\n" ::: "memory");
    uint32_t parity = 0, parity2 = 0, wparity = 0, eparity = 0;
    int cur = 0;
    float o[16];                                          // this thread's observation row (tid < 128), fetched ahead of its use
    bool have_obs = false;

    // ---- embedding of the 128 staged rows: X = relu(obs W^T + b) + pos (transformer_net.py:24-30,57-59) -> sX.
    //      On the tensor cores with K = 32: the fp32 observation row is split into bf16 hi + lo parts (columns 0..13 and
    //      16..29) against the weight duplicated in both halves, so the product keeps ~16 mantissa bits of the input; columns
    //      14 / 15 are ones against the bias.  A operand: this thread's row o[] -> sV; B operand: emb_w2p -> sK (bulk TMA).
    //      position < 0: token r sits at position r % S of its window ----
    auto embed_rows = [&](const BlockW &w, const float *pw, int nvalid, int position) {
        if (tid < 128) {
            float hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                hi[j] = __bfloat162float(__float2bfloat16(o[j]));
                lo[j] = o[j] - hi[j];
            }
            hi[14] = 1.0f; hi[15] = 1.0f;            // against the bias columns of emb_w2p
            *reinterpret_cast<uint4 *>(sV + canon_off(tid, 0, 32)) = pack8(hi);
            *reinterpret_cast<uint4 *>(sV + canon_off(tid, 8, 32)) = pack8(hi + 8);
            *reinterpret_cast<uint4 *>(sV + canon_off(tid, 16, 32)) = pack8(lo);
            *reinterpret_cast<uint4 *>(sV + canon_off(tid, 24, 32)) = pack8(lo + 8);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        mbar_wait(&ebar, eparity); eparity ^= 1;
        if (tid == 0) issue_gemm(tmem, sV, sK, D, 32, &mbar);
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        {
            const bool valid = row < nvalid;
            const int c0 = part * 32;
            float2 ep[16];
            load_cols32(pw + kPPos + (position < 0 ? row % S : position) * kPosStride + c0, ep);
            float v[32];
            tmem_ld32(tmem_lane + c0, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float2 u = __fadd2_rn(make_float2(fmaxf(v[2 * i], 0.0f), fmaxf(v[2 * i + 1], 0.0f)), ep[i]);
                v[2 * i] = valid ? u.x : 0.0f; v[2 * i + 1] = valid ? u.y : 0.0f;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4 *>(sX + canon_off(row, c0 + g * 8, D)) = pack8(v + g * 8);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
    };

    // ---- Q|K = X [Wq|Wk]^T (N = 256), then V = X Wv^T (N = 128) under the K epilogue -> sQ | sK | sV, and the attention over the
    //      5-token window (its output overwrites the Q rows).  all_queries: every token is a query (an inner layer); otherwise
    //      only the newest token of a sample (transformer_net.py:106).  next_w / next_b: the matrix (and bias operand) to stream
    //      into sW once V's MMAs have retired, or NULL ----
    auto qkv_attention = [&](const LayerW &L, int nsamp, bool all_queries, const __nv_bfloat16 *next_w, uint32_t next_w_bytes,
                             const __nv_bfloat16 *next_b, uint32_t next_b_bytes) {
        tc_fence_after();
        mbar_wait(&wbar, wparity); wparity ^= 1;                      // Wq|Wk has landed in sW
        if (tid == 0) issue_gemm(tmem, sX, sW, 2 * D, D, &mbar, sB, sOnes);
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        if (tid == 0) bulk_load2(sW, L.in_wp + 2 * D * D, D * D * 2, sB, L.in_bp + 2 * D * kBiasK, D * kBiasK * 2, &wbar);   // Wv (rows 256..383)
        epilogue_act(tmem_lane, row, part * 32, part * 32 + 32, false, sQ, D, D);
        mbar_wait(&wbar, wparity); wparity ^= 1;                      // Wv has landed
        if (tid == 0) issue_gemm(tmem + 2 * D, sX, sW, D, D, &mbar, sB, sOnes);
        epilogue_act(tmem_lane, row, D + part * 32, D + part * 32 + 32, false, sQ, D, D);
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        if (tid == 0 && next_w) bulk_load2(sW, next_w, next_w_bytes, sB, next_b, next_b_bytes, &wbar);
        epilogue_act(tmem_lane, row, 2 * D + part * 32, 2 * D + part * 32 + 32, false, sQ, D, D);
        tc_fence_before();
        __syncthreads();
        // A warp takes a (query, head) pair and its lanes the samples: the 8 lanes of a quarter-warp then read 8 different rows
        // (5 is odd: row & 7 distinct) of the same 16-byte column chunk - conflict-free.  (One thread per (sample, head, query)
        // in flat order put the heads of a sample, 256 B apart, on the same banks: 8-way conflicts on every access; dense
        // packing of the 1000 items of an inner layer over the 512 threads measured slower than the three rounds here.)
        const int npair = (all_queries ? S : 1) * H;
        for (int pair = warp; pair < npair; pair += kFusedThreads / 32) {
            const int h = pair % H, i = all_queries ? pair / H : S - 1;
            if (lane < nsamp) {
                const int smp = lane, r = smp * S + i;
                unsigned char *pq = sQ + canon_off(r, h * DH, D);
                float2 q2[8];
                {
                    float q[DH];
                    unpack8(*reinterpret_cast<const uint4 *>(pq), q);
                    unpack8(*reinterpret_cast<const uint4 *>(pq + 128), q + 8);
#pragma unroll
                    for (int e = 0; e < 8; ++e) q2[e] = make_float2(q[2 * e], q[2 * e + 1]);
                }
                float sc[S], mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    float kk[DH];
                    const unsigned char *pk = sK + canon_off(smp * S + j, h * DH, D);
                    unpack8(*reinterpret_cast<const uint4 *>(pk), kk);
                    unpack8(*reinterpret_cast<const uint4 *>(pk + 128), kk + 8);
                    float2 acc = make_float2(0.0f, 0.0f), acc1 = make_float2(0.0f, 0.0f);
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        acc = __ffma2_rn(q2[e], make_float2(kk[2 * e], kk[2 * e + 1]), acc);
                        acc1 = __ffma2_rn(q2[e + 1], make_float2(kk[2 * e + 2], kk[2 * e + 3]), acc1);
                    }
                    const float sdot = (acc.x + acc.y) + (acc1.x + acc1.y);
                    sc[j] = s_pad[smp * S + j] ? -INFINITY : sdot * 0.25f;
                    mx = fmaxf(mx, sc[j]);
                }
                float den = 0.0f;
#pragma unroll
                for (int j = 0; j < S; ++j) { sc[j] = __expf(sc[j] - mx); den += sc[j]; }
                const float inv = 1.0f / den;
                float2 o2[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) o2[e] = make_float2(0.0f, 0.0f);
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    float vv[DH];
                    const unsigned char *pv = sV + canon_off(smp * S + j, h * DH, D);
                    unpack8(*reinterpret_cast<const uint4 *>(pv), vv);
                    unpack8(*reinterpret_cast<const uint4 *>(pv + 128), vv + 8);
                    const float pj = sc[j] * inv;
                    const float2 pj2 = make_float2(pj, pj);
#pragma unroll
                    for (int e = 0; e < 8; ++e) o2[e] = __ffma2_rn(pj2, make_float2(vv[2 * e], vv[2 * e + 1]), o2[e]);
                }
                float ov[DH];
#pragma unroll
                for (int e = 0; e < 8; ++e) { ov[2 * e] = o2[e].x; ov[2 * e + 1] = o2[e].y; }
                *reinterpret_cast<uint4 *>(pq) = pack8(ov);
                *reinterpret_cast<uint4 *>(pq + 128) = pack8(ov + 8);
            }
        }
        fence_async_smem();
        __syncthreads();
    };

    // ---- the rest of an encoder layer on the rows of sQ (attention output) and sX (layer input = residual): out-proj +
    //      LayerNorm1, FFN (hidden layer as two column halves: the second half's MMAs run under the first half's epilogue),
    //      LayerNorm2 - in place in sX.  Out-proj weights are in flight on wbar; next_w / next_b follow W2 ----
    auto post_attention = [&](const LayerW &L, const float *pl, const __nv_bfloat16 *next_w, uint32_t next_w_bytes,
                              const __nv_bfloat16 *next_b, uint32_t next_b_bytes) {
        tc_fence_after();
        mbar_wait(&wbar, wparity); wparity ^= 1;
        if (tid == 0) issue_gemm(tmem, sQ, sW, D, D, &mbar, sB, sOnes);
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        if (tid == 0) bulk_load2(sW, L.l1_wp, FF * D * 2, sB, L.l1_bp, FF * kBiasK * 2, &wbar);
        epilogue_residual_ln(tmem_lane, row, part, pl + kPN1W, pl + kPN1B, sX, s_part);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        mbar_wait(&wbar, wparity); wparity ^= 1;
        if (tid == 0) {
            issue_gemm(tmem, sX, sW, FF / 2, D, &mbar, sB, sOnes);
            issue_gemm(tmem + FF / 2, sX, sW + (FF / 2) * D * 2, FF / 2, D, &mbar2, sB + (FF / 2) * kBiasK * 2, sOnes);
        }
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        epilogue_act(tmem_lane, row, part * 32, part * 32 + 32, true, sH, FF, FF);
        mbar_wait(&mbar2, parity2); parity2 ^= 1;
        tc_fence_after();
        if (tid == 0) bulk_load2(sW, L.l2_wp, D * FF * 2, sB, L.l2_bp, D * kBiasK * 2, &wbar);
        epilogue_act(tmem_lane, row, FF / 2 + part * 32, FF / 2 + part * 32 + 32, true, sH, FF, FF);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        mbar_wait(&wbar, wparity); wparity ^= 1;
        if (tid == 0) issue_gemm(tmem, sH, sW, D, FF, &mbar, sB, sOnes);
        mbar_wait(&mbar, parity); parity ^= 1;
        tc_fence_after();
        if (tid == 0) bulk_load2(sW, next_w, next_w_bytes, sB, next_b, next_b_bytes, &wbar);
        epilogue_residual_ln(tmem_lane, row, part, pl + kPN2W, pl + kPN2B, sX, s_part);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
    };

    // Work items are handed out dynamically; the two-layer critic items come first (longest first)
    for (;;) {
        const int item = s_item[cur];
        if (item >= num_items) break;
        if (tid == 0) s_item[cur ^ 1] = atomicAdd(work_counter, 1);   // read after the barriers of this item
        const bool is_critic = item < num_items / 2;
        const BlockW &w = is_critic ? w_critic : w_actor;
        const HeadW &head = is_critic ? head_critic : head_actor;
        const float *const pw = sP + (is_critic ? kPCritic : kPActor);
        const LayerW &LL = w.layer[w.layers - 1];                     // the last layer
        unsigned char *const scr_attn = is_critic ? scr_critic : scr_actor, *const scr_res = scr_attn + (size_t)num_groups * kTileBytes;
        if constexpr (kPhase == 0) {
            const int tile = is_critic ? item : item - num_tiles;
            const int s0 = tile * kTileSamples;
            const int nsamp = min(kTileSamples, B - s0), nrows = nsamp * S;
            if (tid == 0) {   // sW / sB are free since the previous item's last MMAs retired: Wq|Wk has the whole embedding to land
                bulk_load(sK, w.emb_w2p, D * 32 * 2, &ebar);              // embedding weights (B operand, K = 32)
                bulk_load2(sW, w.layer[0].in_wp, 2 * D * D * 2, sB, w.layer[0].in_bp, 2 * D * kBiasK * 2, &wbar);
            }
            if (tid < 128) {   // this tile's token rows (fetched ahead, normally) and the key-padding mask (transformer_net.py:52-54)
                if (!have_obs) load_obs_row(obs, s0, nrows, tid, o);
                float asum = 0.0f;
#pragma unroll
                for (int j = 0; j < 16; ++j) asum += fabsf(o[j]);
                s_pad[tid] = (tid < nrows && asum == 0.0f && tid % S != S - 1) ? 1 : 0;
            }
            embed_rows(w, pw, nrows, -1);
            {   // the next work item's token rows arrive under this item's layers
                const int next = s_item[cur ^ 1];
                have_obs = next < num_items;
                if (have_obs && tid < 128) {
                    const int ns0 = (next < num_tiles ? next : next - num_tiles) * kTileSamples;
                    load_obs_row(obs, ns0, min(kTileSamples, B - ns0) * S, tid, o);
                }
            }
            if (is_critic) {   // the critic's inner layer: every token is a query; Wq|Wk of the last layer follows W2
                qkv_attention(w.layer[0], nsamp, true, w.layer[0].out_wp, D * D * 2, w.layer[0].out_bp, D * kBiasK * 2);
                post_attention(w.layer[0], pw + kPLayer, LL.in_wp, 2 * D * D * 2, LL.in_bp, 2 * D * kBiasK * 2);
            }
            qkv_attention(LL, nsamp, false, nullptr, 0, nullptr, 0);
            // the newest-token rows of this tile -> compact scratch (canonical order inside the 128-sample tile they belong to)
            if (row < nrows && row % S == S - 1) {
                const int gs = s0 + row / S, cr = gs & (kGroupRows - 1);
                unsigned char *ga = scr_attn + (size_t)(gs / kGroupRows) * kTileBytes, *gr = scr_res + (size_t)(gs / kGroupRows) * kTileBytes;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const int c = part * 32 + g * 8;
                    *reinterpret_cast<uint4 *>(ga + canon_off(cr, c, D)) = *reinterpret_cast<const uint4 *>(sQ + canon_off(row, c, D));
                    *reinterpret_cast<uint4 *>(gr + canon_off(cr, c, D)) = *reinterpret_cast<const uint4 *>(sX + canon_off(row, c, D));
                }
            }
            __syncthreads();   // sX / sQ / sK are rewritten by the next item's staging
        } else {
            const int group = is_critic ? item : item - num_groups;
            const int g0 = group * kGroupRows, nvalid = min(kGroupRows, B - g0);
            const float *const pll = pw + kPLayer + (w.layers - 1) * kPLayerSize;
            __nv_bfloat16 *head_hidden = is_critic ? hh_critic : hh_actor;
            if (tid == 0) {   // the 128 attention-output rows -> sQ (A operand of the out-proj), their residual rows -> sX
                bulk_load2(sQ, scr_attn + (size_t)group * kTileBytes, kTileBytes, sX, scr_res + (size_t)group * kTileBytes, kTileBytes, &ebar);
                bulk_load2(sW, LL.out_wp, D * D * 2, sB, LL.out_bp, D * kBiasK * 2, &wbar);
            }
            mbar_wait(&ebar, eparity); eparity ^= 1;
            post_attention(LL, pll, head.w1p, HID * D * 2, head.b1p, HID * kBiasK * 2);
            // ---- head first layer: relu(W1 z + b1) (transformer_net.py:106-108) ----
            tc_fence_after();
            mbar_wait(&wbar, wparity); wparity ^= 1;
            if (tid == 0) issue_gemm(tmem, sX, sW, HID, D, &mbar, sB, sOnes);
            mbar_wait(&mbar, parity); parity ^= 1;
            tc_fence_after();
            if (part < HID / 32) {
                __nv_bfloat16 *dst = head_hidden + (size_t)(g0 + row) * HID;
                const int c0 = part * 32;
                float v[32];
                tmem_ld32(tmem_lane + c0, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
                if (row < nvalid) {
#pragma unroll
                    for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4 *>(dst + c0 + g * 8) = pack8(v + g * 8);
                }
            }
            tc_fence_before();
            __syncthreads();
        }
        cur ^= 1;
    }
    if (warp == 0) tmem_free(tmem, 512);
}

__global__ void __launch_bounds__(kFusedThreads, 1)
fused_tiles_kernel(const float *__restrict__ obs, int B, BlockW w_actor, HeadW head_actor, __nv_bfloat16 *__restrict__ hh_actor,
                   BlockW w_critic, HeadW head_critic, __nv_bfloat16 *__restrict__ hh_critic, int *__restrict__ work_counter,
                   unsigned char *__restrict__ scratch) {
    fused_body<0>(obs, B, w_actor, head_actor, hh_actor, w_critic, head_critic, hh_critic, work_counter, scratch);
}
__global__ void __launch_bounds__(kFusedThreads, 1)
fused_heads_kernel(const float *__restrict__ obs, int B, BlockW w_actor, HeadW head_actor, __nv_bfloat16 *__restrict__ hh_actor,
                   BlockW w_critic, HeadW head_critic, __nv_bfloat16 *__restrict__ hh_critic, int *__restrict__ work_counter,
                   unsigned char *__restrict__ scratch) {
    fused_body<1>(obs, B, w_actor, head_actor, hh_actor, w_critic, head_critic, hh_critic, work_counter, scratch);
}

// actor-only forward: both work counters start at the first actor item (items are numbered critic first), so the kernels
// above run the actor's items only and never write hh_critic
__global__ void start_counters_kernel(int *__restrict__ work_counters, int first0, int first1) {
    work_counters[0] = first0;
    work_counters[1] = first1;
}

// self-test: D[128,N] (fp32) = A[128,K] W[N,K]^T with one CTA: canonical smem operands, K/16 tcgen05.mma steps
// (N = 384 as a 256 + 128 pair), accumulator read back from TMEM.  Validates descriptors and the TMEM lane mapping.
__global__ void __launch_bounds__(128) gemm_tile_selftest_kernel(const __nv_bfloat16 *A, const __nv_bfloat16 *W, float *D,
                                                                  int N, int K) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t mbar;
    __shared__ uint32_t tmem_base_s;
    unsigned char *sA = smem, *sW = smem + 128 * K * 2;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) { mbar_init(&mbar, 1); fence_mbar_init(); }
    load_canon(sA, A, 128, K, K, 128, tid, 128);
    load_canon(sW, W, N, K, K, N, tid, 128);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    if (tid == 0) {
        const uint32_t sbo = (uint32_t)K * 16;
        for (int j = 0; j < K / 16; ++j) {
            const uint64_t ad = smem_desc(smem_u32(sA) + j * 256, 128, sbo);
            for (int n0 = 0; n0 < N; n0 += 256) {
                const int nn = min(256, N - n0);
                const uint64_t bd = smem_desc(smem_u32(sW) + (n0 >> 3) * sbo + j * 256, 128, sbo);
                mma_bf16(tmem + n0, ad, bd, instr_desc_bf16(128, nn), j > 0);
            }
        }
        mma_commit(&mbar);
    }
    mbar_wait(&mbar, 0);
    tc_fence_after();
    const int row = warp * 32 + lane;
    for (int c0 = 0; c0 < N; c0 += 32) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
        for (int i = 0; i < 32; ++i) D[(size_t)row * N + c0 + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 512);
}
}  // namespace

namespace uavp {
int fused_block_prepare() {
    return cudaFuncSetAttribute(fused_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFusedSmem) == cudaSuccess &&
                   cudaFuncSetAttribute(fused_heads_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFusedSmem) == cudaSuccess
               ? 0 : -2;
}
size_t fused_scratch_bytes(int max_batch) { return (size_t)4 * ((max_batch + kGroupRows - 1) / kGroupRows) * kTileBytes; }
int launch_fused_blocks(const float *d_obs, int B, const BlockW &actor, const HeadW &actor_head, __nv_bfloat16 *hh_actor,
                        const BlockW &critic, const HeadW &critic_head, __nv_bfloat16 *hh_critic, int *d_work_counters,
                        unsigned char *d_scratch, cudaStream_t stream, bool actor_only) {
    static int num_sms = 0;                       // one persistent CTA per SM of the device
    if (num_sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -2;
    }
    if (actor.layers != 1 || critic.layers != 2) return -1;   // the kernels' item structure (and their staged parameter layout)
    const int num_tiles = (B + kTileSamples - 1) / kTileSamples, num_groups = (B + kGroupRows - 1) / kGroupRows;
    // items still to hand out per launch: both networks', or the actor's (the second half) alone
    const int items0 = actor_only ? num_tiles : 2 * num_tiles, items1 = actor_only ? num_groups : 2 * num_groups;
    if (actor_only) {
        start_counters_kernel<<<1, 1, 0, stream>>>(d_work_counters, num_tiles, num_groups);
        if (cudaGetLastError() != cudaSuccess) return -2;
    } else if (cudaMemsetAsync(d_work_counters, 0, 2 * sizeof(int), stream) != cudaSuccess) return -2;
    fused_tiles_kernel<<<items0 < num_sms ? items0 : num_sms, kFusedThreads, kFusedSmem, stream>>>(
        d_obs, B, actor, actor_head, hh_actor, critic, critic_head, hh_critic, d_work_counters, d_scratch);
    {   // launched as a programmatic dependent of the first kernel (griddepcontrol.wait in its prologue)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(items1 < num_sms ? items1 : num_sms); cfg.blockDim = dim3(kFusedThreads);
        cfg.dynamicSmemBytes = kFusedSmem; cfg.stream = stream;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        int *ctr = d_work_counters + 1;
        if (cudaLaunchKernelEx(&cfg, fused_heads_kernel, d_obs, B, actor, actor_head, hh_actor, critic, critic_head, hh_critic, ctr,
                               d_scratch) != cudaSuccess) return -2;
    }
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}
}  // namespace uavp

extern "C" int uavpolicy_selftest_gemm_tile(const void *d_A, const void *d_W, float *d_D, int32_t N, int32_t K, void *stream) {
    if (!d_A || !d_W || !d_D || N <= 0 || N > 384 || N % 16 || (K != 128 && K != 256)) return -1;
    const size_t smem = (size_t)(128 + N) * K * 2;
    if (cudaFuncSetAttribute(gemm_tile_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -2;
    gemm_tile_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>((const __nv_bfloat16 *)d_A, (const __nv_bfloat16 *)d_W, d_D, N, K);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}
