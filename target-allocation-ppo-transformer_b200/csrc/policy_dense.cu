// policy_dense.cu - the dense layers of the policy / value network on tcgen05, hand-written for sm_100a:
//     D[M,N] (bf16) = act(A[M,K] W[N,K]^T + bias[N])          act = identity | ReLU | ReLU backward by an aux tensor
// (networks/transformer_net.py:24-91: embedding-sized projections, in_proj / out_proj / FFN / head layers and, in the
// PPO update, the activation-gradient products dX = dY W on pre-transposed weights).  M is the batch (up to ~1e6 token
// rows), N, K <= 384: every product is a tall-skinny GEMM that is HBM-bound by construction, so the kernel is built
// around keeping the weight resident and the activations streaming:
//   * persistent CTAs (one per SM), static round-robin over 128-row tiles; a CTA covers the FULL width N of its tile, so
//     every A row is read exactly once and W (<= 96 KB) is loaded once per CTA and stays in shared memory;
//   * warp-specialised: one thread streams [128 x 64] bf16 boxes of A into a 6-box ring with TMA tensor loads
//     (128-byte swizzle; rows past M arrive as zeros), one thread issues tcgen05.mma.kind::f16 (M = 128, N <= 256 per
//     instruction, K = 16; both operands K-major, 128B-swizzled shared-memory descriptors) into TMEM, eight warps run the
//     epilogue - two per TMEM lane quadrant, each taking half of the columns (tcgen05.ld -> bias / ReLU / mask / residual +
//     LayerNorm -> bf16 -> swizzled staging tile -> TMA tensor store, which also clips the ragged last tile);
//   * the TMEM accumulator is double-buffered whenever 2 N <= 512 columns, so the MMAs of tile i+1 run under the
//     epilogue of tile i (N = 384: two single-buffered units of 256 + 128 columns, so that the next tile's first unit is
//     computed while the second one is still being drained); the staging tile is double-buffered against the TMA store.
#include <cstdlib>

#include <cuda.h>

#include "policy_gemm.cuh"
#include "tcgen05_util.cuh"

namespace uavp {
namespace {

constexpr int kThreads = 320;          // warp 0: TMA producer, warp 1: MMA issuer (+ TMEM owner), warps 2-9: epilogue
constexpr int kEpi = 256;              // epilogue threads: two warps per TMEM lane quadrant, each taking half of the columns
constexpr int kBoxBytes = 128 * 128;   // one [128 rows x 64 columns] bf16 box
constexpr int kRing = 6;               // A boxes in flight
constexpr int kMaxN = 384, kMaxK = 384;

enum Act { kIdentity = 0, kRelu = 1, kDRelu = 2, kAddLN = 3 };

struct DenseArgs {
    int M, N, K, act, ring;            // ring: A boxes in flight (<= kRing)
    const float *bias;                 // [N] or nullptr
    const float *gamma, *beta;         // kAddLN: LayerNorm weight / bias [128]
    float *rstd;                       // kAddLN: 1/sigma of every row [M]
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void *tensor_map, const void *smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(tensor_map),
                 "r"(tc::smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *mbar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(tc::smem_u32(mbar)) : "memory");
}

// shared memory: [W: K/64 boxes of N rows x 128 B][ring: g.ring boxes][staging: 2 boxes][aux: 2 boxes (kDRelu)][bias][barriers]
// tm_aux: kDRelu - the [M, N] bf16 tensor whose sign pattern masks the output (the forward's post-ReLU activations);
// kAddLN (N = 128) - the residual x [M, 128]: the epilogue owns whole rows, so out = LayerNorm(x + A W^T + bias) * gamma + beta
// (post-LN encoder layer, networks/transformer_net.py:34-43) is computed from the fp32 accumulator held in registers (a
// thread owns 64 columns of its row; the two halves exchange their partial sums through shared memory) and leaves through
// tm_d (out) and tm_d2 (the normalised row x^ the backward needs) + rstd.
// The aux [128 x 64] boxes are prefetched two slabs ahead by the epilogue's elected thread.
__global__ void __launch_bounds__(kThreads, 1) dense_kernel(const __grid_constant__ CUtensorMap tm_a,
                                                            const __grid_constant__ CUtensorMap tm_w,
                                                            const __grid_constant__ CUtensorMap tm_d,
                                                            const __grid_constant__ CUtensorMap tm_aux,
                                                            const __grid_constant__ CUtensorMap tm_d2, const DenseArgs g) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms are 1024 B aligned
    const int N = g.N, K = g.K, kboxes = K / 64;
    const int w_box = N * 128;                                   // bytes of one 64-column slab of W
    unsigned char *s_w = smem;
    unsigned char *s_ring = s_w + kboxes * w_box;
    const int ring = g.ring;
    unsigned char *s_stage = s_ring + ring * kBoxBytes;
    unsigned char *s_aux = s_stage + (g.act == kAddLN ? 4 : 2) * kBoxBytes;
    float *s_bias = reinterpret_cast<float *>(s_aux + (g.act >= kDRelu ? 2 * kBoxBytes : 0));
    float *s_part = s_bias + kMaxN;                              // kAddLN: [2 halves][128 rows] partial sums
    uint64_t *full = reinterpret_cast<uint64_t *>(s_part + (g.act == kAddLN ? 256 : 0)), *empty = full + kRing, *w_ready = empty + kRing;
    uint64_t *acc_full = w_ready + 1, *acc_empty = acc_full + 2, *aux_full = acc_empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(aux_full + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles = (g.M + 127) / 128;
    const int my_tiles = (int)blockIdx.x < tiles ? (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int acc_stages = 2 * N <= 512 ? 2 : 1;
    const uint32_t tmem_cols = N <= 64 ? 128u : (N <= 128 ? 256u : 512u);    // power of two >= acc_stages * N

    if (warp == 1) tc::tmem_alloc(tmem_slot, tmem_cols);
    for (int i = tid; i < N; i += kThreads) s_bias[i] = g.bias ? g.bias[i] : 0.0f;
    if (g.act == kAddLN)
        for (int i = tid; i < 128; i += kThreads) { s_bias[128 + i] = g.gamma[i]; s_bias[256 + i] = g.beta[i]; }
    if (tid == 0) {
        for (int s = 0; s < kRing; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
        tc::mbar_init(w_ready, 1);
        for (int a = 0; a < 2; ++a) { tc::mbar_init(&acc_full[a], 1); tc::mbar_init(&acc_empty[a], 1); tc::mbar_init(&aux_full[a], 1); }
        tc::fence_mbar_init();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0 && my_tiles > 0) {                         // ---- producer: W once, then the A boxes of every tile
            tc::mbar_expect_tx(w_ready, (uint32_t)(kboxes * w_box));
            const int wrows = N > 256 ? 128 : N;                 // rows per box of the W tensor map (a box has <= 256 rows)
            for (int kb = 0; kb < kboxes; ++kb)
                for (int n0 = 0; n0 < N; n0 += wrows)
                    tc::tma_load_2d(s_w + kb * w_box + n0 * 128, &tm_w, kb * 64, n0, w_ready);
            int it = 0;
            for (int t = 0; t < my_tiles; ++t) {
                const int r0 = ((int)blockIdx.x + t * (int)gridDim.x) * 128;
                for (int kb = 0; kb < kboxes; ++kb, ++it) {
                    const int s = it % ring;
                    if (it >= ring) tc::mbar_wait(&empty[s], (uint32_t)(((it / ring) - 1) & 1));
                    tc::mbar_expect_tx(&full[s], kBoxBytes);
                    tc::tma_load_2d(s_ring + s * kBoxBytes, &tm_a, kb * 64, r0, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && my_tiles > 0) {                         // ---- MMA issuer
            const int n_lo = N > 256 ? 256 : N, n_hi = N - n_lo; // N = 384: a 256-wide and a 128-wide instruction
            const uint32_t idesc_lo = tc::instr_desc_bf16(128, n_lo), idesc_hi = n_hi ? tc::instr_desc_bf16(128, n_hi) : 0u;
            tc::mbar_wait(w_ready, 0);
            int it = 0;
            for (int t = 0; t < my_tiles; ++t) {
                if (N > 256) {
                    // N = 384 does not fit twice into the 512 TMEM columns: two single-buffered units instead, A = columns
                    // 0..255 (one 256-wide instruction per k-step) and B = 256..383 (128-wide), each with its own full / empty
                    // barrier pair - unit A of tile t+1 is computed while the epilogue still drains unit B of tile t
                    const int it0 = it;
                    if (t > 0) tc::mbar_wait(&acc_empty[0], (uint32_t)((t - 1) & 1));
                    tc::tc_fence_after();
                    for (int kb = 0; kb < kboxes; ++kb, ++it) {
                        const int s = it % ring;
                        tc::mbar_wait(&full[s], (uint32_t)((it / ring) & 1));
                        tc::tc_fence_after();
                        const uint32_t sa = tc::smem_u32(s_ring + s * kBoxBytes), sw = tc::smem_u32(s_w + kb * w_box);
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            tc::mma_bf16(tmem, tc::smem_desc_sw128(sa + j * 32, 16, 1024), tc::smem_desc_sw128(sw + j * 32, 16, 1024),
                                         idesc_lo, (kb > 0 || j > 0) ? 1u : 0u);
                    }
                    tc::mma_commit(&acc_full[0]);
                    if (t > 0) tc::mbar_wait(&acc_empty[1], (uint32_t)((t - 1) & 1));
                    tc::tc_fence_after();
                    for (int kb = 0; kb < kboxes; ++kb) {
                        const int s = (it0 + kb) % ring;
                        const uint32_t sa = tc::smem_u32(s_ring + s * kBoxBytes), sw = tc::smem_u32(s_w + kb * w_box + 256 * 128);
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            tc::mma_bf16(tmem + 256, tc::smem_desc_sw128(sa + j * 32, 16, 1024), tc::smem_desc_sw128(sw + j * 32, 16, 1024),
                                         idesc_hi, (kb > 0 || j > 0) ? 1u : 0u);
                        tc::mma_commit(&empty[s]);               // both passes have read the box
                    }
                    tc::mma_commit(&acc_full[1]);
                    continue;
                }
                const int a = t % acc_stages;
                const int use = t / acc_stages;                  // how often this accumulator has been used before
                if (use > 0) tc::mbar_wait(&acc_empty[a], (uint32_t)((use - 1) & 1));
                tc::tc_fence_after();
                const uint32_t d = tmem + (uint32_t)(a * N);
                for (int kb = 0; kb < kboxes; ++kb, ++it) {
                    const int s = it % ring;
                    tc::mbar_wait(&full[s], (uint32_t)((it / ring) & 1));
                    tc::tc_fence_after();
                    const uint32_t sa = tc::smem_u32(s_ring + s * kBoxBytes), sw = tc::smem_u32(s_w + kb * w_box);
#pragma unroll
                    for (int j = 0; j < 4; ++j)                  // K = 16 per instruction: 32 B further into the 128 B rows
                        tc::mma_bf16(d, tc::smem_desc_sw128(sa + j * 32, 16, 1024), tc::smem_desc_sw128(sw + j * 32, 16, 1024), idesc_lo,
                                     (kb > 0 || j > 0) ? 1u : 0u);
                    tc::mma_commit(&empty[s]);                   // frees the ring slot when these MMAs have read it
                }
                tc::mma_commit(&acc_full[a]);
            }
        }
    } else {                                                     // ---- epilogue: warp w owns TMEM lanes 32 * (w % 4) ..
        const int q = warp & 3, et = tid - 64;                   // et: 0..255 among the epilogue threads
        const int half = (warp - 2) >> 2;                        // which 32 of a slab's 64 columns (kAddLN: which slab) it takes
        const int row = q * 32 + lane;                           // row of the tile = TMEM lane
        int stores = 0;
        const int spt = N / 64, total_slabs = my_tiles * spt;    // output slabs per tile / of this CTA
        auto prefetch_aux = [&](int seq) {                       // aux box of output slab `seq` of this CTA -> buffer seq & 1
            if (seq >= total_slabs) return;
            const int tt = seq / spt, cc = (seq % spt) * 64;
            tc::mbar_expect_tx(&aux_full[seq & 1], kBoxBytes);
            tc::tma_load_2d(s_aux + (seq & 1) * kBoxBytes, &tm_aux, cc, ((int)blockIdx.x + tt * (int)gridDim.x) * 128, &aux_full[seq & 1]);
        };
        if (g.act >= kDRelu && et == 0) { prefetch_aux(0); prefetch_aux(1); }
        for (int t = 0; t < my_tiles; ++t) {
            const bool split = N > 256;                          // N = 384: units A (columns 0..255) and B (256..383), see the MMA issuer
            const int a = split ? 0 : t % acc_stages, use = split ? t : t / acc_stages;
            const int r0 = ((int)blockIdx.x + t * (int)gridDim.x) * 128;
            if (!split) {
                tc::mbar_wait(&acc_full[a], (uint32_t)(use & 1));
                tc::tc_fence_after();
            }
            const uint32_t src = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * N);
            if (g.act == kAddLN) {
                // this thread's half of the row (= residual slab `half`, aux buffer `half` holds slab 2 t + half) in registers:
                // v = accumulator + bias + residual
                tc::mbar_wait(&aux_full[half], (uint32_t)(t & 1));
                float v[64];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    tc::tmem_ld32(src + (uint32_t)(half * 64 + h * 32), v + h * 32);
                    const unsigned char *ab = s_aux + half * kBoxBytes + row * 128;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint4 rw = *reinterpret_cast<const uint4 *>(ab + (((h * 4 + c) ^ (row & 7)) << 4));
                        const uint32_t w4[4] = {rw.x, rw.y, rw.z, rw.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const __nv_bfloat162 r2 = *reinterpret_cast<const __nv_bfloat162 *>(&w4[e]);
                            const int i = h * 32 + c * 8 + 2 * e;
                            v[i] += s_bias[half * 64 + i] + __low2float(r2);
                            v[i + 1] += s_bias[half * 64 + i + 1] + __high2float(r2);
                        }
                    }
                }
                float sum = 0.0f, sq = 0.0f;
#pragma unroll
                for (int i = 0; i < 64; ++i) sum += v[i];
                s_part[half * 128 + row] = sum;
                tc::tc_fence_before();
                named_bar_sync(1, kEpi);                         // partial sums visible; every thread has read the accumulator
                if (et == 0) mbar_arrive(&acc_empty[a]);
                const float mean = (s_part[row] + s_part[128 + row]) * (1.0f / 128.0f);
#pragma unroll
                for (int i = 0; i < 64; ++i) { v[i] -= mean; sq = fmaf(v[i], v[i], sq); }
                named_bar_sync(1, kEpi);                         // (the sums were read before they are overwritten)
                s_part[half * 128 + row] = sq;
                if (t > 0 && et == 0) bulk_wait_read<0>();       // the previous tile's stores have read the staging boxes
                named_bar_sync(1, kEpi);
                const float rstd = rsqrtf((s_part[row] + s_part[128 + row]) * (1.0f / 128.0f) + 1e-5f);
                if (half == 0 && r0 + row < g.M) g.rstd[r0 + row] = rstd;
                unsigned char *sy = s_stage + (2 * half) * kBoxBytes, *sx = sy + kBoxBytes;   // out / x^ boxes of this slab
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    uint32_t py[4], px[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int i = c * 8 + 2 * e, col = half * 64 + i;
                        const float x0 = v[i] * rstd, x1 = v[i + 1] * rstd;
                        const __nv_bfloat162 hx = __floats2bfloat162_rn(x0, x1);
                        const __nv_bfloat162 hy = __floats2bfloat162_rn(fmaf(x0, s_bias[128 + col], s_bias[256 + col]),
                                                                        fmaf(x1, s_bias[128 + col + 1], s_bias[256 + col + 1]));
                        px[e] = *reinterpret_cast<const uint32_t *>(&hx);
                        py[e] = *reinterpret_cast<const uint32_t *>(&hy);
                    }
                    const int off = row * 128 + ((c ^ (row & 7)) << 4);
                    *reinterpret_cast<uint4 *>(sy + off) = make_uint4(py[0], py[1], py[2], py[3]);
                    *reinterpret_cast<uint4 *>(sx + off) = make_uint4(px[0], px[1], px[2], px[3]);
                }
                tc::fence_async_smem();
                named_bar_sync(1, kEpi);                         // staging boxes complete; both residual boxes have been read
                if (et == 0) {
                    tma_store_2d(&tm_d, s_stage, 0, r0);
                    tma_store_2d(&tm_d2, s_stage + kBoxBytes, 0, r0);
                    tma_store_2d(&tm_d, s_stage + 2 * kBoxBytes, 64, r0);
                    tma_store_2d(&tm_d2, s_stage + 3 * kBoxBytes, 64, r0);
                    prefetch_aux(2 * (t + 1)); prefetch_aux(2 * (t + 1) + 1);
                }
                continue;
            }
            for (int c0 = 0; c0 < N; c0 += 64, ++stores) {
                if (split && (c0 == 0 || c0 == 256)) {
                    tc::mbar_wait(&acc_full[c0 >> 8], (uint32_t)(t & 1));
                    tc::tc_fence_after();
                }
                unsigned char *stage = s_stage + (stores & 1) * kBoxBytes;
                if (stores >= 2) {                               // the TMA store that last read this staging box is done with it
                    if (et == 0) bulk_wait_read<1>();
                    named_bar_sync(1, kEpi);
                }
                uint4 mask[4];
                if (g.act == kDRelu) {                           // this slab's aux box (rows past M arrive as zeros: masked)
                    tc::mbar_wait(&aux_full[stores & 1], (uint32_t)((stores >> 1) & 1));
                    const unsigned char *ab = s_aux + (stores & 1) * kBoxBytes + row * 128;
#pragma unroll
                    for (int c = 0; c < 4; ++c) mask[c] = *reinterpret_cast<const uint4 *>(ab + (((half * 4 + c) ^ (row & 7)) << 4));
                }
                float v[32];
                tc::tmem_ld32(src + (uint32_t)(c0 + half * 32), v);
#pragma unroll
                for (int c = 0; c < 4; ++c) {                    // 8 columns = one 16-byte chunk of the output row
                    uint32_t pk[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float x0 = v[c * 8 + 2 * e] + s_bias[c0 + half * 32 + c * 8 + 2 * e];
                        float x1 = v[c * 8 + 2 * e + 1] + s_bias[c0 + half * 32 + c * 8 + 2 * e + 1];
                        if (g.act == kRelu) { x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f); }
                        __nv_bfloat162 p2 = __floats2bfloat162_rn(x0, x1);
                        pk[e] = *reinterpret_cast<uint32_t *>(&p2);
                    }
                    if (g.act == kDRelu) {
                        const uint32_t *mw = reinterpret_cast<const uint32_t *>(&mask[c]);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {            // bf16 > 0  <=>  sign bit clear and magnitude non-zero
                            const uint32_t z = mw[e];
                            const uint32_t lo_ok = ((z & 0x8000u) == 0u && (z & 0x7fffu) != 0u) ? 0xffffu : 0u;
                            const uint32_t hi_ok = ((z & 0x80000000u) == 0u && (z & 0x7fff0000u) != 0u) ? 0xffff0000u : 0u;
                            pk[e] &= (lo_ok | hi_ok);
                        }
                    }
                    const int chunk = half * 4 + c;              // 128-byte swizzle: chunk index XOR (row mod 8)
                    *reinterpret_cast<uint4 *>(stage + row * 128 + ((chunk ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
                tc::fence_async_smem();
                tc::tc_fence_before();
                named_bar_sync(1, kEpi);                         // staging box complete; everyone has read this slab's aux box
                if (et == 0) {
                    tma_store_2d(&tm_d, stage, c0, r0);
                    if (g.act == kDRelu) prefetch_aux(stores + 2);
                    if (split && (c0 == 192 || c0 == 320)) mbar_arrive(&acc_empty[c0 == 192 ? 0 : 1]);   // the unit is drained
                }
            }
            if (split) continue;
            tc::tc_fence_before();
            named_bar_sync(1, kEpi);                             // every epilogue thread has read this accumulator
            if (et == 0) mbar_arrive(&acc_empty[a]);
        }
        if (et == 0) bulk_wait_all();
    }
    __syncthreads();
    if (warp == 1) { tc::tc_fence_after(); tc::tmem_free(tmem, tmem_cols); }
}

int g_sms = 0;
bool g_ready = false;

int ring_depth(int act, int K) { return act == kAddLN ? (K > 128 ? 3 : 4) : (act == kDRelu ? 4 : kRing); }

size_t smem_bytes(int N, int K, int act) {
    return (size_t)(K / 64) * N * 128 + (size_t)(ring_depth(act, K) + (act == kAddLN ? 4 : 2) + (act >= kDRelu ? 2 : 0)) * kBoxBytes +
           (kMaxN + (act == kAddLN ? 256 : 0)) * sizeof(float) + 256 + 1024;
}

int prepare() {
    if (g_ready) return 0;
    if (!tensor_maps_available()) return -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(kMaxN, 128, kIdentity)) != cudaSuccess)
        return -1;
    g_ready = true;
    return 0;
}

int launch(const void *A, int64_t lda, const void *W, const float *bias, const void *aux, int64_t ld_aux, void *D, int M, int N, int K,
           int act, cudaStream_t stream, const float *gamma = nullptr, const float *beta = nullptr, void *xhat = nullptr,
           float *rstd = nullptr) {
    if (M <= 0) return 0;
    // shapes of this network: N in {64, 128, 256, 384}, K a multiple of 64 up to 384, W <= 96 KB
    if (N % 64 || N > kMaxN || (N > 256 && N != 384) || K % 64 || K > kMaxK || (size_t)N * K * 2 > 96 * 1024 || lda % 8 || (aux && ld_aux % 8))
        return -1;
    if (prepare()) return -2;
    if (act >= kDRelu && (!aux || smem_bytes(N, K, act) > smem_bytes(kMaxN, 128, kIdentity))) return -1;
    if (act == kAddLN && (N != 128 || !gamma || !beta || !xhat || !rstd)) return -1;
    CUtensorMap tm_a, tm_w, tm_d, tm_aux, tm_d2;
    if (!make_tensor_map(&tm_a, A, lda, M, K, 128) || !make_tensor_map(&tm_w, W, K, N, K, N > 256 ? 128 : N) ||
        !make_tensor_map(&tm_d, D, N, M, N, 128))
        return -3;
    if (act >= kDRelu) { if (!make_tensor_map(&tm_aux, aux, ld_aux, M, N, 128)) return -3; }
    else tm_aux = tm_d;
    if (act == kAddLN) { if (!make_tensor_map(&tm_d2, xhat, N, M, N, 128)) return -3; }
    else tm_d2 = tm_d;
    DenseArgs g;
    g.M = M; g.N = N; g.K = K; g.act = act; g.ring = ring_depth(act, K); g.bias = bias;
    g.gamma = gamma; g.beta = beta; g.rstd = rstd;
    const int tiles = (M + 127) / 128;
    dense_kernel<<<tiles < g_sms ? tiles : g_sms, kThreads, smem_bytes(N, K, act), stream>>>(tm_a, tm_w, tm_d, tm_aux, tm_d2, g);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

}  // namespace

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encoder() {   // looked up on the first call
    static const EncodeTiledFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
                        q == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<EncodeTiledFn>(f) : nullptr;
    }();
    return fn;
}
}  // namespace

bool tensor_maps_available() { return encoder() != nullptr; }

bool make_tensor_map(CUtensorMap *m, const void *base, int64_t ld, int64_t rows, int cols, int box_rows) {
    const EncodeTiledFn encode = encoder();
    if (!encode) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows}, estr[2] = {1, 1};
    return encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int gemm_bias_act(const void *A, int64_t lda, const void *W, const float *bias, void *D, int M, int N, int K, int relu,
                  cudaStream_t stream) {
    return launch(A, lda, W, bias, nullptr, 0, D, M, N, K, relu ? kRelu : kIdentity, stream);
}

int gemm_drelu(const void *A, int64_t lda, const void *W, const void *aux, int64_t ld_aux, void *D, int M, int N, int K,
               cudaStream_t stream) {
    return launch(A, lda, W, nullptr, aux, ld_aux, D, M, N, K, kDRelu, stream);
}


int gemm_add_ln(const void *A, int64_t lda, const void *W, const float *bias, const void *X, int64_t ldx, const float *gamma,
                const float *beta, void *out, void *xhat, float *rstd, int M, int K, cudaStream_t stream) {
    return launch(A, lda, W, bias, X, ldx, out, M, 128, K, kAddLN, stream, gamma, beta, xhat, rstd);
}

}  // namespace uavp

// self-test hook: one dense product on caller-provided device buffers (act: 0 identity, 1 ReLU, 2 ReLU backward by d_aux)
extern "C" int uavpolicy_selftest_dense(const void *d_a, int64_t lda, const void *d_w, const float *d_bias, const void *d_aux,
                                        int64_t ld_aux, void *d_out, int32_t M, int32_t N, int32_t K, int32_t act, void *stream) {
    if (act == 2) return uavp::gemm_drelu(d_a, lda, d_w, d_aux, ld_aux, d_out, M, N, K, (cudaStream_t)stream);
    if (act == 3) return -1;   // residual + LayerNorm: uavpolicy_selftest_dense_ln
    return uavp::gemm_bias_act(d_a, lda, d_w, d_bias, d_out, M, N, K, act, (cudaStream_t)stream);
}

// self-test hook of the fused residual + LayerNorm epilogue: d_out = LayerNorm(d_x + d_a d_w^T + d_bias) * d_gamma + d_beta,
// d_xhat = the normalised rows, d_rstd = 1/sigma (N = 128)
extern "C" int uavpolicy_selftest_dense_ln(const void *d_a, int64_t lda, const void *d_w, const float *d_bias, const void *d_x,
                                           int64_t ldx, const float *d_gamma, const float *d_beta, void *d_out, void *d_xhat,
                                           float *d_rstd, int32_t M, int32_t K, void *stream) {
    return uavp::gemm_add_ln(d_a, lda, d_w, d_bias, d_x, ldx, d_gamma, d_beta, d_out, d_xhat, d_rstd, M, K, (cudaStream_t)stream);
}
