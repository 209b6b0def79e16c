// policy_wgrad.cu - weight gradients of the PPO update on tcgen05: dW[Nout, Kin] += dY[rows, Nout]^T X[rows, Kin].
//
// The contraction runs over the batch rows (hundreds of thousands) while the output is a single small matrix, so this
// is a split-K problem: every CTA owns a strided set of 64-row slabs, streams the dY and X tiles of each slab into
// shared memory (TMA tensor loads into a 4-6 stage ring) and accumulates its partial dW in TMEM across ALL its slabs -
// one tcgen05.mma chain, no intermediate traffic - then adds the partial to the fp32 gradient with coalesced RED.ADD.
// Both operands are read MN-major straight from the row-major activations (tcgen05_util.cuh: instr_desc_bf16_mn): no
// transposed copy of dY or X is ever made.  blockIdx.y selects a 128-column block of dY (= 128 rows of dW).  The bias
// gradient (column sums of dY) rides along as dY^T 1: one more N = 16 MMA per k-step against an all-ones operand.
#include <cstdlib>

#include <cuda.h>

#include "policy_gemm.cuh"
#include "policy_weights.cuh"
#include "tcgen05_util.cuh"

namespace uavp {
namespace {

// (A first version staged the tiles with a cp.async / LDGSTS ring: it topped out at ~25 GB/s per SM - the L1 miss
// path - i.e. 3.6 TB/s, whatever the ring depth or thread count; bulk tensor copies do not go through that path.)
// One thread streams [64 rows x 64 columns] boxes (128-byte rows, CU_TENSOR_MAP_SWIZZLE_128B) of dY and X into the
// ring, one thread issues the MMAs and four warps run the epilogue.  A box is exactly one MN-major swizzle-atom column
// of the UMMA operand: 8-row groups 1024 B apart (SBO), 64-column blocks one box apart (LBO); rows beyond the matrix
// arrive as zeros (TMA out-of-bounds fill).
constexpr int kTmaThreads = 192;
template <int KIN>
struct WgTma {
    static constexpr int kSlab = 64;
    static constexpr int kBox = kSlab * 128;                 // bytes of one [64 x 64] bf16 box
    static constexpr int kA = 2 * kBox, kB = (KIN / 64) * kBox, kStage = kA + kB;
    static constexpr int kStages = KIN == 64 ? 8 : KIN == 128 ? 6 : 4;
    static constexpr int kOnes = kSlab * 16 * 2;
    static constexpr int kTotal = kStages * kStage + kOnes + 256 + 1024;    // + barriers + alignment slack
    static_assert(4 * 32 * (KIN + 1) * 4 <= kStages * kStage, "the epilogue transposes through the operand buffers");
};

template <int KIN>
__global__ void __launch_bounds__(kTmaThreads, 1) wgrad_tma_kernel(const __grid_constant__ CUtensorMap tm_dy,
                                                                   const __grid_constant__ CUtensorMap tm_x, int rows,
                                                                   float *__restrict__ dW, int nout_valid, float *__restrict__ dbias,
                                                                   int out_ld, int kin_valid) {
    using SM = WgTma<KIN>;
    constexpr int kSlab = SM::kSlab, kStages = SM::kStages;
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms are 1024 B aligned
    unsigned char *ones = smem + kStages * SM::kStage;
    uint64_t *full = reinterpret_cast<uint64_t *>(ones + SM::kOnes), *empty = full + kStages, *accum = empty + kStages;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accum + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int slabs = (rows + kSlab - 1) / kSlab;
    if ((int)blockIdx.x >= slabs) return;
    const int cnt = (slabs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int nb = blockIdx.y;
    constexpr int kCols = KIN <= 128 ? 2 * KIN : KIN;        // accumulators (+ 16 columns for the bias block when KIN <= 128)

    if (warp == 1) tc::tmem_alloc(tmem_slot, kCols);
    if (dbias) {
        for (int i = tid; i < SM::kOnes / 4; i += kTmaThreads) reinterpret_cast<uint32_t *>(ones)[i] = 0x3F803F80u;
        tc::fence_async_smem();
    }
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
        tc::mbar_init(accum, 1);
        tc::fence_mbar_init();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                     // ---- producer
            for (int it = 0; it < cnt; ++it) {
                const int s = it % kStages;
                if (it >= kStages) tc::mbar_wait(&empty[s], (uint32_t)(((it / kStages) - 1) & 1));
                unsigned char *a = smem + s * SM::kStage, *b = a + SM::kA;
                const int r0 = ((int)blockIdx.x + it * (int)gridDim.x) * kSlab;
                tc::mbar_expect_tx(&full[s], SM::kStage);
#pragma unroll
                for (int cb = 0; cb < 2; ++cb) tc::tma_load_2d(a + cb * SM::kBox, &tm_dy, nb * 128 + cb * 64, r0, &full[s]);
#pragma unroll
                for (int cb = 0; cb < KIN / 64; ++cb) tc::tma_load_2d(b + cb * SM::kBox, &tm_x, cb * 64, r0, &full[s]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                     // ---- MMA issuer
            constexpr uint32_t idesc = tc::instr_desc_bf16_mn(128, KIN);
            for (int it = 0; it < cnt; ++it) {
                const int s = it % kStages;
                tc::mbar_wait(&full[s], (uint32_t)((it / kStages) & 1));
                tc::tc_fence_after();
                const uint32_t a = tc::smem_u32(smem + s * SM::kStage), b = a + SM::kA;
#pragma unroll
                for (int j = 0; j < kSlab / 16; ++j) {       // 16 rows = two 8-row groups = 2048 B further into every box
                    const uint64_t ad = tc::smem_desc_sw128(a + j * 2048, SM::kBox, 1024);
                    const uint64_t bd = tc::smem_desc_sw128(b + j * 2048, SM::kBox, 1024);
                    tc::mma_bf16(tmem, ad, bd, idesc, (it > 0 || j > 0) ? 1u : 0u);
                    if (KIN <= 128 && dbias)
                        tc::mma_bf16(tmem + KIN, ad, tc::smem_desc(tc::smem_u32(ones), 16 * 16, 128), tc::instr_desc_bf16_mn(128, 16),
                                     (it > 0 || j > 0) ? 1u : 0u);
                }
                tc::mma_commit(&empty[s]);                   // frees the stage when these MMAs have read it
            }
            tc::mma_commit(accum);
        }
    } else {                                                 // ---- epilogue: warp w owns TMEM lanes 32 * (w % 4) ..
        tc::mbar_wait(accum, 0);
        tc::tc_fence_after();
        const int q = warp & 3;
        float *stage_f = reinterpret_cast<float *>(smem) + (size_t)q * 32 * (KIN + 1);
        const int rows_out = min(128, nout_valid - nb * 128) - q * 32;       // rows of this warp's block that exist
#pragma unroll 1
        for (int c = 0; c < KIN; c += 32) {
            float v[32];
            tc::tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + c, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) stage_f[lane * (KIN + 1) + c + i] = v[i];
        }
        __syncwarp();
        float *out = dW + ((size_t)nb * 128 + q * 32) * out_ld;
        for (int r = 0; r < min(32, rows_out); ++r)
            for (int c = lane; c < kin_valid; c += 32) atomicAdd(out + r * out_ld + c, stage_f[r * (KIN + 1) + c]);
        if (KIN <= 128 && dbias) {
            float v[32];
            tc::tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + KIN, v);
            if (lane < rows_out) atomicAdd(dbias + nb * 128 + q * 32 + lane, v[0]);
        }
        tc::tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) { tc::tc_fence_after(); tc::tmem_free(tmem, kCols); }
}

}  // namespace

int wgrad_prepare() {
    if (!tensor_maps_available()) return -1;
    if (cudaFuncSetAttribute(wgrad_tma_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, WgTma<128>::kTotal) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(wgrad_tma_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, WgTma<256>::kTotal) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(wgrad_tma_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, WgTma<64>::kTotal) != cudaSuccess) return -1;
    return 0;
}

// dW[Nout, Kin] (fp32, dense) += dY[rows, Nout]^T X[rows, Kin];  Nout % 128 == 0, Kin in {128, 256}, ld % 8 == 0.
// Only the first nout_valid rows of dW are written (dY columns beyond that are padding).  dbias (optional, Kin <= 128):
// dbias[Nout] += column sums of dY, computed by the tensor cores as dY^T 1 alongside the main product.
// Kin = 64: X is padded to 64 columns; the first kin_valid columns go out with row stride out_ld (the embedding's [128,14]).
int wgrad(const __nv_bfloat16 *dY, int64_t ld_dy, const __nv_bfloat16 *X, int64_t ld_x, int rows, int Nout, int Kin, float *dW,
          int nout_valid, float *dbias, int num_sms, cudaStream_t stream, int out_ld, int kin_valid) {
    if (rows <= 0 || Nout % 128 || (Kin != 64 && Kin != 128 && Kin != 256) || ld_dy % 8 || ld_x % 8 || (dbias && Kin > 128)) return -1;
    if (out_ld <= 0) out_ld = Kin;
    if (kin_valid <= 0) kin_valid = Kin;
    const int slab = WgTma<128>::kSlab;
    const int gy = Nout / 128, slabs = (rows + slab - 1) / slab;
    const int gx = max(1, min(slabs, num_sms / gy));
    CUtensorMap tm_dy, tm_x;
    if (!make_tensor_map(&tm_dy, dY, ld_dy, rows, Nout, 64) || !make_tensor_map(&tm_x, X, ld_x, rows, Kin, 64)) return -3;
    if (Kin == 64) wgrad_tma_kernel<64><<<dim3(gx, gy), kTmaThreads, WgTma<64>::kTotal, stream>>>(tm_dy, tm_x, rows, dW, nout_valid, dbias, out_ld, kin_valid);
    else if (Kin == 128) wgrad_tma_kernel<128><<<dim3(gx, gy), kTmaThreads, WgTma<128>::kTotal, stream>>>(tm_dy, tm_x, rows, dW, nout_valid, dbias, out_ld, kin_valid);
    else wgrad_tma_kernel<256><<<dim3(gx, gy), kTmaThreads, WgTma<256>::kTotal, stream>>>(tm_dy, tm_x, rows, dW, nout_valid, dbias, out_ld, kin_valid);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

}  // namespace uavp

// self-test hook: one weight-gradient product on caller-provided device buffers
extern "C" int uavpolicy_selftest_wgrad(const void *d_dy, int64_t ld_dy, const void *d_x, int64_t ld_x, int32_t rows, int32_t n_out,
                                        int32_t k_in, float *d_dw, float *d_dbias, void *stream) {
    if (uavp::wgrad_prepare()) return -2;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -2;
    return uavp::wgrad(static_cast<const __nv_bfloat16 *>(d_dy), ld_dy, static_cast<const __nv_bfloat16 *>(d_x), ld_x, rows, n_out,
                       k_in, d_dw, n_out, d_dbias, sms, (cudaStream_t)stream, 0, 0);
}
