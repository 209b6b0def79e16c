// policy_weights.cuh - parameter views and dimensions of TransformerActorCritic shared by the policy kernels.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "uavpolicy_b200.h"

namespace uavp {

constexpr int S = 5, F = 14, D = 128, H = 8, DH = 16, FF = 256, HID = 64, NACT = 2;
constexpr int kLayerParams = 3 * D * D + 3 * D + D * D + D + FF * D + FF + D * FF + D + 4 * D;  // 132480
constexpr int kBlockBase = S * D + D * F + D;                                                   // pos, emb w, emb b
constexpr int kActorHead = HID * D + HID + NACT * HID + NACT;
constexpr int kCriticHead = HID * D + HID + HID + 1;
constexpr int kBiasK = 16;                                    // K of a bias operand (one tcgen05.mma k-step)
constexpr int kLayerBiasElems = (3 * D + D + FF + D) * kBiasK;  // bias operands of one encoder layer
static_assert(kBlockBase + kLayerParams + kActorHead + kBlockBase + 2 * kLayerParams + kCriticHead == UAVPOLICY_NUM_PARAMS,
              "parameter layout");

struct LayerW {  // views of the parameters of one encoder layer
    const __nv_bfloat16 *in_w, *out_w, *l1_w, *l2_w;  // [384,128] [128,128] [256,128] [128,256] bf16 row-major (PPO update)
    const __nv_bfloat16 *in_wp, *out_wp, *l1_wp, *l2_wp;  // the same matrices pre-packed in UMMA canonical K-major order (fused kernel)
    // the four biases as [N x 16] bf16 B-operands of one more k-step (canonical order): column 0 = bf16(b), column 1 = the
    // rounding remainder, the rest zero - against an A-operand of ones the tensor core adds the bias (fused kernel only)
    const __nv_bfloat16 *in_bp = nullptr, *out_bp = nullptr, *l1_bp = nullptr, *l2_bp = nullptr;
    const float *in_b, *out_b, *l1_b, *l2_b, *n1_w, *n1_b, *n2_w, *n2_b;
};
struct BlockW {
    const float *pos, *emb_w, *emb_b;
    const __nv_bfloat16 *emb_w2p;  // [128 x 32] bf16, UMMA canonical order: columns 0..13 and 16..29 both hold emb_w (the fused kernel feeds the
                                   // embedding to the tensor cores with the observation split into bf16 hi + lo parts);
                                   // columns 14 / 15 hold emb_b as bf16 + remainder (the A operand has ones there)
    LayerW layer[2];
    int layers;
};
struct HeadW { const __nv_bfloat16 *w1p; const float *b1, *w2, *b2; const __nv_bfloat16 *b1p = nullptr; };  // w1p: W1 [64,128] packed bf16; b1p: b1 as a bias operand; rest fp32


// fused encoder blocks (policy_fused.cu): embedding + all post-LN encoder layers + first head layer of BOTH networks for a
// batch of windows in TWO launches (per-tile work, then the newest-token rows of every 128 samples on full tiles), every GEMM
// on tcgen05 with operands resident in shared memory.  Writes relu(W1 z_last + b1) as bf16 [B,64] per network.
// d_work_counters: two ints; d_scratch: fused_scratch_bytes(max_batch) bytes (zero-initialised once).
// actor_only: run the actor's work items alone (hh_critic is neither read nor written).
int launch_fused_blocks(const float *d_obs, int B, const BlockW &actor, const HeadW &actor_head, __nv_bfloat16 *hh_actor,
                        const BlockW &critic, const HeadW &critic_head, __nv_bfloat16 *hh_critic, int *d_work_counters,
                        unsigned char *d_scratch, cudaStream_t stream, bool actor_only = false);
size_t fused_scratch_bytes(int max_batch);
int fused_block_prepare();   // one-time kernel attribute setup; 0 on success

}  // namespace uavp
