// policy_weights.cuh - dimensions, parameter map and parameter views of TransformerActorCritic shared by the policy kernels
// and the two handles (policy_forward.cu, policy_train.cu).
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "uavpolicy_b200.h"

namespace uavp {

constexpr int S = 5, F = 14, D = 128, H = 8, DH = 16, FF = 256, HID = 64, NACT = 2;
constexpr int kBiasK = 16;                                    // K of a bias operand (one tcgen05.mma k-step)
constexpr int kLayerBiasElems = (3 * D + D + FF + D) * kBiasK;  // bias operands of one encoder layer

// The parameter map: element offset of every tensor of one network (trunk + head) in the flat parameter vector, in the
// order of uavpolicy_set_weights (uavpolicy_b200.h).
struct LayerOff { size_t in_w, in_b, out_w, out_b, l1_w, l1_b, l2_w, l2_b, n1_w, n1_b, n2_w, n2_b; };
struct HeadOff { size_t w1, b1, w2, b2; };
struct NetOff {
    int layers;
    size_t pos, emb_w, emb_b;
    LayerOff layer[2];
    HeadOff head;
    size_t end;                                               // one past the network's last parameter
};
constexpr NetOff net_offsets(size_t off, int layers, int outs) {
    NetOff n{};
    n.layers = layers;
    n.pos = off; off += S * D;
    n.emb_w = off; off += D * F;
    n.emb_b = off; off += D;
    for (int l = 0; l < layers; ++l) {
        LayerOff &L = n.layer[l];
        L.in_w = off; off += 3 * D * D;
        L.in_b = off; off += 3 * D;
        L.out_w = off; off += D * D;
        L.out_b = off; off += D;
        L.l1_w = off; off += FF * D;
        L.l1_b = off; off += FF;
        L.l2_w = off; off += D * FF;
        L.l2_b = off; off += D;
        L.n1_w = off; off += D;
        L.n1_b = off; off += D;
        L.n2_w = off; off += D;
        L.n2_b = off; off += D;
    }
    n.head.w1 = off; off += HID * D;
    n.head.b1 = off; off += HID;
    n.head.w2 = off; off += (size_t)outs * HID;
    n.head.b2 = off; off += outs;
    n.end = off;
    return n;
}
constexpr NetOff kActorOff = net_offsets(0, 1, NACT);
constexpr NetOff kCriticOff = net_offsets(kActorOff.end, 2, 1);
static_assert(kCriticOff.end == UAVPOLICY_NUM_PARAMS, "parameter layout");

// the GEMM weights, [N,K] row-major fp32 in the flat vector: four per encoder layer and each head's W1, network by network
struct GemmW { size_t off; int N, K; };
constexpr int kNumGemmW = 4 * (1 + 2) + 2;
struct GemmList { GemmW w[kNumGemmW]; };
constexpr GemmList gemm_weights() {
    GemmList g{};
    int i = 0;
    const NetOff nets[2] = {kActorOff, kCriticOff};
    for (const NetOff &n : nets) {
        for (int l = 0; l < n.layers; ++l) {
            g.w[i++] = {n.layer[l].in_w, 3 * D, D};
            g.w[i++] = {n.layer[l].out_w, D, D};
            g.w[i++] = {n.layer[l].l1_w, FF, D};
            g.w[i++] = {n.layer[l].l2_w, D, FF};
        }
        g.w[i++] = {n.head.w1, HID, D};
    }
    return g;
}
constexpr GemmList kGemmW = gemm_weights();

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

// points the fp32 members of a network's views at the flat parameter vector w (the bf16 members are left alone)
inline void bind_fp32(BlockW &b, HeadW &h, const NetOff &o, const float *w) {
    b.layers = o.layers;
    b.pos = w + o.pos; b.emb_w = w + o.emb_w; b.emb_b = w + o.emb_b;
    for (int l = 0; l < o.layers; ++l) {
        LayerW &L = b.layer[l];
        const LayerOff &lo = o.layer[l];
        L.in_b = w + lo.in_b; L.out_b = w + lo.out_b; L.l1_b = w + lo.l1_b; L.l2_b = w + lo.l2_b;
        L.n1_w = w + lo.n1_w; L.n1_b = w + lo.n1_b; L.n2_w = w + lo.n2_w; L.n2_b = w + lo.n2_b;
    }
    h.b1 = w + o.head.b1; h.w2 = w + o.head.w2; h.b2 = w + o.head.b2;
}

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
