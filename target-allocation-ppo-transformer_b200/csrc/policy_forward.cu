// policy_forward.cu - rollout forward of TransformerActorCritic (networks/transformer_net.py:47-122) on sm_100a.
//
// Two fused launches (policy_fused.cu) run the embedding, every encoder layer and the first head layer of both networks
// with all dense contractions on tcgen05, and write the two [B,64] head-hidden rows in bf16.  heads_out_kernel below then
// forms the second head layers in fp32 with softmax, the Categorical sample, log-prob and entropy.  The host side owns
// the handle: a private fp32 copy of the parameters, the GEMM weights and biases pre-packed in the operand layouts the
// fused kernels stage with bulk TMA, and the buffers passed between the launches.  uavpolicy_act (uavpolicy_eval_b200.h)
// runs the same launches on the actor's work items alone and actor_out_kernel in place of heads_out_kernel.
#include "uavpolicy_b200.h"
#include "uavpolicy_eval_b200.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "philox.cuh"
#include "handle.cuh"
#include "policy_kernels.cuh"
#include "policy_weights.cuh"
#include "tcgen05_util.cuh"

namespace {
using namespace uavp;

// ------------------------------------------------------------------------------------------------ kernels

// Weight packing (uavpolicy_set_weights): bf16 operands in the UMMA canonical K-major order the fused kernels stage
// with one bulk TMA copy each (tc::canon_off is in bytes, hence / 2 for an element offset).

// [128 x 14] fp32 embedding weight -> [128 x 32] bf16, canonical order, the 14 columns duplicated at 0.. and 16..
// columns 14 / 15: the embedding bias as bf16 + rounding remainder (the A operand carries ones in these two columns)
__global__ void emb_w2_kernel(const float *__restrict__ w, const float *__restrict__ b, __nv_bfloat16 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D * 32) return;
    const int d = i / 32, c = i % 32, j = c % 16;
    float v = j < F ? w[d * F + j] : 0.0f;
    if (c == 14) v = b[d];
    if (c == 15) v = b[d] - __bfloat162float(__float2bfloat16(b[d]));
    out[tc::canon_off(d, c, 32) / 2] = __float2bfloat16(v);
}

// bias [N] fp32 -> [N x 16] bf16 B-operand in canonical order: column 0 = bf16(b), column 1 = b - bf16(b), rest zero
__global__ void pack_bias_kernel(const float *__restrict__ b, __nv_bfloat16 *__restrict__ out, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * 16) return;
    const int n = i / 16, c = i % 16;
    const float hi = __bfloat162float(__float2bfloat16(b[n]));
    out[tc::canon_off(n, c, 16) / 2] = __float2bfloat16(c == 0 ? hi : (c == 1 ? b[n] - hi : 0.0f));
}

// row-major fp32 [N x K] -> bf16 in canonical order (one bulk TMA copy then stages a whole B operand)
__global__ void pack_canon_kernel(const float *__restrict__ w, __nv_bfloat16 *__restrict__ out, int N, int K) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * K) return;
    out[tc::canon_off(i / K, i % K, K) / 2] = __float2bfloat16(w[i]);
}

// log-softmax of the two logits and the Categorical sample (transformer_net.py:116-120) of env `env` at `step`: u is the
// top 24 bits of one Philox block keyed by the seed (k0, k1).  heads_out_kernel and actor_out_kernel both draw here, so
// a sample of uavpolicy_act is bit-identical to uavpolicy_get_action's for the same keys.
__device__ __forceinline__ int draw_action(float l0, float l1, uint32_t k0, uint32_t k1, uint64_t step, uint64_t env, float &lp0,
                                           float &lp1) {
    const float m = fmaxf(l0, l1), e0 = expf(l0 - m), e1 = expf(l1 - m), lse = m + logf(e0 + e1);
    lp0 = l0 - lse; lp1 = l1 - lse;
    const uint4 r = philox4x32(k0, k1, (uint32_t)env, (uint32_t)step, (uint32_t)(step >> 32), 0x00B01C70u ^ (uint32_t)(env >> 32));
    const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);   // uniform [0,1)
    return u < expf(lp1) ? 1 : 0;                               // Categorical(probs).sample()
}

// head outputs: logits and value (head_out), then the sample (draw_action), log-prob and entropy
// (transformer_net.py:116-122).  One thread per sample.
__global__ void __launch_bounds__(256) heads_out_kernel(const __nv_bfloat16 *__restrict__ Ha, const __nv_bfloat16 *__restrict__ Hc,
                                                        HeadW ha, HeadW hc, int B, uint32_t k0, uint32_t k1, uint64_t step,
                                                        uint64_t env_base, int64_t *__restrict__ action,
                                                        float *__restrict__ logp, float *__restrict__ value,
                                                        float *__restrict__ entropy, float *__restrict__ logits_out) {
    int b;
    float l0, l1, vv, lp0, lp1;
    if (!head_out<true>(Ha, Hc, ha.w2, ha.b2, hc.w2, hc.b2, B, b, l0, l1, vv)) return;
    const int a = draw_action(l0, l1, k0, k1, step, env_base + (uint64_t)b, lp0, lp1);
    const float p0 = expf(lp0), p1 = expf(lp1);
    action[b] = a;
    if (logp) logp[b] = a ? lp1 : lp0;
    if (value) value[b] = vv;
    if (entropy) entropy[b] = -fmaf(p0, lp0, p1 * lp1);          // contraction written out: it fixes the rounding
    if (logits_out) { logits_out[2 * b] = l0; logits_out[2 * b + 1] = l1; }
}

// uavpolicy_act: the actor half of heads_out_kernel.  greedy = 1 takes argmax, a tie going to action 0 (torch.argmax).
// The critic's head-hidden rows are stale in this mode and are not read.
__global__ void __launch_bounds__(256) actor_out_kernel(const __nv_bfloat16 *__restrict__ Ha, HeadW ha, int B, int greedy,
                                                        uint32_t k0, uint32_t k1, uint64_t step, uint64_t env_base,
                                                        int64_t *__restrict__ action, float *__restrict__ logp,
                                                        float *__restrict__ logits_out) {
    int b;
    float l0, l1, unused, lp0, lp1;
    if (!head_out<false>(Ha, nullptr, ha.w2, ha.b2, nullptr, nullptr, B, b, l0, l1, unused)) return;
    int a = draw_action(l0, l1, k0, k1, step, env_base + (uint64_t)b, lp0, lp1);
    if (greedy) a = l1 > l0 ? 1 : 0;
    action[b] = a;
    if (logp) logp[b] = a ? lp1 : lp0;
    if (logits_out) { logits_out[2 * b] = l0; logits_out[2 * b + 1] = l1; }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side

struct uavpolicy : capi::Handle {
    int max_batch = 0;
    float *w32 = nullptr;                 // private fp32 copy of the flat parameters
    __nv_bfloat16 *emb2_a = nullptr, *emb2_c = nullptr;   // [128 x 32] tensor-core form of the two embedding weights
    __nv_bfloat16 *wpk = nullptr;         // GEMM weights pre-packed in canonical order, each at pk(its offset in w32)
    __nv_bfloat16 *bpk = nullptr;         // their biases as [N x 16] B-operands (3 layers + 2 heads)
    BlockW actor, critic;
    HeadW actor_head, critic_head;
    __nv_bfloat16 *hh_actor = nullptr, *hh_critic = nullptr;   // [max_batch, 64] bf16: relu(W1 z + b1) of the two heads
    int *work_counter = nullptr;          // dynamic work-item counters of the two fused launches
    unsigned char *fused_scratch = nullptr;   // newest-token rows handed from the first fused launch to the second
    bool have_weights = false;
};

constexpr size_t UPK_SIZE = (size_t)UAVPOLICY_NUM_PARAMS + 64;   // packed copies live at (offset rounded up to 8 elements)
static inline size_t pk(size_t off) { return (off + 7) / 8 * 8; }   // 16 B aligned for the bulk TMA copy

extern "C" int uavpolicy_abi_version(void) { return UAVPOLICY_ABI_VERSION; }

extern "C" const char *uavpolicy_last_error(const uavpolicy_t *p) { return capi::last_error(p); }

extern "C" int uavpolicy_create(int32_t device, int32_t max_batch, uavpolicy_t **out) {
    uavpolicy *p;
    if (const int rc = capi::check_create_args("uavpolicy_create", "max_batch", max_batch, out)) return rc;
    if (const int rc = capi::new_handle("uavpolicy_create", device, p)) return rc;
    p->max_batch = max_batch;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = alloc(p, &p->w32, (size_t)UAVPOLICY_NUM_PARAMS);
    if (e == cudaSuccess) e = alloc(p, &p->hh_actor, (size_t)max_batch * HID);
    if (e == cudaSuccess) e = alloc(p, &p->hh_critic, (size_t)max_batch * HID);
    if (e == cudaSuccess) e = alloc(p, &p->work_counter, 2);
    if (e == cudaSuccess) e = alloc(p, &p->fused_scratch, uavp::fused_scratch_bytes(max_batch));
    if (e == cudaSuccess) e = cudaMemset(p->fused_scratch, 0, uavp::fused_scratch_bytes(max_batch));
    if (e == cudaSuccess) e = alloc(p, &p->wpk, (size_t)UPK_SIZE);
    if (e == cudaSuccess) e = alloc(p, &p->bpk, (size_t)3 * uavp::kLayerBiasElems + 2 * HID * uavp::kBiasK);
    if (e == cudaSuccess) e = alloc(p, &p->emb2_a, (size_t)D * 32);
    if (e == cudaSuccess) e = alloc(p, &p->emb2_c, (size_t)D * 32);
    if (e != cudaSuccess) return capi::abandon_handle(p, fail(p, -2, "uavpolicy_create: %s", cudaGetErrorString(e)));
    if (uavp::fused_block_prepare() != 0)
        return capi::abandon_handle(p, fail(p, -2, "uavpolicy_create: cannot reserve shared memory for the fused kernel"));
    bind_fp32(p->actor, p->actor_head, kActorOff, p->w32);
    bind_fp32(p->critic, p->critic_head, kCriticOff, p->w32);
    p->actor.emb_w2p = p->emb2_a; p->critic.emb_w2p = p->emb2_c;
    {   // packed GEMM weights, and the bias operands: layers of the actor, then of the critic, then the two heads
        __nv_bfloat16 *q = p->bpk;
        auto packed = [&](size_t off) { return p->wpk + pk(off); };
        const NetOff *offs[2] = {&kActorOff, &kCriticOff};
        BlockW *blocks[2] = {&p->actor, &p->critic};
        for (int n = 0; n < 2; ++n)
            for (int l = 0; l < blocks[n]->layers; ++l) {
                LayerW &L = blocks[n]->layer[l];
                const LayerOff &o = offs[n]->layer[l];
                L.in_wp = packed(o.in_w); L.out_wp = packed(o.out_w); L.l1_wp = packed(o.l1_w); L.l2_wp = packed(o.l2_w);
                L.in_bp = q; q += 3 * D * uavp::kBiasK;
                L.out_bp = q; q += D * uavp::kBiasK;
                L.l1_bp = q; q += FF * uavp::kBiasK;
                L.l2_bp = q; q += D * uavp::kBiasK;
            }
        p->actor_head.w1p = packed(kActorOff.head.w1); p->critic_head.w1p = packed(kCriticOff.head.w1);
        p->actor_head.b1p = q; q += HID * uavp::kBiasK;
        p->critic_head.b1p = q;
    }
    *out = p;
    return 0;
}

extern "C" int uavpolicy_destroy(uavpolicy_t *p) { return capi::destroy_handle(p); }

extern "C" int uavpolicy_set_weights(uavpolicy_t *p, const float *d_flat_params, void *stream) {
    if (!p || !d_flat_params) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    CU_TRY(p, cudaSetDevice(p->device));
    CU_TRY(p, cudaMemcpyAsync(p->w32, d_flat_params, (size_t)UAVPOLICY_NUM_PARAMS * sizeof(float), cudaMemcpyDeviceToDevice, s));
    // canonical-order copies of every GEMM weight for the fused kernel's bulk-TMA staging
    for (const GemmW &w : kGemmW.w)
        pack_canon_kernel<<<(w.N * w.K + 255) / 256, 256, 0, s>>>(p->w32 + w.off, p->wpk + pk(w.off), w.N, w.K);
    {
        auto packb = [&](const __nv_bfloat16 *dst, const float *bias, int N) {
            pack_bias_kernel<<<(N * 16 + 255) / 256, 256, 0, s>>>(bias, const_cast<__nv_bfloat16 *>(dst), N);
        };
        const BlockW *blocks[2] = {&p->actor, &p->critic};
        for (const BlockW *b : blocks)
            for (int l = 0; l < b->layers; ++l) {
                const LayerW &L = b->layer[l];
                packb(L.in_bp, L.in_b, 3 * D); packb(L.out_bp, L.out_b, D); packb(L.l1_bp, L.l1_b, FF); packb(L.l2_bp, L.l2_b, D);
            }
        packb(p->actor_head.b1p, p->actor_head.b1, HID);
        packb(p->critic_head.b1p, p->critic_head.b1, HID);
    }
    emb_w2_kernel<<<(D * 32 + 255) / 256, 256, 0, s>>>(p->actor.emb_w, p->actor.emb_b, p->emb2_a);
    emb_w2_kernel<<<(D * 32 + 255) / 256, 256, 0, s>>>(p->critic.emb_w, p->critic.emb_b, p->emb2_c);
    CU_TRY(p, cudaGetLastError());
    p->have_weights = true;
    return 0;
}

extern "C" int uavpolicy_get_action(uavpolicy_t *p, const float *d_obs, int32_t B, uint64_t seed, uint64_t step,
                                    uint64_t env_id_base, int64_t *d_action, float *d_logp, float *d_value,
                                    float *d_entropy, float *d_logits, void *stream) {
    if (!p) return -1;
    if (!d_obs || !d_action) return fail(p, -1, "uavpolicy_get_action: obs / action must be non-NULL");
    if (B <= 0 || B > p->max_batch) return fail(p, -1, "uavpolicy_get_action: B=%d outside (0, %d]", B, p->max_batch);
    if (!p->have_weights) return fail(p, -4, "uavpolicy_get_action before uavpolicy_set_weights");
    CU_TRY(p, cudaSetDevice(p->device));
    const cudaStream_t s = (cudaStream_t)stream;
    // two fused launches (actor block + head layer 1, critic block + head layer 1), then the per-sample outputs
    if (uavp::launch_fused_blocks(d_obs, B, p->actor, p->actor_head, p->hh_actor, p->critic, p->critic_head, p->hh_critic,
                                  p->work_counter, p->fused_scratch, s))
        return fail(p, -2, "fused block launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    heads_out_kernel<<<(B + 255) / 256, 256, 0, s>>>(p->hh_actor, p->hh_critic, p->actor_head, p->critic_head, B, (uint32_t)seed,
                                                     (uint32_t)(seed >> 32), step, env_id_base, d_action, d_logp, d_value,
                                                     d_entropy, d_logits);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

extern "C" int uavpolicy_act(uavpolicy_t *p, const float *d_obs, int32_t B, int32_t mode, uint64_t seed, uint64_t step,
                             uint64_t env_id_base, int64_t *d_action, float *d_logp, float *d_logits, void *stream) {
    // the checks that need no handle come first, so that they report their own message
    if (!d_obs || !d_action) return fail(p, -1, "uavpolicy_act: obs / action must be non-NULL");
    if (B <= 0) return fail(p, -1, "uavpolicy_act: B=%d must be > 0", B);
    if (mode != UAVPOLICY_ACT_SAMPLE && mode != UAVPOLICY_ACT_GREEDY)
        return fail(p, -1, "uavpolicy_act: mode %d is neither 0 (sample) nor 1 (greedy)", mode);
    if (!p) return fail(p, -1, "uavpolicy_act: handle is NULL");
    if (B > p->max_batch) return fail(p, -1, "uavpolicy_act: B=%d outside (0, %d]", B, p->max_batch);
    if (!p->have_weights) return fail(p, -1, "uavpolicy_act before uavpolicy_set_weights");
    CU_TRY(p, cudaSetDevice(p->device));
    const cudaStream_t s = (cudaStream_t)stream;
    if (uavp::launch_fused_blocks(d_obs, B, p->actor, p->actor_head, p->hh_actor, p->critic, p->critic_head, p->hh_critic,
                                  p->work_counter, p->fused_scratch, s, /*actor_only=*/true))
        return fail(p, -2, "fused block launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    actor_out_kernel<<<(B + 255) / 256, 256, 0, s>>>(p->hh_actor, p->actor_head, B, mode == UAVPOLICY_ACT_GREEDY, (uint32_t)seed,
                                                     (uint32_t)(seed >> 32), step, env_id_base, d_action, d_logp, d_logits);
    CU_TRY(p, cudaGetLastError());
    return 0;
}
