/*
 * uavpolicy_b200.h - C ABI of the sm_100a rollout forward of the policy / value network.
 *
 * Replaces TransformerActorCritic.get_action (networks/transformer_net.py:96-122) as called once per rollout
 * step by PPOAgent.select_action (agents/ppo.py:52-62): for a batch of observation windows [B,5,14] it returns
 * the sampled action, its log-probability, the state value and the policy entropy.  All dense contractions run
 * on the 5th-generation tensor cores (tcgen05.mma, operands staged by TMA, fp32 accumulators in TMEM; bf16
 * operands) in the two hand-written fused encoder-block kernels of csrc/policy_fused.cu, which keep the activations
 * of a tile in shared memory / TMEM across the embedding, all layers and the first head layer; one more kernel
 * (csrc/policy_forward.cu) forms the second head layers and the sample.  No CUTLASS, cuBLAS or other library kernel
 * is on the path.
 *
 * Conventions as in uavenv_b200.h: 0 on success, negative error code otherwise; d_ = device pointers; work is
 * enqueued on the caller's stream; a handle is not thread-safe; no CPU fallback.
 */
#ifndef UAVPOLICY_B200_H
#define UAVPOLICY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UAVPOLICY_NUM_PARAMS 419267 /* parameters of TransformerActorCritic (SURVEY.md section 2) */

typedef struct uavpolicy uavpolicy_t;

/* max_batch: largest B the handle will be called with (activation workspaces are allocated once). */
int uavpolicy_create(int32_t device, int32_t max_batch, uavpolicy_t **out);
int uavpolicy_destroy(uavpolicy_t *p);
const char *uavpolicy_last_error(const uavpolicy_t *p);
/* version of this ABI (struct layouts, argument lists); the Python binding refuses a library that reports another */
#define UAVPOLICY_ABI_VERSION 3
int uavpolicy_abi_version(void);

/* Load the network weights from ONE flat fp32 device buffer holding every parameter in
 * `TransformerActorCritic.named_parameters()` order (== state_dict order of the reference network):
 *   actor_net.{pos_embedding[5*128], embedding.0.{weight[128*14], bias[128]},
 *              transformer.layers.0.{self_attn.in_proj_weight[384*128], in_proj_bias[384], out_proj.{weight[128*128],
 *              bias[128]}, linear1.{weight[256*128], bias[256]}, linear2.{weight[128*256], bias[128]},
 *              norm1.{weight,bias}[128], norm2.{weight,bias}[128]}},
 *   actor_head.{0.{weight[64*128], bias[64]}, 2.{weight[2*64], bias[2]}},
 *   critic_net.{... as actor_net with layers.0 and layers.1}, critic_head.{0.{...}, 2.{weight[64], bias[1]}}
 * GEMM weights are converted to bf16, everything else stays fp32. */
int uavpolicy_set_weights(uavpolicy_t *p, const float *d_flat_params, void *stream);

/* get_action for B windows.  d_obs [B,5,14] f32 (rows that are entirely zero are padding, except the newest row:
 * transformer_net.py:52-54).  The action of env b is drawn from Categorical(softmax(logits_b)) with a counter RNG
 * keyed (seed, step, env_id_base + b).  Outputs (each may be NULL except d_action): d_action [B] int64,
 * d_logp [B], d_value [B], d_entropy [B], d_logits [B,2]. */
int uavpolicy_get_action(uavpolicy_t *p, const float *d_obs, int32_t B, uint64_t seed, uint64_t step,
                         uint64_t env_id_base, int64_t *d_action, float *d_logp, float *d_value, float *d_entropy,
                         float *d_logits, void *stream);

/* self-test of the hand-written tcgen05 path: D[128,N] (f32) = A[128,K] W[N,K]^T for one 128-row tile
 * (A, W bf16 row-major on the device; N <= 384, N % 16 == 0; K = 128 or 256). */
int uavpolicy_selftest_gemm_tile(const void *d_A, const void *d_W, float *d_D, int32_t N, int32_t K, void *stream);

/* ---- PPO update: forward + backward of the two transformer trunks (csrc/policy_train.cu) ---------------------
 * Replaces the trunk part of policy.evaluate(state, action) (networks/transformer_net.py:124-143 -> :47-65, called
 * from agents/ppo.py:126) and of loss.backward() (agents/ppo.py:157) for a minibatch of n windows.  bf16 activations
 * and GEMM operands with fp32 accumulation, fp32 LayerNorm / softmax / parameter gradients.  The MLP heads and the
 * loss stay with the caller: features out, feature gradients in. */
typedef struct uavtrain uavtrain_t;

int uavtrain_create(int32_t device, int32_t max_samples, uavtrain_t **out);
int uavtrain_destroy(uavtrain_t *p);
const char *uavtrain_last_error(const uavtrain_t *p);   /* p may be NULL (create failures) */

/* d_flat_params: the UAVPOLICY_NUM_PARAMS fp32 parameters in uavpolicy_set_weights order (read in place; must stay
 * valid and unchanged until the matching uavtrain_backward returned); d_obs [n,5,14] f32 (likewise);
 * d_feat [n,2,128] f32 out: last-token features of the actor trunk ([:,0,:]) and of the critic trunk ([:,1,:]),
 * i.e. the inputs of actor_head / critic_head (transformer_net.py:106,114). */
int uavtrain_forward(uavtrain_t *p, const float *d_flat_params, const float *d_obs, int32_t n, float *d_feat, void *stream);

/* d_dfeat [n,2,128] f32: gradient of the loss w.r.t. d_feat.  d_flat_grad [UAVPOLICY_NUM_PARAMS] f32 is OVERWRITTEN:
 * trunk parameter gradients at their parameter offsets, zeros at the head parameters' offsets. */
int uavtrain_backward(uavtrain_t *p, const float *d_dfeat, float *d_flat_grad, void *stream);

/* The same with the two MLP heads inside (transformer_net.py:78-91,106-115): d_logits [n,2] f32 = actor_head(actor
 * features), d_value [n] f32 = critic_head(critic features).  The backward takes the loss gradients w.r.t. both and
 * OVERWRITES d_flat_grad with the gradient of every parameter, heads included. */
int uavtrain_forward_heads(uavtrain_t *p, const float *d_flat_params, const float *d_obs, int32_t n, float *d_logits,
                           float *d_value, void *stream);
int uavtrain_backward_heads(uavtrain_t *p, const float *d_dlogits, const float *d_dvalue, float *d_flat_grad, void *stream);

/* PPO loss of agents/ppo.py:126-153 on the heads' outputs, value and gradient in one call:
 *   L = -mean(min(r A, clip(r, 1-eps, 1+eps) A)) + c_value * max(mean((v-R)^2), mean((v_clip-R)^2)) - c_entropy * mean(H)
 * with r = exp(log pi(a|s) - old_logp), v_clip = old_value + clip(v - old_value, -eps, eps).  All arrays [n] f32 on the
 * device except d_logits / d_dlogits [n,2] and d_action [n] int64.  Out: d_dlogits, d_dvalue = dL/dlogits, dL/dvalue
 * (ready for uavtrain_backward_heads); d_stats (optional) [3] = {actor loss, critic loss, mean entropy} (ppo.py:162-168). */
int uavtrain_ppo_loss(uavtrain_t *p, const float *d_logits, const float *d_value, const int64_t *d_action, const float *d_old_logp,
                      const float *d_adv, const float *d_ret, const float *d_old_value, int32_t n, float eps_clip, float c_value,
                      float c_entropy, float *d_dlogits, float *d_dvalue, float *d_stats, void *stream);

/* self-test of the hand-written dense-layer kernel (csrc/policy_dense.cu: persistent, TMA-fed tcgen05 GEMM with fused
 * epilogues): d_out[M,N] (bf16, dense) = act(d_a[M,K] d_w[N,K]^T + d_bias[N]); bf16 row-major inputs, row stride lda of
 * d_a (elements, multiple of 8); N in {64,128,256,384}, K a multiple of 64 <= 384, N*K*2 <= 96 KiB.  act: 0 identity,
 * 1 ReLU, 2 ReLU backward (no bias; the product is zeroed where d_aux[M,N] (bf16, row stride ld_aux) is not > 0). */
int uavpolicy_selftest_dense(const void *d_a, int64_t lda, const void *d_w, const float *d_bias, const void *d_aux,
                             int64_t ld_aux, void *d_out, int32_t M, int32_t N, int32_t K, int32_t act, void *stream);

/* the same kernel with the residual + LayerNorm epilogue of a post-LN encoder layer (networks/transformer_net.py:34-43):
 * d_out[M,128] = LayerNorm(d_x[M,128] + d_a[M,K] d_w[128,K]^T + d_bias) * d_gamma + d_beta (eps 1e-5), d_xhat[M,128] (bf16) =
 * the normalised rows and d_rstd[M] (fp32) = 1/sigma, which the backward keeps.  d_x: bf16 with row stride ldx. */
int uavpolicy_selftest_dense_ln(const void *d_a, int64_t lda, const void *d_w, const float *d_bias, const void *d_x, int64_t ldx,
                                const float *d_gamma, const float *d_beta, void *d_out, void *d_xhat, float *d_rstd, int32_t M,
                                int32_t K, void *stream);

/* self-test of the tcgen05 weight-gradient kernel (csrc/policy_wgrad.cu): d_dw[n_out,k_in] (f32) +=
 * dY[rows,n_out]^T X[rows,k_in]; bf16 row-major inputs with row strides ld_dy / ld_x (elements, multiples of 8);
 * n_out % 128 == 0, k_in = 128 or 256.  d_dbias (optional, k_in = 128): d_dbias[n_out] += column sums of dY. */
int uavpolicy_selftest_wgrad(const void *d_dy, int64_t ld_dy, const void *d_x, int64_t ld_x, int32_t rows, int32_t n_out,
                             int32_t k_in, float *d_dw, float *d_dbias, void *stream);

#ifdef __cplusplus
}
#endif
#endif
