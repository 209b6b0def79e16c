/*
 * uavpolicy_eval_b200.h - C ABI of the actor-only policy forward used to evaluate a checkpoint.
 *
 * An evaluation needs the action and nothing else: the value head, the entropy and the two-layer critic trunk, which
 * is most of uavpolicy_get_action's work, are skipped.  The same two fused tcgen05 launches run with the actor's work
 * items only (csrc/policy_fused.cu), then one kernel forms the actor's second head layer in fp32 and picks the action.
 * The handle is the uavpolicy_t of uavpolicy_b200.h; conventions are those of that header.
 */
#ifndef UAVPOLICY_EVAL_B200_H
#define UAVPOLICY_EVAL_B200_H

#include <stdint.h>

#include "uavpolicy_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define UAVPOLICY_ACT_SAMPLE 0 /* draw from Categorical(softmax(logits)), the counter RNG of uavpolicy_get_action */
#define UAVPOLICY_ACT_GREEDY 1 /* argmax of the logits; a tie goes to action 0, as torch.argmax */

/* Action of the actor for B windows d_obs [B,5,14] f32 (padding rows as in uavpolicy_get_action).
 * mode UAVPOLICY_ACT_SAMPLE draws with the key (seed, step, env_id_base + b): the action and d_logp are bit-identical
 * to uavpolicy_get_action's for the same keys and observations.  Outputs: d_action [B] int64 (required), d_logp [B] f32
 * log-probability of the chosen action (may be NULL), d_logits [B,2] f32 (may be NULL; bit-identical to
 * uavpolicy_get_action's).  Returns -1 with a message for B outside [1, max_batch], another mode, a NULL d_obs /
 * d_action or a handle without weights; the GPU is not touched then. */
int uavpolicy_act(uavpolicy_t *p, const float *d_obs, int32_t B, int32_t mode, uint64_t seed, uint64_t step,
                  uint64_t env_id_base, int64_t *d_action, float *d_logp, float *d_logits, void *stream);

#ifdef __cplusplus
}
#endif
#endif
