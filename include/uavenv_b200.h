/*
 * uavenv_b200.h - C ABI of the B200-native batched UAV->target allocation environment.
 *
 * This is the drop-in boundary for the rollout path of
 * Dingyf717/target-allocation-ppo-transformer (SURVEY.md §8b).  Each entry point names the
 * reference interface it replaces (file:line under the reference tree).  The reference is pure
 * Python, so the binding a maintainer adds is a ctypes stub (INTEGRATION.md); the same symbols can
 * be bound from any FFI: plain pointers, sizes and C structs only - no torch / C++ types.
 *
 * Conventions
 *   - every function returns 0 on success and a negative UAVENV_E* code on failure; the message is
 *     available from uavenv_last_error().  No C++ exception crosses the boundary.
 *   - pointers prefixed d_ are DEVICE pointers on the handle's device, h_ are HOST pointers.
 *   - all device work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as
 *     void*; NULL = the legacy default stream).  No call synchronises unless stated.
 *   - a handle is not thread-safe; use one handle per device / per host thread.
 *   - B = num_envs, N = num_uavs, M = num_targets, K1 = num_nfz, K2 = num_interceptors.
 *   - there is no CPU fallback: creation fails when no CUDA device is usable.
 */
#ifndef UAVENV_B200_H
#define UAVENV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UAVENV_ABI_VERSION 2
#define UAVENV_STATE_DIM 14 /* configs/config.py:61 STATE_DIM */
#define UAVENV_SEQ_LEN 5    /* configs/config.py:62 SEQ_LEN   */

enum {
    UAVENV_OK = 0,
    UAVENV_EINVAL = -1,  /* bad argument                         */
    UAVENV_ECUDA = -2,   /* a CUDA runtime call / launch failed  */
    UAVENV_ENOMEM = -3,  /* host or device allocation failed     */
    UAVENV_ESTATE = -4   /* call not valid in the current state  */
};

/* The constants the path reads from the reference's `cfg` singleton (configs/config.py:7-12,33-58,
 * 61-63,83) plus the batching knobs the reference has no need for. */
typedef struct uavenv_cfg {
    int32_t num_uavs;         /* NUM_UAVS            :42 */
    int32_t num_targets;      /* NUM_TARGETS         :43 */
    int32_t num_nfz;          /* NUM_NFZ             :48 */
    int32_t num_interceptors; /* NUM_INTERCEPTORS    :49 */
    int32_t reset_episodes;   /* RESET_EPISODES      :83 ; main_train.py:79 schedule. <=0: never regenerate */
    int32_t auto_reset;       /* 1: finished envs restart inside the same step launch (batched use);
                                 0: they stay finished until uavenv_reset (reference single-env contract) */
    double param_zeta_d;      /* PARAM_ZETA_D        :7  */
    double param_k;           /* PARAM_K             :8  */
    double param_c1, param_c2, param_c3, param_c4; /* :9-12 */
    double cost_weight_omega; /* COST_WEIGHT_OMEGA   :53 */
    double weather_speed_factor, weather_load_factor; /* :57-58 */
    double map_width, map_height;                  /* :33-34 */
    double uav_gen_x_lo, uav_gen_x_hi;             /* UAV_GEN_X_RANGE    :39 */
    double target_gen_x_lo, target_gen_x_hi;       /* TARGET_GEN_X_RANGE :40 */
    double intercept_rad;                          /* INTERCEPT_RAD      :50 */
    double tie_band;          /* Eq.21 `new_r >= prev_r` (envs/uav_env.py:317) is decided from carried sums; when the two
                                 rewards agree to within tie_band * max(|new_r|, |prev_r|) both are re-summed over the targets
                                 in the reference's list order (uav_env.py:244-269) and THAT decides.  Default 1e-12 (the carried
                                 sums are good to ~1e-14); a huge value takes the exact path always (tests) */
} uavenv_cfg_t;

/* Per-step diagnostics = the `info` dict of envs/uav_env.py:426-433, one value per env.
 * Every pointer is a device array of length B and may be NULL (not wanted). */
typedef struct uavenv_info {
    float *d_J_val;           /* "J_val"           */
    int32_t *d_num_assigned;  /* "num_assigned" = covered-target count N0 */
    int8_t *d_is_valid_action;/* "is_valid_action": -1 = None, 0 = False, 1 = True */
    float *d_avg_p_dmg;       /* "avg_p_dmg"       */
    float *d_avg_p_final;     /* "avg_p_final"     */
    double *d_reward_f64;     /* extension: the step reward before the cast to float */
} uavenv_info_t;

/* Scene of `count` consecutive envs as HOST structure-of-arrays in the reference's list order
 * (targets AFTER the shuffle of envs/uav_env.py:173), env-major: field[e*N + i].
 * = the public attributes env.uavs / env.targets / env.nfz_list / env.interceptors
 * (envs/uav_env.py:27-30, envs/entities.py:13-61).  On load, uav_type / nfz_radius may be NULL. */
typedef struct uavenv_scene {
    double *uav_x, *uav_y, *uav_vx, *uav_vy, *uav_load, *uav_cost; /* [count*N]  */
    int32_t *uav_type;                                               /* [count*N]  */
    double *tgt_x, *tgt_y, *tgt_vx, *tgt_vy, *tgt_value;            /* [count*M]  */
    int32_t *tgt_id;                                                 /* [count*M]  */
    double *nfz_x, *nfz_y, *nfz_radius;                              /* [count*K1] */
    double *int_x, *int_y, *int_vx, *int_vy;                         /* [count*K2] */
} uavenv_scene_t;

/* Mutable allocation state of `count` consecutive envs (HOST arrays; any pointer may be NULL).
 * = uav_idx / target_idx (envs/uav_env.py:33-34), UAV.assigned_target_id (entities.py:30),
 * len(Target.locked_by_uavs) (entities.py:46) and the running objective. */
typedef struct uavenv_state {
    int32_t *uav_idx, *target_idx;     /* [count]    */
    int32_t *assigned_target_id;       /* [count*N], -1 = unassigned */
    int32_t *lock_count;               /* [count*M], list order      */
    double *not_hit, *not_hit_pure;    /* [count*M]  prod(1-p_final), prod(1-p_damage) over the lock list */
    double *J_val;                     /* [count]    envs/uav_env.py:244-269 */
    int32_t *episode, *scene_index;    /* [count]    1-based episode counter, scenes generated so far */
    uint8_t *finished;                 /* [count]    only ever 1 with auto_reset = 0 */
} uavenv_state_t;

typedef struct uavenv uavenv_t;

/* configs/config.py defaults (the live "easy mode" file) with reset_episodes = 200, auto_reset = 1 */
void uavenv_default_cfg(uavenv_cfg_t *cfg);

/* replaces UAVEnv.__init__ (envs/uav_env.py:14-40).  Allocates every device array once;
 * `seed` keys the counter-based scene generator and `env_id_base` is the GLOBAL id of env 0 of
 * this handle, so a shard [base, base+B) reproduces the same envs on any GPU count. */
int uavenv_create(const uavenv_cfg_t *cfg, int32_t num_envs, int32_t device, uint64_t seed,
                  uint64_t env_id_base, uavenv_t **out);
int uavenv_destroy(uavenv_t *h);
/* message of the last failure on this handle; with h NULL, of this thread's last failure that had no handle: a
 * uavenv_create, or a call without a handle (uavenv_episode_accumulate, the ppo_* entry points) */
const char *uavenv_last_error(const uavenv_t *h);
int uavenv_abi_version(void);
int32_t uavenv_num_envs(const uavenv_t *h);

/* replaces UAVEnv.reset(full_reset) (envs/uav_env.py:42-63) for the envs whose d_env_mask byte is
 * non-zero (NULL = all).  full_reset != 0: _generate_scene (uav_env.py:65-173) with the counter
 * RNG; 0: _reset_state_only (:175-182).  Writes the first observation window (4 zero rows + the
 * row of pointer pair (0,0)) to d_obs[B,5,14] for the reset envs; d_obs may be NULL. */
int uavenv_reset(uavenv_t *h, int32_t full_reset, const uint8_t *d_env_mask, float *d_obs, void *stream);

/* replaces UAVEnv.step(action) (envs/uav_env.py:295-435) for all B envs in ONE kernel launch.
 * d_actions[B] int64 (the dtype torch.distributions.Categorical.sample() yields): 1 = Assign,
 * anything else = Skip (:344).  Outputs: d_obs[B,5,14] f32, d_reward[B] f32, d_done[B] u8, info.
 * With auto_reset the observation of a finished env is the first window of its next episode
 * (reference: a zero row the training loop never reads, :188-189); without it the window is zero. */
int uavenv_step(uavenv_t *h, const int64_t *d_actions, float *d_obs, float *d_reward, uint8_t *d_done,
                const uavenv_info_t *info, void *stream);

/* same step through HOST buffers (the reference's caller lives on the host: main_train.py:111-113):
 * moves h_actions host->device, steps, moves reward/done back and synchronises the stream.  Pinned,
 * device-mapped host buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are read and written
 * in place by the fused kernel over PCIe; pageable buffers go through staging copies.
 * The observation window stays on the device (d_obs, or the handle's own buffer when NULL -
 * see uavenv_obs_buffer) where the policy consumes it. */
int uavenv_step_host(uavenv_t *h, const int64_t *h_actions, float *h_reward, uint8_t *h_done, float *d_obs,
                     void *stream);
/* the same with one byte per action (the action space is {0,1}, envs/uav_env.py:18): 8x less PCIe traffic */
int uavenv_step_host_i8(uavenv_t *h, const int8_t *h_actions, float *h_reward, uint8_t *h_done, float *d_obs,
                        void *stream);
float *uavenv_obs_buffer(uavenv_t *h); /* device [B,5,14] owned by the handle */

/* replaces assigning env.uavs / env.targets / env.nfz_list / env.interceptors by hand: injects
 * scenes (e.g. exported from the reference) into envs [first_env, first_env+count) and leaves them
 * in the reset(full_reset=False) state, episode 1; their first observation windows are written to
 * d_obs[B,5,14] (rows of the loaded envs only; NULL = the handle's own buffer).  Synchronous. */
int uavenv_load_scene(uavenv_t *h, const uavenv_scene_t *scene, int32_t first_env, int32_t count, float *d_obs);
/* the same from DEVICE arrays, with replication: d_scene holds num_scenes scenes as device structure-of-arrays (fields
 * and layout of uavenv_scene_t, scene-major).  Scene s goes to envs first_env + s*copies + c, c in [0, copies), which are
 * left as uavenv_load_scene leaves them (reset, episode 1); their first windows are written to d_obs (NULL = the handle's
 * buffer).  Asynchronous on `stream`: the scene arrays must stay valid until the work enqueued there has run.  Returns
 * UAVENV_EINVAL before the GPU is touched on a NULL required array, copies <= 0 or a range outside [0, B). */
int uavenv_load_scene_device(uavenv_t *h, const uavenv_scene_t *d_scene, int32_t num_scenes, int32_t copies,
                             int32_t first_env, float *d_obs, void *stream);
/* replaces reading env.uavs / env.targets / ... (main.py:35-42, test_visualize.py:61-94). Synchronous. */
int uavenv_get_scene(uavenv_t *h, uavenv_scene_t *scene, int32_t first_env, int32_t count);
int uavenv_get_state(uavenv_t *h, uavenv_state_t *state, int32_t first_env, int32_t count);

/* restores the 1-based per-env episode counters that drive the main_train.py:79 regeneration
 * schedule (resume of a run; staggered steady state for benchmarks).  h_episode[count] is a HOST
 * array.  Synchronous. */
int uavenv_set_episode_counters(uavenv_t *h, const int32_t *h_episode, int32_t first_env, int32_t count);

/* replaces the double loop over mechanics.calc_advantage of main.py:38-45 (mechanics.py:167-181):
 * p_final / p_damage for every (env, UAV, target), [B,N,M] list order.  Either pair may be NULL. */
int uavenv_score_matrix(uavenv_t *h, float *d_p_final, float *d_p_damage, void *stream);
int uavenv_score_matrix_f64(uavenv_t *h, double *d_p_final, double *d_p_damage, void *stream);

/* re-derives every running aggregate (J, N0, cost / value sums) from the per-target products with
 * a warp per env, exactly as envs/uav_env.py:244-293 sums them; writes the largest |carried-fresh|
 * J difference seen to *h_max_abs_diff (may be NULL).  Synchronous.  Used to bound drift. */
int uavenv_recompute_objective(uavenv_t *h, double *h_max_abs_diff, void *stream);

/* Bernoulli(1/2) actions keyed (action_seed, step, global env id): the synthetic action stream of
 * the env-only benchmarks (SURVEY.md §8d) */
int uavenv_random_actions(uavenv_t *h, uint64_t action_seed, uint64_t step, int64_t *d_actions, void *stream);

/* Actions of the best-target heuristic, an evaluation baseline: at the pointer (k, m) UAV k Assigns iff m is the target
 * j* that maximises the paper reward (Eq.19) after a tentative assignment of UAV k (lowest index on a tie), and that
 * reward is not below the current one (csrc/uavenv_kernels.cuh states the rule).  d_cache: device int64 [B], caller-owned,
 * zeroed before the first call; it keeps j* per env keyed by (episode counter, UAV pointer), so j* is computed once per
 * UAV row, and auto-resets, new rows and skipped calls are detected.  uavenv_reset(full_reset = 1) and uavenv_load_scene
 * restart the episode counter at 1: zero d_cache after them unless the next call is made before the next step.
 * d_actions: device int64 [B].  Call on the env's stream after a step and before the next one. */
int uavenv_best_target_actions(uavenv_t *h, int64_t *d_cache, int64_t *d_actions, void *stream);

/* Best-of-K read-out (a handle with auto_reset = 0, whose finished envs keep their final allocation).  For the groups
 * g in [0, num_groups) of group_size consecutive envs starting at first_env: the member with the highest
 * J = rev - omega * cost_sum (the value uavenv_get_state reports as J_val, bit for bit), the lowest member index winning a
 * tie.  d_best[g] (int32, member index within the group), d_J_best[g] (its J), d_assigned_best[g*N + i] (its
 * assigned_target_id row: Target.id, -1 = unassigned) and d_num_covered[g] (its covered-target count N0).  d_J_all
 * [num_groups*group_size] (may be NULL) receives every member's J.  A group with a member that has not finished gets
 * d_best = -1, d_J_best = NaN, d_num_covered = -1 and a row of -1.  All outputs are device arrays; one launch on
 * `stream`, asynchronous.  UAVENV_EINVAL (before the GPU is touched) on a NULL output or a range outside [0, B);
 * UAVENV_ESTATE on a handle with auto_reset = 1 or before any reset / scene load. */
int uavenv_group_best(uavenv_t *h, int32_t first_env, int32_t num_groups, int32_t group_size, int32_t *d_best,
                      double *d_J_best, int32_t *d_assigned_best, int32_t *d_num_covered, double *d_J_all, void *stream);

/* Steepest-ascent local search on allocations of the scenes held by envs first_env + s*env_stride, s in [0, count).
 * Row s of d_assigned_in [count*N] (group_best's layout: Target.id, -1 = none) is the start; the search maximises
 *   J = sum_j value_j * (1 - prod_{k -> j} (1 - p[k][j])) - omega * sum_{k assigned} cost_k
 * with p[k][j] = damage_prob(uav k, target j) * p_pen_k in fp64, list order (the bits of uavenv_score_matrix_f64's
 * p_final).  t(k) is UAV k's target position (-1 = none), nh_j the product over the UAVs on j and nh_excl_k the product
 * over the OTHER UAVs on t(k), each taken in ascending UAV index (never by dividing by 1 - p: p can be 1).  Candidates:
 *   move (k, b), b in {-1} u [0, M), b != a = t(k):
 *     gain = ([a>=0] v_a (nh_a - nh_excl_k) + [b>=0] (v_b nh_b) p[k][b]) + (omega c_k) ([a>=0] - [b>=0])
 *   swap (k1 < k2), a1 = t(k1) != a2 = t(k2), either may be -1; k1 takes a2 and k2 takes a1:
 *     gain = ([a1>=0] v_a1 (nh_a1 - nh_excl_k1 (1 - p[k2][a1])) + [a2>=0] v_a2 (nh_a2 - nh_excl_k2 (1 - p[k1][a2])))
 *            + (omega (c_k1 - c_k2)) ([a1>=0] - [a2>=0])     (the cost term is 0 unless one side is -1)
 * in that operation order.  Candidate order: moves before swaps, moves by ascending k then b from -1 up, swaps by
 * (k1, k2) lexicographic; the first candidate with the largest gain wins an exact tie.  A round applies the winner iff its
 * gain > 1e-12 * max(1, |J_run|), where J_run is J_in plus the gains applied so far; after a move the products of the
 * touched targets and their UAVs are recomputed from scratch.  The search stops when no candidate qualifies
 * (d_converged = 1: the row is a local optimum) or when a qualifying candidate is found after max_moves applied moves
 * (d_converged = 0).  Outputs per s: d_assigned_out row (may be d_assigned_in), d_J_in (may be NULL) and d_J_out - J from
 * scratch: products in ascending UAV index, targets summed in list order, then minus omega times the assigned UAVs'
 * costs summed in UAV order -, d_num_covered (N0, distinct targets), d_moves (applied moves).  A row holding an id below
 * -1 or one that is not a Target.id of its scene gets moves = -1, J_in = J_out = NaN, N0 = -1, converged = 0 and a row of
 * -1; other rows are unaffected.  max_moves = 0 returns the input rows with their J.  d_workspace: device memory of
 * uavenv_improve_workspace_bytes(h) bytes, not needed (may be NULL) when that is 0.  One launch on `stream`,
 * asynchronous; results do not depend on count, env_stride or the launch.  UAVENV_EINVAL (before the GPU is touched) on
 * a NULL required pointer or workspace, count <= 0, env_stride <= 0, max_moves < 0 or an env outside [0, B);
 * UAVENV_ESTATE before any reset / scene load. */
int uavenv_improve_allocation(uavenv_t *h, int32_t first_env, int32_t count, int32_t env_stride,
                              const int32_t *d_assigned_in, int32_t max_moves, int32_t *d_assigned_out, double *d_J_in,
                              double *d_J_out, int32_t *d_num_covered, int32_t *d_moves, uint8_t *d_converged,
                              void *d_workspace, void *stream);
/* bytes of the workspace uavenv_improve_allocation and uavenv_upper_bound need: 0 when p[N][M] fits the kernel's shared memory (N*M <= 8192),
 * otherwise N*M*8 per SM of the handle's device (L2-resident slices). */
size_t uavenv_improve_workspace_bytes(const uavenv_t *h);

/* Certified upper bound on the best J of the scenes held by envs first_env + s*env_stride, s in [0, count): no
 * allocation of scene s has J above d_bound[s].  With a_kj = min(-log1p(-p[k][j]), A), A = 40 (p as in
 * uavenv_improve_allocation; the cap keeps a finite where p = 1) and x_kj in {0,1}, sum_j x_kj <= 1, every allocation has
 *   J(x) <= F(x) + sum_j v_j e^-A,   F(x) = sum_j v_j (1 - exp(-sum_k a_kj x_kj)) - omega sum_k c_k sum_j x_kj
 * (where a cap is active, exp(-sum_k a_kj x_kj) <= e^-A, so target j loses at most v_j e^-A).  F is concave, so over the
 * relaxation x_kj in [0,1], sum_j x_kj <= 1, every feasible x gives F* <= F(x) + max_{vertex y} grad F(x).(y - x) =: U;
 * U is a valid bound at every feasible x, whatever the step sizes that reached it.  x enters only through
 * s_j = sum_k a_kj x_kj and C = sum_k c_k sum_j x_kj, which the iteration keeps (never x), in fp64:
 *   start s = 0, C = 0 (the empty allocation).  Iteration t = 1, 2, ...:
 *     nh_j = exp(-s_j), w_j = v_j nh_j;  F = sum_j v_j (1 - nh_j) - omega C, targets in list order;
 *     g_kj = w_j a_kj - omega c_k; UAV k picks j*_k = argmax_j g_kj (lowest j on a tie) if that maximum is > 0, else none;
 *     U_t = (F + sum_{k picks} g_kj*) - (sum_j w_j s_j - omega C), both sums in ascending index;
 *     stop if U_t - F <= 1e-9 max(1, |U_t|) (the relaxation is solved) or t = iters;
 *     sigma_j = sum_{k picks j} a_kj and C_sigma = sum_{k picks} c_k in ascending k; d = sigma - s, dC = C_sigma - C;
 *     gamma in [0,1] (every gamma keeps x feasible: validity never depends on it) maximises the concave
 *     phi(gamma) = F(s + gamma d, C + gamma dC) by: gamma = 1 if phi'(1) >= 0; otherwise lo = 0, hi = 1, gamma = 1 and
 *     up to 10 times { c = gamma - phi'(gamma)/phi''(gamma); stop if c == gamma (converged: without this test a
 *     sub-ulp step would land on the bracket end and send gamma to the midpoint); the midpoint of (lo, hi) unless
 *     lo < c < hi; gamma = c; phi'(gamma) > 0 ? lo = gamma : hi = gamma }, with phi'(gamma) = sum_j (v_j e_j) d_j - omega dC and
 *     -phi''(gamma) = sum_j ((v_j e_j) d_j) d_j, e_j = exp(-(s_j + gamma d_j)), each reduced over targets in a fixed
 *     order (csrc/uavenv_kernels.cuh, block_sum2);
 *     s += gamma d, C += gamma dC.
 * Outputs per s: d_bound = min_t U_t + (sum_j v_j) e^-A + 1e-12 (sum_j v_j + omega sum_k c_k) (the last term covers fp64
 * rounding), d_relaxed = F at the last iterate (d_bound - d_relaxed shows whether more iterations would help) and
 * d_iters = the iterations run (<= iters; iteration t takes no step when it stops).  d_workspace as for
 * uavenv_improve_allocation (uavenv_improve_workspace_bytes).  One launch on `stream`, asynchronous; results do not depend
 * on count, env_stride or the launch.  UAVENV_EINVAL (before the GPU is touched) on a NULL output or required workspace,
 * count <= 0, env_stride <= 0, iters < 1 or an env outside [0, B); UAVENV_ESTATE before any reset / scene load. */
int uavenv_upper_bound(uavenv_t *h, int32_t first_env, int32_t count, int32_t env_stride, int32_t iters, double *d_bound,
                       double *d_relaxed, int32_t *d_iters, void *d_workspace, void *stream);

/* ---- per-episode records of an evaluation (csrc/uavenv_episodes.cu) ---------------------------------------------
 * One finished episode.  ret sums the fp64 step rewards (info d_reward_f64) in step order; J_val, avg_p_dmg,
 * avg_p_final and num_assigned are the info of the episode's last step, i.e. of its final allocation. */
typedef struct uavenv_episode {
    double ret;
    float J_val, avg_p_dmg, avg_p_final;
    int32_t length;           /* steps of the episode */
    int32_t num_assigned;     /* covered targets N0 at the end */
    int32_t assigns;          /* steps with action == 1 */
    int32_t valid;            /* steps with is_valid_action == 1 (the reference's "valid assign") */
} uavenv_episode_t;           /* 40 bytes */

/* Running state of the episodes in progress: device arrays [B], zeroed by the caller before the first step, plus
 * d_envs_complete, one device int counting the envs that have recorded their quota. */
typedef struct uavenv_episode_acc {
    double *d_ret;
    int32_t *d_length, *d_assigns, *d_valid;
    int32_t *d_episodes;      /* episodes recorded so far per env */
    int32_t *d_envs_complete;
} uavenv_episode_acc_t;

/* Folds one step's d_actions [B], d_done [B] and info into acc (one thread per env, one launch).  When env b finishes
 * its k-th episode (k < episodes_per_env) the record goes to d_records[b * episodes_per_env + k]; later episodes are
 * dropped, and *d_envs_complete is incremented once, when env b records its last one.  Every info pointer must be
 * non-NULL; argument errors return UAVENV_EINVAL before the GPU is touched. */
int uavenv_episode_accumulate(int32_t B, const int64_t *d_actions, const uint8_t *d_done, const uavenv_info_t *info,
                              int32_t episodes_per_env, const uavenv_episode_acc_t *acc, uavenv_episode_t *d_records,
                              int32_t device, void *stream);

/* ---- PPO rollout post-processing (agents/ppo.py:77-94) ------------------------------------------
 * GAE(gamma, lambda) over a [T,B] rollout (time-major) followed by the global advantage
 * normalisation (mean, unbiased std, +1e-7).  d_last_value[B] is V(s_T) for bootstrapping (NULL = 0,
 * the reference's episodic case, ppo.py:77).  d_adv_stats (optional, device double[3]) receives
 * {count, sum, sum of squares} BEFORE normalisation so multi-GPU callers can all-reduce them and
 * call ppo_normalize_advantages themselves (normalize = 0). */
int ppo_gae_advantages(const float *d_rewards, const float *d_values, const uint8_t *d_dones,
                       const float *d_last_value, int32_t T, int32_t B, float gamma, float lam,
                       float *d_returns, float *d_advantages, int32_t normalize, double *d_adv_stats,
                       int32_t device, void *stream);
int ppo_normalize_advantages(float *d_advantages, int64_t n, const double *d_adv_stats, int32_t device,
                             void *stream);

/* ---- PPO update: fused attention over the 5-token window (agents/ppo.py:126 -> the self-attention of
 * nn.TransformerEncoderLayer, networks/transformer_net.py:34-43,63), forward and backward in fp32 ---------------------
 * d_q: [n, num_queries, 128] rows of stride q_stride floats; d_k, d_v: [n, 5, 128] rows of stride kv_stride (views into a
 * packed in_proj output are fine); d_pad [n,5]: 1 = the key is a padding row.  num_queries = 5 (every token attends) or 1
 * (only the newest token, the last encoder layer).  d_out / d_grad_out: dense [n, num_queries, 128].  The gradients are
 * written with the strides of their inputs (d_grad_k / d_grad_v: every row; d_grad_q: every query row). */
int ppo_attn5_forward(const float *d_q, int64_t q_stride, const float *d_k, const float *d_v, int64_t kv_stride,
                      const uint8_t *d_pad, int64_t n, int32_t num_queries, float *d_out, int32_t device, void *stream);
int ppo_attn5_backward(const float *d_q, int64_t q_stride, const float *d_k, const float *d_v, int64_t kv_stride,
                       const uint8_t *d_pad, int64_t n, int32_t num_queries, const float *d_grad_out, float *d_grad_q,
                       float *d_grad_k, float *d_grad_v, int32_t device, void *stream);

/* ---- PPO update: the post-backward chain of one minibatch step on FLAT fp32 buffers -------------------------------
 * Replaces torch.nn.utils.clip_grad_norm_(policy.parameters(), GRAD_NORM_CLIP) + optimizer.step() of
 * agents/ppo.py:160-162 (Adam with the four parameter groups of agents/ppo.py:17-22) - and the division by the
 * world size that follows the NCCL gradient sum - with two launches:
 *   g = d_grad * grad_scale;  g *= min(1, max_norm / (||g||_2 + 1e-6));  Adam(beta1, beta2, eps, lr of the segment).
 * d_params / d_grad / d_exp_avg / d_exp_avg_sq: [n] fp32, same element order (d_grad is left holding the clipped g).
 * seg_end / seg_lr (HOST arrays, num_segments <= PPO_OPTIM_MAX_GROUPS): exclusive end offsets (ascending, last == n)
 * and learning rates of the contiguous parameter ranges.  d_step: device int64 Adam step counter (incremented by the
 * call, so CUDA-graph replays advance it).  d_partials: device double[ppo_optim_partials()] scratch.  d_norm_out
 * (optional): the pre-clip gradient norm.  The norm is reduced in a fixed order: bit-identical on every rank.
 * max_norm <= 0 disables clipping. */
#define PPO_OPTIM_MAX_GROUPS 8
int ppo_clip_adam_step(float *d_params, float *d_grad, float *d_exp_avg, float *d_exp_avg_sq, int64_t n,
                       const int64_t *seg_end, const float *seg_lr, int32_t num_segments, float grad_scale,
                       float max_norm, float beta1, float beta2, float eps, int64_t *d_step, double *d_partials,
                       float *d_norm_out, int32_t device, void *stream);
int ppo_optim_partials(void);

#ifdef __cplusplus
}
#endif
#endif /* UAVENV_B200_H */
