// uavenv_kernels.cuh - the kernels of the batched UAV->target allocation environment (sm_100a).
//
//   step_kernel          one fused launch per env.step for all B envs (envs/uav_env.py:295-435):
//                        action/accept rule -> target products, cover flags, UAV assignment ->
//                        reward / done / info -> auto-reset of finished envs (counter RNG scene
//                        generation, uav_env.py:65-182) -> pair score + observation row of the new
//                        pointer pair (mechanics.py:167-241) -> [B,5,14] window.
//   reset_kernel         UAVEnv.reset for a masked subset (uav_env.py:42-63), one warp per env.
//   pack_scene_kernel    scene injection (device SoA -> records, each scene into `copies` consecutive envs) +
//                        per-scene derived values.
//   score_matrix_kernel  p_final / p_damage [B,N,M] (main.py:38-45 over mechanics.py:167-181).
//   recompute_kernel     fresh J / N0 / sums from the per-target products, a warp per env with
//                        shuffle reductions (uav_env.py:244-293) - drift bound for the running sums.
//   best_target_kernel   the best-target heuristic's actions (evaluation baseline): a warp per 32 envs,
//                        one cooperative row of pair scores when a UAV's row is entered.
//   group_best_kernel    the best finished member of each group of consecutive envs (best-of-K allocation):
//                        a warp per group, shuffle arg-max over J, coalesced copy of the winner's allocation.
//   improve_kernel       steepest-ascent local search (UAV moves and swaps) on given allocations: persistent CTAs,
//                        a scene per CTA, block arg-max over the candidates of a round.
//   bound_kernel         certified upper bound on each scene's best J (Frank-Wolfe on the concave relaxation):
//                        improve_kernel's launch shape, a warp-per-UAV arg-max and fixed-order reductions per iteration.
#pragma once

#include "uavenv_b200.h"
#include "uavenv_device.cuh"

namespace uavk {

#ifndef UAV_STEP_THREADS
#define UAV_STEP_THREADS 128
#endif
constexpr int kStepThreads = UAV_STEP_THREADS;   // envs per CTA in step_kernel (thread-per-env main phases)
constexpr int kWarpsPerCta = kStepThreads / 32;
constexpr int kResetThreads = 128;
constexpr int kServiceScratchPerWarp = 32 * kObsFloats * 4;   // a service warp's obstacle scratch = its idle window tile (8960 B)

struct StepIO {
    const void *actions;     // [B] int64 (action_bytes = 8) or int8 (action_bytes = 1)
    int32_t action_bytes;
    int32_t actions_bulk;    // 1: the actions sit in mapped host memory - one bulk copy per CTA brings its slice (16 B aligned)
    float *obs;              // [B,5,14]
    float *reward;           // [B]
    uint8_t *done;           // [B]
    float *J_val;            // info (nullable each)
    int32_t *num_assigned;
    int8_t *is_valid;
    float *avg_p_dmg, *avg_p_final;
    double *reward_f64;
};

// ------------------------------------------------------------------------------------------------
// warp-cooperative helpers (all 32 lanes of the warp must call).  A finished env is restarted by the
// warp that owns it, so the step kernel needs no CTA-wide barrier on its hot path.

constexpr unsigned kFullMask = 0xffffffffu;

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

// Shuffle arg-max of (best, bi) over the warp, every lane ending with the winner (best_target, group_best): the larger
// value wins, on equal values the lower index; index INT_MAX means "no candidate" and never beats a real one.  Branching
// on the index first keeps each step's compare chain as short as the unguarded rule's (best_target's row is latency-bound).
__device__ __forceinline__ void warp_argmax(double &best, int &bi) {
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(kFullMask, best, o);
        const int oi = __shfl_xor_sync(kFullMask, bi, o);
        if (oi < bi ? (ob >= best || bi == INT_MAX) : (ob > best && oi != INT_MAX)) { best = ob; bi = oi; }
    }
}

__device__ __forceinline__ double quiet_nan() { return __longlong_as_double(0x7ff8000000000000ll); }

// position of element i in a sort of keys[0..n) by (key, index): a uniformly random permutation
__device__ __forceinline__ int rank_of(const uint32_t *keys, int n, int i) {
    const uint32_t ki = keys[i];
    int r = 0;
    for (int j = 0; j < n; ++j) {
        const uint32_t kj = keys[j];
        r += (kj < ki) || (kj == ki && j < i);
    }
    return r;
}

// _reset_state_only (envs/uav_env.py:175-182) for env b (scene in `slot`): every UAV available again, every
// lock list empty
__device__ __forceinline__ void warp_clear_allocation(const Params &P, int slot, int b, int lane) {
    int32_t *asg = P.assigned + (size_t)b * P.N;
    for (int i = lane; i < P.N; i += 32) asg[i] = -1;
    TgtRec *T = P.tgt + P.toff(slot, b);
    for (int j = lane; j < P.M; j += 32) clear_locks(T, j);
}

// ---- _generate_scene (envs/uav_env.py:65-173) with the counter RNG, in independent chunks of 32 entities ----
// A scene is a pure function of (seed, global env id, scene index); it is produced chunk by chunk so that the
// pre-generation service can spread one scene over several launches.  Chunk order: target chunks first
// (chunk 0 also draws the obstacles), then UAV chunks (their p_pen needs the obstacles, already visible).

__device__ __forceinline__ int scene_chunks(const Params &P) { return (P.M + 31) / 32 + (P.N + 31) / 32; }

// number of value-6 targets, n2 = randint(1, n_remain+1)   (uav_env.py:121-126)
__device__ __forceinline__ int scene_n2(const Params &P, uint32_t env, uint32_t scene) {
    const int n_remain = P.M - P.M / 2 - 1;
    if (n_remain < 1) return 0;
    return 1 + (int)(((uint64_t)philox4x32(P.seed_lo, P.seed_hi, 0u, S_N2, scene, env).x * (uint64_t)n_remain) >> 32);
}

// total_swarm_cost (uav_env.py:118) and sum of target values (:198) of a generated scene, in closed form
// (type / value class counts are fixed by construction; all terms are exact in fp64)
__device__ __forceinline__ void scene_totals(const Params &P, int b, uint32_t scene, double &total_val, double &total_cost) {
    const int n1 = P.M / 2, n_remain = P.M - n1 - 1, n2 = scene_n2(P, P.env_id_base + (uint32_t)b, scene);
    total_val = 4.0 * n1 + 6.0 * n2 + 8.0 * (n_remain > 0 ? n_remain - n2 : 0) + 16.0;
    total_cost = 1.0 * (P.N - P.N / 4) + 1.25 * (P.N / 4);
}

// obstacles of a scene (uav_env.py:146-170) into Z[K1], I[K2] (global records, or a warp's shared-memory scratch)
__device__ __forceinline__ void warp_generate_obstacles(const Params &P, int b, uint32_t scene, NfzRec *Z, IntRec *I) {
    const int lane = threadIdx.x & 31;
    const uint32_t k0 = P.seed_lo, k1 = P.seed_hi, env = P.env_id_base + (uint32_t)b;
    for (int i = lane; i < P.K1; i += 32) {
        const uint4 a = philox4x32(k0, k1, i, S_NFZ_A, scene, env);
        const uint4 c = philox4x32(k0, k1, i, S_NFZ_B, scene, env);
        Z[i].radius = 5.0 + (10.0 - 5.0) * u53(a.x, a.y);
        Z[i].x = 120.0 + (140.0 - 120.0) * u53(a.z, a.w);
        Z[i].y = 0.0 + (P.map_h - 0.0) * u53(c.x, c.y);
    }
    for (int i = lane; i < P.K2; i += 32) {
        const uint4 a = philox4x32(k0, k1, i, S_INT_A, scene, env);
        const uint4 c = philox4x32(k0, k1, i, S_INT_B, scene, env);
        I[i].x = 140.0 + (160.0 - 140.0) * u53(a.x, a.y);
        I[i].y = 0.0 + (P.map_h - 0.0) * u53(a.z, a.w);
        const double sp = 0.30 + (0.32 - 0.30) * u53(c.x, c.y);
        const double ang = 0.0 + (2.0 * 3.141592653589793 - 0.0) * u53(c.z, c.w);
        I[i].vx = cos(ang) * sp;
        I[i].vy = sin(ang) * sp;
    }
}

// entities [32*c, 32*c+32) of chunk c: target chunks first, then UAV chunks; Z / I: the scene's obstacles, already
// visible to this warp (the UAV chunks need them for p_pen).  A UAV chunk can be produced in two stages (the pre-generation
// service runs them in different launches: p_pen - two acos, four exp - is as long as everything else of the chunk):
// stage 0 = the whole record, 1 = everything but p_pen, 2 = p_pen of the records stage 1 has written
__device__ void warp_generate_chunk(const Params &P, int slot, int b, uint32_t scene, int chunk, uint32_t *s_keys,
                                    const NfzRec *Z, const IntRec *I, int stage = 0) {
    const int lane = threadIdx.x & 31;
    const uint32_t k0 = P.seed_lo, k1 = P.seed_hi, env = P.env_id_base + (uint32_t)b;
    const int N = P.N, M = P.M, tchunks = (M + 31) / 32;
    __syncwarp();
    if (chunk < tchunks) {
        // targets [32*chunk, 32*chunk+32): value by rank among the value keys (uav_env.py:121-129), list position
        // by rank among the list keys (the shuffle of :173: target id i lands at list position rank_i)
        const int i = chunk * 32 + lane;
        const int n1 = M / 2, n_remain = M - n1 - 1, n2 = scene_n2(P, env, scene);
        for (int j = lane; j < M; j += 32) s_keys[j] = philox4x32(k0, k1, j, S_TGT_VAL, scene, env).x;
        __syncwarp();
        double value = 0.0;
        if (i < M) {
            const int q = rank_of(s_keys, M, i);
            value = q < n1 ? 4.0 : (q < n1 + n2 ? 6.0 : (q < n1 + n_remain ? 8.0 : 16.0));
        }
        __syncwarp();
        for (int j = lane; j < M; j += 32) s_keys[j] = philox4x32(k0, k1, j, S_TGT_LIST, scene, env).x;
        __syncwarp();
        if (i < M) {
            const int pos = rank_of(s_keys, M, i);
            const uint4 a = philox4x32(k0, k1, i, S_TGT_POS, scene, env);
            const uint4 v = philox4x32(k0, k1, i, S_TGT_VEL, scene, env);
            TgtRec t;
            t.x = P.tgt_x_lo + (P.tgt_x_hi - P.tgt_x_lo) * u53(a.x, a.y);            // :134
            t.y = 0.0 + (P.map_h - 0.0) * u53(a.z, a.w);                              // :135
            const double vx = (u53(v.x, v.y) - 0.5) * 0.03, vy = (u53(v.z, v.w) - 0.5) * 0.03;  // :139
            t.speed = sqrt(vx * vx + vy * vy);
            t.value = value;
            clear_locks(&t, 0); t.id = i;
            P.tgt[P.toff(slot, b) + pos] = t;
            P.tgt_vel[P.toff(slot, b) + pos] = make_double2(vx, vy);
        }
    } else {
        // UAVs [32*c, 32*c+32): N//4 of type 2, uniformly permuted (uav_env.py:81-84); kinematics (:88-111)
        const int i = (chunk - tchunks) * 32 + lane;
        if (stage == 2) {
            if (i < N) {
                UavRec *up = P.uav + P.uoff(slot, b) + i;
                const UavRec u = *up;
                up->p_pen = penetration_prob(P, Z, I, u);
            }
            __syncwarp();
            return;
        }
        for (int j = lane; j < N; j += 32) s_keys[j] = philox4x32(k0, k1, j, S_UAV_TYPE, scene, env).x;
        __syncwarp();
        if (i < N) {
            const int type = rank_of(s_keys, N, i) >= N - N / 4 ? 2 : 1;
            const uint4 a = philox4x32(k0, k1, i, S_UAV_POS, scene, env);
            const uint4 d = philox4x32(k0, k1, i, S_UAV_DYN, scene, env);
            UavRec u;
            u.x = P.uav_x_lo + (P.uav_x_hi - P.uav_x_lo) * u53(a.x, a.y);            // :88
            u.y = 0.0 + (P.map_h - 0.0) * u53(a.z, a.w);                              // :89
            double base_speed, base_load;
            if (type == 1) { base_speed = 0.35 + (0.50 - 0.35) * u53(d.x, d.y); u.cost = 1.0; base_load = 0.95; }
            else { base_speed = 0.75 + (0.90 - 0.75) * u53(d.x, d.y); u.cost = 1.25; base_load = 1.0; }  // :93-102
            const double real_speed = base_speed * P.weather_speed;                   // :106
            u.load = base_load * P.weather_load;                                      // :107
            const double ang = (-15.0 + (15.0 - (-15.0)) * u53(d.z, d.w)) * (3.141592653589793 / 180.0);  // :110
            const double vx = cos(ang) * real_speed, vy = sin(ang) * real_speed;      // :111
            if (stage == 0) finish_uav(P, Z, I, u, vx, vy);
            else { finish_uav_kinematics(u, vx, vy); u.p_pen = 1.0; }
            P.uav[P.uoff(slot, b) + i] = u;
            P.uav_vel[P.uoff(slot, b) + i] = make_double2(vx, vy);
            P.uav_type[P.uoff(slot, b) + i] = type;
        }
    }
    __syncwarp();
}

// whole scene in one go (reset(), and the fallback when the next scene was not pre-generated in time)
__device__ __noinline__ void warp_generate_scene(const Params &P, int slot, int b, uint32_t scene, uint32_t *s_keys) {
    const int nchunks = scene_chunks(P);
    NfzRec *Z = P.nfz + P.zoff(slot, b);
    IntRec *I = P.intc + P.ioff(slot, b);
    warp_generate_obstacles(P, b, scene, Z, I);
    __threadfence_block();  // obstacles visible to the UAV chunks of this warp
    __syncwarp();
    for (int c = 0; c < nchunks; ++c) warp_generate_chunk(P, slot, b, scene, c, s_keys, Z, I);
    warp_clear_allocation(P, slot, b, threadIdx.x & 31);
    __syncwarp();
}

// ---- pre-generation service: the first CTAs of the step grid (blockIdx < service CTAs) -----------------------------
// Every env always has its NEXT scene (index I_GEN >> 1) prepared in the slot it is not playing on, so that the
// scheduled regeneration of main_train.py:79 is a slot flip for its owner: three header stores, NO fence and NO extra
// load on the step's critical path.  That works because the service never acts on a request in the launch in which it
// first sees it, and never publishes in a launch in which it still writes records - kernel boundaries do the ordering:
//   a period = kServicePeriod launches, counted by every service CTA on its own (all counters are equal)
//   launch 0            SCAN     each CTA reads I_GEN / I_NEXT_TAG of its 1024 envs; an env whose other slot does not hold
//                                scene I_GEN >> 1 yet is appended to the period's queue (its I_GEN word is captured)
//   launches 1..P-2     PROCESS  job j = (queue entry, chunk of 32 entities) -> warp j of the round; jobs are independent, so a
//                                whole batch of scenes costs ONE job latency per stage, hidden behind the step's main CTAs;
//                                jobs whose env has moved on since the scan (I_GEN changed, or the scene was delivered by
//                                reset()) are dropped.  A UAV chunk is two jobs in different launches - the record without
//                                p_pen, then p_pen (from the obstacle records the scene's first job wrote): as one job it
//                                outlasted the main CTAs by ~9 us (every 16th step read 27-29 us instead of 18.5)
//   launch P-1          PUBLISH  entries with all chunks in: I_NEXT_TAG = scene index (I_GEN still unchanged)
// Single writer per word: owner -> I_GEN; service -> I_NEXT_TAG, the queues and the other slot's records.  An owner that
// sees the tag flips; its record reads are ordered after the service's writes by >= 1 kernel boundary.  Whatever is not
// ready when an env needs it (RESET_EPISODES of a few steps) is generated in place by the owner's warp - same result.
constexpr int kServicePeriod = 16;
constexpr int kServiceEnvsPerCta = kStepThreads * 8;  // every thread scans 8 envs

__device__ __noinline__ void pregen_service(const Params &P, int service_cta, int n_service, uint32_t *s_keys,
                                            unsigned char *s_scratch) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ uint32_t s_tick;
    __shared__ int s_n, s_base;
    if (tid == 0) {
        const uint32_t t = P.svc_ctr[service_cta];
        P.svc_ctr[service_cta] = t + 1u;
        s_tick = t;
        s_n = 0;
    }
    __syncthreads();
    const uint32_t phase = s_tick % (uint32_t)kServicePeriod;
    const int q = (int)((s_tick / (uint32_t)kServicePeriod) & 1u);
    int32_t *const q_env = P.q_env + (size_t)q * P.B, *const q_gen = P.q_gen + (size_t)q * P.B;
    int32_t *const q_done = P.q_done + (size_t)q * P.B;
    // jobs of a queue entry: its target chunks, its UAV chunks without p_pen (space A), then p_pen of its UAV chunks (space B,
    // in launches AFTER the last launch of space A: stage 2 reads what stage 1 wrote)
    const int tchunks = (P.M + 31) / 32, uchunks = (P.N + 31) / 32, chunks_a = tchunks + uchunks, nchunks = chunks_a + uchunks;
    if (phase == 0u) {
        // ---- SCAN: 8 consecutive envs per thread = one 32 B run of the I_GEN row and of the I_NEXT_TAG row of a tile
        if (service_cta == 0 && tid == 0) P.q_count[q ^ 1] = 0u;   // the other queue is idle during this whole period
        int *const s_list = reinterpret_cast<int *>(s_scratch);
        const int e0 = service_cta * kServiceEnvsPerCta + tid * 8;
        if (e0 < P.B) {
            const Hdr h = P.header(e0);
            const int4 g0 = *reinterpret_cast<const int4 *>(&h.n(I_GEN)), g1 = *reinterpret_cast<const int4 *>(&h.n(I_GEN) + 4);
            const int4 t0 = *reinterpret_cast<const int4 *>(&h.n(I_NEXT_TAG)), t1 = *reinterpret_cast<const int4 *>(&h.n(I_NEXT_TAG) + 4);
            const int gen[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
            const int tag[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (e0 + i < P.B && tag[i] != (gen[i] >> 1)) {
                    const int at = atomicAdd(&s_n, 1);
                    s_list[2 * at] = e0 + i;
                    s_list[2 * at + 1] = gen[i];
                }
        }
        __syncthreads();
        const int n = s_n;
        if (n == 0) return;
        if (tid == 0) s_base = (int)atomicAdd(&P.q_count[q], (uint32_t)n);
        __syncthreads();
        for (int i = tid; i < n; i += blockDim.x) {
            q_env[s_base + i] = s_list[2 * i];
            q_gen[s_base + i] = s_list[2 * i + 1];
            q_done[s_base + i] = 0;
        }
        return;
    }
    const int count = (int)P.q_count[q];
    if (count == 0) return;
    if (phase == (uint32_t)kServicePeriod - 1u) {
        // ---- PUBLISH
        for (int i = service_cta * blockDim.x + tid; i < count; i += n_service * blockDim.x) {
            const int eb = q_env[i], gen = q_gen[i];
            const Hdr h = P.header(eb);
            if (q_done[i] == nchunks && h.n(I_GEN) == gen) h.n(I_NEXT_TAG) = gen >> 1;
        }
        return;
    }
    // ---- PROCESS, round phase-1: one job per warp
    const long long cap = (long long)n_service * kWarpsPerCta, jobs_a = (long long)count * chunks_a, jobs_b = (long long)count * uchunks;
    const long long rounds_a = (jobs_a + cap - 1) / cap, widx = (long long)service_cta * kWarpsPerCta + warp;
    long long round = (long long)phase - 1;
    int entry, chunk, stage;
    if (round < rounds_a) {
        const long long job = round * cap + widx;
        if (job >= jobs_a) return;
        entry = (int)(job / chunks_a); chunk = (int)(job % chunks_a); stage = 1;
    } else {
        const long long job = (round - rounds_a) * cap + widx;
        if (job >= jobs_b) return;
        entry = (int)(job / uchunks); chunk = tchunks + (int)(job % uchunks); stage = 2;
    }
    const int eb = q_env[entry], gen = q_gen[entry];
    const Hdr h = P.header(eb);
    if (*(volatile int32_t *)&h.n(I_GEN) != gen || *(volatile int32_t *)&h.n(I_NEXT_TAG) == (gen >> 1)) return;  // stale
    const int scene = gen >> 1, slot = (gen & 1) ^ 1;
    // the obstacles: chunk 0 generates them (in its shared-memory scratch) and writes the records; the p_pen jobs run in a
    // later launch and read those records - nobody else needs them
    NfzRec *Zg = P.nfz + P.zoff(slot, eb);
    IntRec *Ig = P.intc + P.ioff(slot, eb);
    const NfzRec *Z = Zg;
    const IntRec *I = Ig;
    if (chunk == 0) {
        NfzRec *Zs = reinterpret_cast<NfzRec *>(s_scratch + (size_t)warp * kServiceScratchPerWarp);
        IntRec *Is = reinterpret_cast<IntRec *>(Zs + P.K1);
        warp_generate_obstacles(P, eb, (uint32_t)scene, Zs, Is);
        __syncwarp();
        for (int i = lane; i < P.K1; i += 32) Zg[i] = Zs[i];
        for (int i = lane; i < P.K2; i += 32) Ig[i] = Is[i];
    }
    warp_generate_chunk(P, slot, eb, (uint32_t)scene, chunk, s_keys, Z, I, stage);
    if (lane == 0) atomicAdd(&q_done[entry], 1);
}

// ------------------------------------------------------------------------------------------------
// thread-level pieces

// calc_advantage of the pointer pair + its observation row (uav_env.py:184-242 -> mechanics.py:185-241)
// from the two gathered records and the running aggregates.
__device__ __forceinline__ void eval_pointer_pair(const Params &P, const UavRec &u, const TgtRec &t, double cost_sum,
                                                  double covered_val, double total_cost, double total_val,
                                                  double &pf, double &pd, float *row) {
    pf = pair_score(P, u, t.x, t.y, t.speed, &pd);
    const double inv_tc = 1.0 / (total_cost + 1e-6);
    const double chi_c = cost_sum * inv_tc;                             // uav_env.py:195-196
    const double chi_v = covered_val / (total_val + 1e-6);              // :198-200
    const double chi_mc = t.lock_cost * inv_tc;                         // :202-206
    const double P_prev = 1.0 - t.nh, P_pure = 1.0 - t.nh_pure;         // :226-227
    state_vector(u.cost, t.value, chi_c, chi_v, chi_mc, pf, pd, P_prev, P_prev * t.value, P_pure, row);
}

// the decision pointers, counters and running sums of an env; age = valid rows of its observation window
__device__ __forceinline__ void store_progress(const Hdr &h, int k, int m, int nA, int n0, int age, double rev, double cost_sum,
                                               double covered_val, double sum_pd, double sum_pf) {
    h.n(I_K) = k; h.n(I_M) = m; h.n(I_NASSIGNED) = nA; h.n(I_NCOVERED) = n0; h.n(I_AGE) = age;
    h.f(F_REV) = rev; h.f(F_COST_SUM) = cost_sum; h.f(F_COVERED_VAL) = covered_val;
    h.f(F_SUM_PD) = sum_pd; h.f(F_SUM_PF) = sum_pf;
}

// capture the new current pair in the header (the next step's accept rule reads only these)
// (t: the record as seen in the current episode, lock_cnt = target_view(t, episode))
__device__ __forceinline__ void store_current_pair(const Hdr &h, const UavRec &u, const TgtRec &t, int lock_cnt, double pf, double pd) {
    h.f(F_CUR_PF) = pf; h.f(F_CUR_PD) = pd; h.f(F_CUR_VALUE) = t.value; h.f(F_CUR_NH) = t.nh; h.f(F_CUR_NHP) = t.nh_pure;
    h.f(F_CUR_LOCK_COST) = t.lock_cost; h.f(F_CUR_UCOST) = u.cost; h.n(I_CUR_LOCK_CNT) = lock_cnt; h.n(I_CUR_TID) = t.id;
}

// ---- async copy / TMA helpers (sm_100a) --------------------------------------------------------------
__device__ __forceinline__ void cp_async_8(void *smem_dst, const void *gmem_src) {   // LDGSTS, 8 bytes
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
// TMA bulk store shared::cta -> global (UBLKCP): bytes % 16 == 0, both addresses 16 B aligned
__device__ __forceinline__ void bulk_store(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gmem_dst),
                 "r"((uint32_t)__cvta_generic_to_shared(smem_src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
// wait until the bulk stores of this thread have READ their shared-memory source (the CTA may then exit)
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// The fused step.  Thread t of a CTA owns env b = blockIdx.x*128 + t for the O(1) state machine.
// Memory-level parallelism is what bounds this kernel (every env touches ~1 KB scattered over a few
// hundred MB), so the dependent chain is kept to TWO round trips and there is no CTA-wide barrier:
//   trip 1  scalar state (SoA, coalesced) + action + ring head; the four older window rows start
//           streaming into the warp's shared-memory tile with cp.async (LDGSTS) as soon as the head is known
//   trip 2  the two 64 B records of the NEW pointer pair - the accept rule itself needs no gather because the
//           current pair's values were captured in the header when its observation row was computed
// The [5,14] windows of a warp (32 x 280 B, contiguous in obs) leave through one TMA bulk store.
// A finished env restarts inside the launch.  The common case (same scene, uav_env.py:175-182) stays on the
// two-trip chain: its owner simply evaluates pointer pair (0,0) with the target's products taken as cleared,
// and the warp clears the allocation arrays afterwards with fire-and-forget stores (warp_soft_reset).
// The scheduled regeneration (every RESET_EPISODES-th episode, main_train.py:79) is a slot flip: the env's
// next scene was prepared in the other storage slot by the pre-generation service (the CTAs past the main
// grid, pregen_service above) - so it, too, stays on the two-trip chain.  Only when that scene is not ready
// (first episodes after a reset with a very short schedule) does the owner's warp generate it in place, in a
// second pass of the evaluation loop (out of line, so nothing but a few scalars is live across the call).

// Eq.21 near-tie (uav_env.py:317): r(X) and r(X') re-summed exactly as _calc_J_X does (uav_env.py:244-269): targets in
// list order, one running fp64 sum; X' differs from X in target m's product (nh2) only.  One thread, rare, out of line.
__device__ __noinline__ void exact_rewards(const Params &P, int slot, int b, int episode, int m, double nh2, double cost_sum,
                                           double cost2, int n0, int n02, double &prev_r, double &new_r) {
    const TgtRec *T = P.tgt + P.toff(slot, b);
    double rev = 0.0, rev2 = 0.0;
    for (int j = 0; j < P.M; ++j) {
        const double nh = tag_current(T[j].lock_tag, episode) ? T[j].nh : 1.0, value = T[j].value;
        rev += (1.0 - nh) * value;                                    // :264-265
        rev2 += (1.0 - (j == m ? nh2 : nh)) * value;
    }
    prev_r = paper_reward(objective(P, rev, cost_sum), n0, P.M);      // :268, :287-291
    new_r = paper_reward(objective(P, rev2, cost2), n02, P.M);
}

// restart bookkeeping of the finished envs in mask (their scene is in slot_of[lane]): stores only
__device__ __noinline__ void warp_soft_reset(const Params &P, unsigned soft_mask, int b0, int my_slot) {
    const int lane = threadIdx.x & 31;
    __syncwarp();  // orders the owners' accept stores before the clears
    while (soft_mask) {
        const int src = __ffs(soft_mask) - 1;
        soft_mask &= soft_mask - 1;
        const int slot = __shfl_sync(kFullMask, my_slot, src);
        warp_clear_allocation(P, slot, b0 + src, lane);
    }
    __syncwarp();
}

// fallback regeneration in place (the next scene was not pre-generated in time) of the envs in mask
__device__ __noinline__ void warp_regen_inline(const Params &P, unsigned mask, int b0, int my_slot, int my_scene,
                                               uint32_t *s_keys) {
    while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const int slot = __shfl_sync(kFullMask, my_slot, src), scene = __shfl_sync(kFullMask, my_scene, src);
        __syncwarp();
        warp_generate_scene(P, slot, b0 + src, (uint32_t)scene, s_keys);
    }
    __threadfence_block();
}

__global__ void __launch_bounds__(kStepThreads, 512 / kStepThreads) step_kernel(const __grid_constant__ Params P, const StepIO io,
                                                               const int n_service) {
    extern __shared__ __align__(16) unsigned char s_dyn[];
    __shared__ __align__(128) float s_tile[kWarpsPerCta][32 * kObsFloats];
    __shared__ __align__(16) unsigned char s_act[kStepThreads * 8];   // the CTA's actions when they come over PCIe (bulk copy)
    __shared__ uint64_t s_act_bar;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *const s_keys = reinterpret_cast<uint32_t *>(s_dyn) + (size_t)warp * max(P.N, P.M);  // per-warp scratch
    if ((int)blockIdx.x < n_service) {  // service CTAs: prepare next scenes, off the step's critical path
        pregen_service(P, (int)blockIdx.x, n_service, s_keys, reinterpret_cast<unsigned char *>(&s_tile[0][0]));
        return;
    }
    const int n_main = (int)gridDim.x - n_service;
    const int b0 = ((int)blockIdx.x - n_service) * kStepThreads + warp * 32;   // first env of this warp
    const int b = b0 + lane;
    const bool live = b < P.B;
    const int bc = live ? b : P.B - 1;  // clamped index: idle tail lanes issue harmless loads
    const int N = P.N, M = P.M;
    // actions in mapped host memory: a 32 B read per warp is one PCIe read request per warp (2048 of them at c3, +5.7 us on
    // the chain); one bulk copy per CTA is a quarter of the requests and is in flight before anything else
    const int cta_first = b0 - warp * 32, cta_envs = min(kStepThreads, P.B - cta_first);
    const bool bulk_actions = io.actions_bulk && ((cta_envs * io.action_bytes) & 15) == 0;
    if (bulk_actions && tid == 0) {
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_act_bar), bytes = (uint32_t)(cta_envs * io.action_bytes);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(s_act)),
                     "l"(static_cast<const unsigned char *>(io.actions) + (size_t)cta_first * io.action_bytes), "r"(bytes), "r"(bar)
                     : "memory");
    }
    const Hdr H = P.header(bc);
    float *tile = s_tile[warp] + lane * kObsFloats;

    // ---- trip 1: everything that depends on b only (all loads issued before anything is consumed) ----
    const uint32_t head_old = P.step_ctr[0];
    int k = H.n(I_K), m = H.n(I_M), nA = H.n(I_NASSIGNED), n0 = H.n(I_NCOVERED), age = H.n(I_AGE);
    double rev = H.f(F_REV), cost_sum = H.f(F_COST_SUM), covered_val = H.f(F_COVERED_VAL);
    double sum_pd = H.f(F_SUM_PD), sum_pf = H.f(F_SUM_PF);
    double total_val = H.f(F_TOTAL_VAL), total_cost = H.f(F_TOTAL_COST);
    const double c_pf = H.f(F_CUR_PF), c_pd = H.f(F_CUR_PD), c_value = H.f(F_CUR_VALUE), c_nh = H.f(F_CUR_NH);
    const double c_nhp = H.f(F_CUR_NHP), c_lock_cost = H.f(F_CUR_LOCK_COST), c_ucost = H.f(F_CUR_UCOST);
    const int c_lock_cnt = H.n(I_CUR_LOCK_CNT), c_tid = H.n(I_CUR_TID);
    const int episode_new = H.n(I_EPISODE) + 1;
    const int gen = H.n(I_GEN), next_tag = H.n(I_NEXT_TAG);
    int slot = gen & 1;                                                  // storage slot of the current scene
    const bool was_finished = !P.auto_reset && H.n(I_FINISHED);
    int64_t action = 0;
    if (!bulk_actions)
        action = io.action_bytes == 8 ? static_cast<const int64_t *>(io.actions)[bc]
                                      : (int64_t) static_cast<const int8_t *>(io.actions)[bc];
    const uint32_t head_new = (head_old + 1u) % (uint32_t)kSeqLen;       // ring slot of this step's row
    // older rows of the window: ring tile [slot][feature pair][32 lanes] -> tile rows 0..3 (time order)
    float2 *const ring = P.ring(bc);
#pragma unroll
    for (int a = kSeqLen - 1; a >= 1; --a) {
        const uint32_t slot = (head_new + (uint32_t)(kSeqLen - a)) % (uint32_t)kSeqLen;
        const float2 *src = ring + slot * (kStateDim / 2) * 32;
        float *dst = tile + (kSeqLen - 1 - a) * kStateDim;
#pragma unroll
        for (int f = 0; f < kStateDim / 2; ++f) cp_async_8(dst + 2 * f, src + f * 32);
    }
    if (tid == 0) {
        // arrive; the last CTA to have READ the head publishes the new one (kept on the device so that
        // CUDA-graph replays stay correct).  The increment depends on head_old, so the read is ordered first.
        if (atomicAdd(&P.step_ctr[1], 1u + (head_old >> 31)) == (unsigned)n_main - 1u) {
            P.step_ctr[1] = 0u;
            P.step_ctr[0] = head_new;
        }
    }

    if (bulk_actions) {   // (uniform per CTA) the barrier publishes the mbarrier's initialisation; the loads above are in flight
        __syncthreads();
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_act_bar);
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "ACT_WAIT:\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t"
            "@p bra ACT_DONE;\n\t"
            "bra ACT_WAIT;\n\t"
            "ACT_DONE:\n\t"
            "}\n" ::"r"(bar) : "memory");
        const int ia = live ? tid : 0;
        action = io.action_bytes == 8 ? reinterpret_cast<const int64_t *>(s_act)[ia] : (int64_t) reinterpret_cast<const int8_t *>(s_act)[ia];
    }
    // ---- accept rule -> state update -> reward / done / info (uav_env.py:295-363, :426-433) ----------
    bool done = false, restarted = false;
    if (live) {
        double reward = 0.0;
        if (!was_finished) {
            double prev_r = paper_reward(objective(P, rev, cost_sum), n0, M);           // :301
            double cur_r = prev_r;
            bool advance_uav = false;
            if (action == 1) {                                                           // :306
                const Tentative x = tentative_assign(P, rev, cost_sum, n0, c_nh, c_value, c_lock_cnt, c_pf, c_ucost);
                double new_r = x.new_r;
                // the carried sums differ from the reference's fresh sums by O(1e-14) relative: inside the tie band the
                // decision (and the reward) come from the exact re-summation.  Only with a cost term: at omega = 0 an Assign
                // can only grow one term of J and N0, so new_r >= prev_r holds under rounding in the reference's summation
                // and in the carried one alike (and near-ties are the NORM there once a target's product has underflowed)
                if (P.omega != 0.0 && fabs(new_r - prev_r) <= P.tie_band * fmax(fabs(new_r), fabs(prev_r)))
                    exact_rewards(P, slot, b, episode_new - 1, m, x.nh2, cost_sum, x.cost2, n0, x.n02, prev_r, new_r);
                if (new_r >= prev_r) {                                                   // :317 (Eq.21)
                    reward = new_r - prev_r;                                             // :321
                    cur_r = new_r;
                    TgtRec *tp = P.tgt + P.toff(slot, b) + m;
                    tp->nh = x.nh2; tp->nh_pure = c_nhp * (1.0 - c_pd);
                    tp->lock_cost = c_lock_cost + c_ucost; tp->lock_tag = make_tag(c_lock_cnt + 1, episode_new - 1);
                    tp->id = c_tid;   // (unchanged value: the record's second 32 B sector is then written WHOLE - no fill read)
                    P.assigned[(size_t)b * N + k] = c_tid;                               // :308
                    rev = x.rev2; cost_sum = x.cost2;
                    if (c_lock_cnt == 0) { covered_val += c_value; n0 = x.n02; }
                    sum_pd += c_pd; sum_pf += c_pf; nA += 1;
                    advance_uav = true;                                                  // :324-325
                }
            }
            if (advance_uav) { k += 1; m = 0; }
            else {                                                                       // :336-342, :347-352
                m += 1;
                // a UAV that passes every target stays unassigned: its slot may hold the previous episode's value
                if (m >= M) { P.assigned[(size_t)b * N + k] = -1; k += 1; m = 0; }
            }
            done = k >= N;                                                               // :355
            if (done) reward += cur_r;                                                   // :361-363
            if (io.is_valid) io.is_valid[b] = (action == 1) ? (reward != 0.0 ? 1 : 0) : -1;  // :429
        } else {
            done = true;  // a finished env without auto-reset is inert
            if (io.is_valid) io.is_valid[b] = -1;
        }
        io.reward[b] = (float)reward;
        io.done[b] = done ? 1 : 0;
        if (io.reward_f64) io.reward_f64[b] = reward;
        if (io.J_val) io.J_val[b] = (float)objective(P, rev, cost_sum);                  // :427
        if (io.num_assigned) io.num_assigned[b] = n0;                                    // :428
        if (io.avg_p_dmg) io.avg_p_dmg[b] = nA > 0 ? (float)(sum_pd / nA) : 0.0f;        // :409
        if (io.avg_p_final) io.avg_p_final[b] = nA > 0 ? (float)(sum_pf / nA) : 0.0f;    // :416
        if (done && !was_finished) {
            if (P.auto_reset) restarted = true;
            else H.n(I_FINISHED) = 1;
        }
    }
    const bool inert = live && done && !restarted;  // finished, no auto-reset: zero window, frozen state
    const bool regen = restarted && P.reset_episodes > 0 && (episode_new % P.reset_episodes) == 0;  // main_train.py:79
    bool inline_regen = false;
    if (restarted) {  // pointers and running sums of the next episode (uav_env.py:54-55, :175-182)
        k = 0; m = 0; nA = 0; n0 = 0; age = 0;
        rev = 0.0; cost_sum = 0.0; covered_val = 0.0; sum_pd = 0.0; sum_pf = 0.0;
        H.n(I_EPISODE) = episode_new;
        if (regen) {
            const int scene = gen >> 1;
            scene_totals(P, b, (uint32_t)scene, total_val, total_cost);
            H.f(F_TOTAL_VAL) = total_val; H.f(F_TOTAL_COST) = total_cost;
            // the pre-generated scene: flip the storage slot (its records were written >= 1 launch ago) - or generate in
            // place (second pass).  The service picks the new I_GEN up at its next scan: no fence, no request store.
            if (next_tag == scene) slot ^= 1;
            else inline_regen = true;
            H.n(I_GEN) = ((scene + 1) << 1) | slot;
        }
    }
    const bool soft = restarted && !inline_regen;
    // a restart leaves the allocation arrays alone: target records carry their episode (target_view) and UAV slots at or
    // past the pointer are read as unassigned.  Every 2^16-th episode of an env the arrays are wiped, so that a record's
    // 18-bit episode tag can never alias
    const bool wipe = soft && (episode_new & 0xffff) == 0;
    const int episode_eval = restarted ? episode_new : episode_new - 1;   // the episode the new pointer pair belongs to

    // ---- trip 2 + evaluation.  pass 0: every env but the (rare) inline-regenerated ones; pass 1: those ----
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1) {
            const unsigned soft_mask = __ballot_sync(kFullMask, wipe);
            if (soft_mask) warp_soft_reset(P, soft_mask, b0, slot);
            const unsigned regen_mask = __ballot_sync(kFullMask, inline_regen);
            if (regen_mask == 0u) break;
            warp_regen_inline(P, regen_mask, b0, slot, gen >> 1, s_keys);
        }
        if (live && (pass == 0 ? (!done || soft) : inline_regen)) {
            const UavRec u = P.uav[P.uoff(slot, b) + k];
            TgtRec t = P.tgt[P.toff(slot, b) + m];   // sees this thread's own accept store on target m
            const int t_cnt = target_view(t, episode_eval);   // (a restarted env sees every record as cleared)
            cp_async_wait_all();                        // ring rows have landed in the tile (gathers still in flight)
            const int nprev = age < kSeqLen - 1 ? age : kSeqLen - 1;
#pragma unroll
            for (int a = kSeqLen - 1; a >= 1; --a) {     // rows older than the episode are zero (uav_env.py:58-61)
                if (a > nprev) {
                    float *dst = tile + (kSeqLen - 1 - a) * kStateDim;
#pragma unroll
                    for (int f = 0; f < kStateDim; f += 2) *reinterpret_cast<float2 *>(dst + f) = make_float2(0.f, 0.f);
                }
            }
            double pf, pd;
            float row[kStateDim];
            eval_pointer_pair(P, u, t, cost_sum, covered_val, total_cost, total_val, pf, pd, row);
            store_current_pair(H, u, t, t_cnt, pf, pd);
            float2 *dsth = ring + head_new * (kStateDim / 2) * 32;
#pragma unroll
            for (int f = 0; f < kStateDim / 2; ++f) {
                const float2 v = make_float2(row[2 * f], row[2 * f + 1]);
                dsth[f * 32] = v;
                *reinterpret_cast<float2 *>(tile + (kSeqLen - 1) * kStateDim + 2 * f) = v;
            }
            store_progress(H, k, m, nA, n0, nprev + 1, rev, cost_sum, covered_val, sum_pd, sum_pf);
        }
    }
    cp_async_wait_all();
    if (inert) {
#pragma unroll
        for (int f = 0; f < kObsFloats; f += 2) *reinterpret_cast<float2 *>(tile + f) = make_float2(0.f, 0.f);
        if (!was_finished)  // the step that finished the episode: freeze the final pointers
            store_progress(H, k, m, nA, n0, 0, rev, cost_sum, covered_val, sum_pd, sum_pf);
    }
    // ---- window out: one TMA bulk store per warp (32 x 280 B contiguous in obs) ------------------------
    fence_proxy_async_smem();
    __syncwarp();
    {
        const int nenv = min(32, P.B - b0);
        if (nenv > 0) {
            float *dst = io.obs + (size_t)b0 * kObsFloats;
            const float *src = s_tile[warp];
            const uint32_t bytes = (uint32_t)nenv * kObsFloats * sizeof(float);
            if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0 && (bytes & 15u) == 0) {
                if (lane == 0) { bulk_store(dst, src, bytes); bulk_store_wait_read(); }
            } else {  // ragged tail / unaligned caller buffer
                for (int i = lane; i < nenv * kObsFloats; i += 32) dst[i] = src[i];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// UAVEnv.reset (envs/uav_env.py:42-63) for the masked envs: one warp per env.
// mode: 0 = state only, 1 = generate a new scene, 2 = scene already packed (load_scene)

__global__ void __launch_bounds__(kResetThreads) reset_kernel(const __grid_constant__ Params P, int mode,
                                                               const uint8_t *mask, int first_env, int count,
                                                               float *obs) {
    extern __shared__ __align__(16) unsigned char s_dyn[];
    __shared__ float s_row[kResetThreads / 32][kStateDim];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    uint32_t *s_keys = reinterpret_cast<uint32_t *>(s_dyn) + (size_t)warp * max(P.N, P.M);
    for (int e = blockIdx.x * wpb + warp; e < count; e += gridDim.x * wpb) {
        const int b = first_env + e;
        if (mask && !mask[b]) continue;  // uniform across the warp
        const Hdr H = P.header(b);
        const int gen = H.n(I_GEN), slot = gen & 1;
        __syncwarp();
        const bool ahead = P.auto_reset && P.reset_episodes > 0;  // keep the NEXT scene prepared in the other slot
        if (mode == 1) {
            // a new scene now, in place (index gen >> 1) ...
            const int scene = gen >> 1;
            warp_generate_scene(P, slot, b, (uint32_t)scene, s_keys);
            // ... and the one after it into the other slot, so that the first scheduled regeneration is a flip
            // (a reset is off the hot path; the step-time service only has to keep up with later flips)
            if (ahead) warp_generate_scene(P, slot ^ 1, b, (uint32_t)(scene + 1), s_keys);
            if (lane == 0) {
                double tv, tc;
                scene_totals(P, b, (uint32_t)scene, tv, tc);
                H.f(F_TOTAL_VAL) = tv; H.f(F_TOTAL_COST) = tc;
                H.n(I_GEN) = ((scene + 1) << 1) | slot;
                if (ahead) H.n(I_NEXT_TAG) = scene + 1;
            }
        } else if (mode == 2) {
            // injected scene (already packed into the current slot); prepare the generated scene that follows it
            if (ahead) {
                warp_generate_scene(P, slot ^ 1, b, (uint32_t)(gen >> 1), s_keys);
                if (lane == 0) H.n(I_NEXT_TAG) = gen >> 1;
            }
            warp_clear_allocation(P, slot, b, lane);
        } else {
            warp_clear_allocation(P, slot, b, lane);
        }
        __syncwarp();
        if (lane == 0) {
            const double total_cost = H.f(F_TOTAL_COST), total_val = H.f(F_TOTAL_VAL);
            double pf, pd;
            float row[kStateDim];
            const UavRec u = P.uav[P.uoff(slot, b)];
            const TgtRec t = P.tgt[P.toff(slot, b)];       // (just cleared)
            eval_pointer_pair(P, u, t, 0.0, 0.0, total_cost, total_val, pf, pd, row);
            store_current_pair(H, u, t, 0, pf, pd);
            store_progress(H, 0, 0, 0, 0, 1, 0.0, 0.0, 0.0, 0.0, 0.0);
            H.n(I_FINISHED) = 0;
            H.n(I_EPISODE) = (mode == 0) ? H.n(I_EPISODE) + 1 : 1;
            const uint32_t head = P.step_ctr[0] % (uint32_t)kSeqLen;
            float2 *dsth = P.ring(b) + head * (kStateDim / 2) * 32;
            for (int f = 0; f < kStateDim / 2; ++f) dsth[f * 32] = make_float2(row[2 * f], row[2 * f + 1]);
            for (int f = 0; f < kStateDim; ++f) s_row[warp][f] = row[f];
        }
        __syncwarp();
        if (obs) {
            float *o = obs + (size_t)b * kObsFloats;
            for (int i = lane; i < kObsFloats; i += 32)
                o[i] = i < (kSeqLen - 1) * kStateDim ? 0.0f : s_row[warp][i - (kSeqLen - 1) * kStateDim];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// Scene injection: device uavenv_scene_t -> records.  Env first_env + e of the range receives scene e / copies, so
// every replica of a scene is packed from the same values by the same instructions: the copies are bit-identical.

__global__ void __launch_bounds__(kResetThreads) pack_scene_kernel(const __grid_constant__ Params P,
                                                                    const uavenv_scene_t s, int first_env, int count,
                                                                    int copies) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (int env = blockIdx.x * wpb + warp; env < count; env += gridDim.x * wpb) {
        const int b = first_env + env;
        const int e = env / copies;    // the scene
        const int slot = P.header(b).n(I_GEN) & 1;
        for (int i = lane; i < P.K1; i += 32) {
            NfzRec z; z.x = s.nfz_x[(size_t)e * P.K1 + i]; z.y = s.nfz_y[(size_t)e * P.K1 + i];
            z.radius = s.nfz_radius ? s.nfz_radius[(size_t)e * P.K1 + i] : 0.0;
            P.nfz[P.zoff(slot, b) + i] = z;
        }
        for (int i = lane; i < P.K2; i += 32) {
            IntRec r; r.x = s.int_x[(size_t)e * P.K2 + i]; r.y = s.int_y[(size_t)e * P.K2 + i];
            r.vx = s.int_vx[(size_t)e * P.K2 + i]; r.vy = s.int_vy[(size_t)e * P.K2 + i];
            P.intc[P.ioff(slot, b) + i] = r;
        }
        __syncwarp();
        double cost_part = 0.0, val_part = 0.0;
        for (int i = lane; i < P.N; i += 32) {
            const size_t g = (size_t)e * P.N + i;
            UavRec u;
            u.x = s.uav_x[g]; u.y = s.uav_y[g];
            u.load = s.uav_load[g]; u.cost = s.uav_cost[g];
            finish_uav(P, P.nfz + P.zoff(slot, b), P.intc + P.ioff(slot, b), u, s.uav_vx[g], s.uav_vy[g]);
            P.uav[P.uoff(slot, b) + i] = u;
            P.uav_vel[P.uoff(slot, b) + i] = make_double2(s.uav_vx[g], s.uav_vy[g]);
            P.uav_type[P.uoff(slot, b) + i] = s.uav_type ? s.uav_type[g] : 1;
            cost_part += u.cost;
        }
        for (int j = lane; j < P.M; j += 32) {
            const size_t g = (size_t)e * P.M + j;
            TgtRec t;
            t.x = s.tgt_x[g]; t.y = s.tgt_y[g];
            const double vx = s.tgt_vx[g], vy = s.tgt_vy[g];
            t.speed = sqrt(vx * vx + vy * vy);
            t.value = s.tgt_value[g];
            clear_locks(&t, 0); t.id = s.tgt_id[g];
            P.tgt[P.toff(slot, b) + j] = t;
            P.tgt_vel[P.toff(slot, b) + j] = make_double2(vx, vy);
            val_part += t.value;
        }
        const double total_cost = warp_sum(cost_part);
        const double total_val = warp_sum(val_part);
        if (lane == 0) { P.header(b).f(F_TOTAL_COST) = total_cost; P.header(b).f(F_TOTAL_VAL) = total_val; }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// Score matrix (main.py:38-45 over mechanics.py:167-181): p_final / p_damage [B,N,M].
// A warp owns (env, chunk of 32 targets): lane = target (its x, y, speed stay in registers; stores are coalesced along
// the target index), the loop runs over the env's UAVs, whose 64 B records arrive as warp-uniform loads.  Index
// arithmetic and the header read happen once per warp, not once per pair: the first version (a thread per pair with
// 64-bit div / mod and its own record loads) was ISSUE-bound - 81 % of the issue slots, fp64 pipe 47 % active
// (profiles/r2_score_matrix_ncu.md).

template <typename OutT>
__global__ void __launch_bounds__(256) score_matrix_kernel(const __grid_constant__ Params P, OutT *p_final,
                                                            OutT *p_damage) {
    const int lane = threadIdx.x & 31;
    const int chunks = (P.M + 31) >> 5;
    const long long items = (long long)P.B * chunks;
    const long long wstride = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < items; w += wstride) {
        const int b = (int)(w / chunks), m = (int)(w % chunks) * 32 + lane;
        const bool ok = m < P.M;
        const int slot = P.header(b).n(I_GEN) & 1;
        const TgtRec *t = P.tgt + P.toff(slot, b) + (ok ? m : P.M - 1);
        const double tx = t->x, ty = t->y, ts = t->speed;
        const UavRec *U = P.uav + P.uoff(slot, b);
        const size_t out0 = (size_t)b * P.N * P.M + m;
#pragma unroll 2
        for (int k = 0; k < P.N; ++k) {
            const UavRec u = U[k];                                    // warp-uniform address
            double pd;
            const double pf = pair_score(P, u, tx, ty, ts, &pd);
            if (ok) {
                if (p_damage) p_damage[out0 + (size_t)k * P.M] = (OutT)pd;
                if (p_final) p_final[out0 + (size_t)k * P.M] = (OutT)pf;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Fresh objective from the per-target products, a warp per env (uav_env.py:244-293): shuffle
// reductions over targets (revenue, covered value, N0) and UAVs (cost of assigned).  With fix != 0
// the running aggregates are re-anchored to the fresh values.

__global__ void __launch_bounds__(256) recompute_kernel(const __grid_constant__ Params P, int fix,
                                                         double *max_abs_diff) {
    const int lane = threadIdx.x & 31;
    const int wglobal = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    double worst = 0.0;
    for (int b = wglobal; b < P.B; b += nwarps) {
        double rev = 0.0, cval = 0.0, cost = 0.0;
        int n0 = 0;
        const int slot = P.header(b).n(I_GEN) & 1;
        const TgtRec *T = P.tgt + P.toff(slot, b);
        const int episode = P.header(b).n(I_EPISODE), kptr = P.header(b).n(I_K);
        for (int j = lane; j < P.M; j += 32) {
            TgtRec t = T[j];
            const int cnt = target_view(t, episode);
            rev += (1.0 - t.nh) * t.value;
            if (cnt > 0) { cval += t.value; n0 += 1; }
        }
        const UavRec *U = P.uav + P.uoff(slot, b);
        const int32_t *asg = P.assigned + (size_t)b * P.N;
        for (int i = lane; i < min(P.N, kptr); i += 32) if (asg[i] >= 0) cost += U[i].cost;   // slots at / past the pointer are stale
        rev = warp_sum(rev); cval = warp_sum(cval); cost = warp_sum(cost);
        n0 = (int)__reduce_add_sync(kFullMask, (unsigned)n0);
        if (lane == 0) {
            const double J_fresh = objective(P, rev, cost);
            const double J_run = objective(P, P.header(b).f(F_REV), P.header(b).f(F_COST_SUM));
            worst = fmax(worst, fabs(J_fresh - J_run));
            if (n0 != P.header(b).n(I_NCOVERED)) worst = fmax(worst, 1e30);  // integer state must agree exactly
            if (fix) { P.header(b).f(F_REV) = rev; P.header(b).f(F_COST_SUM) = cost; P.header(b).f(F_COVERED_VAL) = cval; }
        }
    }
    if (lane == 0 && max_abs_diff && worst > 0.0) {
        // doubles >= 0 order like their bit patterns
        atomicMax(reinterpret_cast<unsigned long long *>(max_abs_diff), (unsigned long long)__double_as_longlong(worst));
    }
}

// uavenv_set_episode_counters: the new counters, and the records written in an env's current episode follow it (their
// episode tag is what makes them current).  One warp per env.
__global__ void __launch_bounds__(256) set_episode_kernel(const __grid_constant__ Params P, const int32_t *episodes, int first_env,
                                                           int count) {
    const int lane = threadIdx.x & 31;
    const int wglobal = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int e = wglobal; e < count; e += nwarps) {
        const int b = first_env + e;
        const Hdr h = P.header(b);
        const int old_ep = h.n(I_EPISODE), new_ep = episodes[e];
        TgtRec *T = P.tgt + P.toff(h.n(I_GEN) & 1, b);
        for (int j = lane; j < P.M; j += 32)
            if (tag_current(T[j].lock_tag, old_ep)) T[j].lock_tag = make_tag(tag_count(T[j].lock_tag), new_ep);
        __syncwarp();
        if (lane == 0) h.n(I_EPISODE) = new_ep;
    }
}

// Bernoulli(1/2) action stream keyed (seed, step, global env id)
__global__ void random_actions_kernel(const __grid_constant__ Params P, uint32_t s0, uint32_t s1, uint64_t step,
                                      int64_t *actions) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < P.B) {
        const uint4 r = philox4x32(s0, s1, P.env_id_base + (uint32_t)b, (uint32_t)step, (uint32_t)(step >> 32),
                                   0x00AC7101u);
        actions[b] = (int64_t)(r.x >> 31);
    }
}

// ------------------------------------------------------------------------------------------------
// Best-target heuristic (include/uavenv_b200.h, uavenv_best_target_actions).  At the pointer (k, m) of an env:
//   prev_r    = paper_reward(J, N0) (Eq.19) from the carried header sums, as the step kernel's accept test forms it;
//   new_r(j)  = the paper reward after tentatively assigning UAV k to target j: nh' = nh_j * (1 - p_final(k,j)),
//               revenue += (nh_j - nh') * value_j, cost += cost_k, N0 += 1 if target j was uncovered;
//   j*        = argmax_j new_r(j), the lowest index winning a tie;
//   action    = Assign (1) iff m == j* and new_r(j*) >= prev_r, otherwise Skip (0).
// Only an accepted Assign changes the scene's state, and it ends UAV k's row, so j* computed when the pointer enters row
// k holds for the whole row.  A rejected Assign (the env's exact Eq.21 path) lets the row run out.
//
// The caller's cache holds one entry per env: bits 32..63 the episode counter, 16..31 the UAV pointer k, 0..15 the target
// to assign in that row (kNoTarget: none).  An entry is recomputed when its key differs from the env's (episode, k) - an
// auto-reset, a new row, a call skipped at the row's first step - and whenever m == 0 (the first step of every row, so a
// reset() / load_scene(), which restart at (0, 0), never meet a stale entry on their first step).

constexpr int kBestTargetThreads = 256;
constexpr uint32_t kNoTarget = 0xffffu;

__device__ __forceinline__ uint64_t best_target_key(int episode, int k) {
    return ((uint64_t)(uint32_t)episode << 16) | (uint32_t)k;
}

// j* of env e's row k (warp-cooperative, all lanes return it): lanes = targets, as in score_matrix_kernel, pair scores
// (pair_score) and new_r (tentative_assign) as in the step kernel; then a shuffle arg-max
__device__ __noinline__ uint32_t warp_best_target(const Params &P, int e, int k, int episode) {
    const int lane = threadIdx.x & 31;
    const Hdr h = P.header(e);
    const int slot = h.n(I_GEN) & 1, n0 = h.n(I_NCOVERED);
    const double rev = h.f(F_REV), cost_sum = h.f(F_COST_SUM);
    const UavRec u = P.uav[P.uoff(slot, e) + k];                        // warp-uniform address
    const double prev_r = paper_reward(objective(P, rev, cost_sum), n0, P.M);
    const TgtRec *T = P.tgt + P.toff(slot, e);
    double best = -INFINITY;
    int bj = INT_MAX;
    for (int j = lane; j < P.M; j += 32) {
        TgtRec t = T[j];
        const int cnt = target_view(t, episode);
        const double pf = pair_score(P, u, t.x, t.y, t.speed);
        const double r = tentative_assign(P, rev, cost_sum, n0, t.nh, t.value, cnt, pf, u.cost).new_r;
        if (r > best) { best = r; bj = j; }                            // j ascends within a lane: the first maximum stays
    }
    warp_argmax(best, bj);
    return (bj < P.M && best >= prev_r) ? (uint32_t)bj : kNoTarget;
}

__global__ void __launch_bounds__(kBestTargetThreads) best_target_kernel(const __grid_constant__ Params P, int64_t *cache,
                                                                        int64_t *actions) {
    const int lane = threadIdx.x & 31;
    const int b0 = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) & ~(size_t)31);   // first env of this warp
    if (b0 >= P.B) return;                                              // (uniform per warp)
    const int b = b0 + lane;
    const bool live = b < P.B;
    const int bc = live ? b : P.B - 1;
    const Hdr H = P.header(bc);
    const int k = H.n(I_K), m = H.n(I_M), episode = H.n(I_EPISODE);
    const bool active = live && k < P.N && (P.auto_reset || !H.n(I_FINISHED));   // a finished env without auto-reset is inert
    uint64_t entry = (uint64_t)cache[bc];
    const uint64_t key = best_target_key(episode, k);
    const bool stale = active && (m == 0 || (entry >> 16) != key);
    unsigned mask = __ballot_sync(kFullMask, stale);
    while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const int ks = __shfl_sync(kFullMask, k, src), es = __shfl_sync(kFullMask, episode, src);
        const uint32_t j = warp_best_target(P, b0 + src, ks, es);
        if (lane == src) entry = (key << 16) | j;
    }
    if (live) {
        if (stale) cache[b] = (int64_t)entry;
        actions[b] = (active && (uint32_t)(entry & 0xffffu) == (uint32_t)m) ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------
// Best member of each group of group_size consecutive envs (include/uavenv_b200.h, uavenv_group_best): one warp per group.
// Lanes stride over the members (a warp's 32 loads of one header field hit one tile row), keep their first maximum of
// J = objective(rev, cost_sum) (uavenv_get_state's J), and a shuffle arg-max picks the group's member.  The warp then
// copies the winner's assigned[] row along the UAV index.  A group with an unfinished member reports best = -1, J = NaN,
// N0 = -1 and a row of -1.

constexpr int kGroupBestThreads = 256;

__global__ void __launch_bounds__(kGroupBestThreads) group_best_kernel(const __grid_constant__ Params P, int first_env,
                                                                      int num_groups, int group_size, int32_t *best,
                                                                      double *J_best, int32_t *assigned_best,
                                                                      int32_t *num_covered, double *J_all) {
    const int lane = threadIdx.x & 31;
    const int g = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (g >= num_groups) return;                                            // (uniform per warp)
    const int b0 = first_env + g * group_size;
    double bJ = -INFINITY;
    int bi = INT_MAX;
    bool unfinished = false;
    for (int i = lane; i < group_size; i += 32) {
        const Hdr H = P.header(b0 + i);
        const double J = objective(P, H.f(F_REV), H.f(F_COST_SUM));
        if (J_all) J_all[(size_t)g * group_size + i] = J;
        unfinished |= H.n(I_FINISHED) == 0;
        if (bi == INT_MAX || J > bJ) { bJ = J; bi = i; }           // i ascends within a lane: the first maximum stays
    }
    warp_argmax(bJ, bi);
    unfinished = __any_sync(kFullMask, unfinished);
    const Hdr W = P.header(b0 + bi);                                 // (member 0 always exists: bi is a member)
    const int kptr = unfinished ? 0 : W.n(I_K);                      // slots at / past the pointer are stale
    const int32_t *src = P.assigned + (size_t)(b0 + bi) * P.N;
    int32_t *dst = assigned_best + (size_t)g * P.N;
    for (int k = lane; k < P.N; k += 32) dst[k] = k < kptr ? src[k] : -1;
    if (lane == 0) {
        best[g] = unfinished ? -1 : bi;
        J_best[g] = unfinished ? quiet_nan() : bJ;
        num_covered[g] = unfinished ? -1 : W.n(I_NCOVERED);
    }
}

// ------------------------------------------------------------------------------------------------
// Local search on allocations (include/uavenv_b200.h, uavenv_improve_allocation; the rule is stated there and in
// DESIGN §4.9).  Persistent CTAs, one scene at a time per CTA.  The CTA computes its scene's p[N][M] once (warps over UAV
// rows, lanes over targets, score_matrix_kernel's expression) into shared memory when N*M*8 <= kImproveSmemPBytes,
// otherwise into its slice of the caller's workspace (L2-resident: one slice per SM).  t[N], nh[M], nh_excl[N], the
// values and costs live in shared memory.  A round:
//   1. every thread scores a strided share of the N*(M+1) moves and N*(N-1)/2 swaps in candidate order, keeping its
//      first maximum, with the old targets of its best candidate packed beside it;
//   2. a warp-shuffle arg-max, then every warp reduces the 8 warp winners itself (no second barrier): largest gain,
//      lowest candidate index on an exact tie;
//   3. if the winner qualifies, every thread knows the new allocation t' from the winner alone, so the products of the two
//      touched targets (nh) and of their UAVs (nh_excl) are recomputed from scratch over t' in ascending UAV order while
//      thread 0 writes t.  Two barriers per round.

constexpr int kImproveThreads = 256;
constexpr int kImproveWarps = kImproveThreads / 32;
#ifndef UAV_IMPROVE_SMEM_P_BYTES
#define UAV_IMPROVE_SMEM_P_BYTES (64 * 1024)
#endif
constexpr size_t kImproveSmemPBytes = UAV_IMPROVE_SMEM_P_BYTES;   // p in shared memory up to this size (64x64: 32 KB)

struct ImproveIO {
    const int32_t *assigned_in;  // [count][N] Target.id, -1 = none
    int32_t *assigned_out;       // [count][N] (may alias assigned_in: a CTA reads its row before it writes it)
    double *J_in, *J_out;        // [count] (J_in may be NULL)
    int32_t *num_covered, *moves;
    uint8_t *converged;
    double *workspace;           // [gridDim.x][N*M] when p does not fit shared memory, else NULL
    int32_t first_env, count, env_stride, max_moves;
};

__host__ __device__ __forceinline__ bool improve_p_in_smem(int N, int M) {
    return (size_t)N * M * sizeof(double) <= kImproveSmemPBytes;
}
__host__ __device__ __forceinline__ size_t improve_smem_bytes(int N, int M) {
    return (improve_p_in_smem(N, M) ? (size_t)N * M * sizeof(double) : 0) + (size_t)(2 * M + 2 * N) * sizeof(double) +
           (size_t)(N + M) * sizeof(int32_t);
}

// out[k][j] = f(p[k][j]) for the scene's N x M pairs, p = pair_score (uavenv_score_matrix_f64's p_final bits): warps over
// UAV rows, lanes over targets.  The local search keeps p itself, the upper bound a = min(-log1p(-p), A).
template <int kWarps, typename F>
__device__ __forceinline__ void fill_pair_matrix(const Params &P, const UavRec *U, const TgtRec *T, double *out, F f) {
    const int lane = threadIdx.x & 31, M = P.M;
    for (int k = threadIdx.x >> 5; k < P.N; k += kWarps) {
        const UavRec u = U[k];                                               // warp-uniform address
        for (int j = lane; j < M; j += 32) {
            const double tx = T[j].x, ty = T[j].y, ts = T[j].speed;
            out[(size_t)k * M + j] = f(pair_score(P, u, tx, ty, ts));
        }
    }
}

// prod over UAVs i != skip with t'(i) == j, ascending i, of (1 - p[i][j]); t' is t with t'(k1) = n1 and t'(k2) = n2.
// (t[k1] / t[k2] may be rewritten concurrently: their loaded values are never used)
__device__ __forceinline__ double improve_prod(const double *p, const int32_t *t, int N, int M, int j, int skip, int k1,
                                               int n1, int k2, int n2) {
    double q = 1.0;
    for (int i = 0; i < N; ++i) {
        const int ti = i == k1 ? n1 : (i == k2 ? n2 : t[i]);
        if (ti == j && i != skip) q *= 1.0 - p[(size_t)i * M + j];
    }
    return q;
}

// J of the allocation t from its products: targets summed in list order, then the assigned UAVs' costs in UAV order
__device__ __forceinline__ double improve_J(const Params &P, const double *nh, const double *val, const double *cost,
                                            const int32_t *t, int N, int M) {
    double rev = 0.0, c = 0.0;
    for (int j = 0; j < M; ++j) rev += (1.0 - nh[j]) * val[j];
    for (int k = 0; k < N; ++k) if (t[k] >= 0) c += cost[k];
    return objective(P, rev, c);
}

__global__ void __launch_bounds__(kImproveThreads) improve_kernel(const __grid_constant__ Params P, const ImproveIO io) {
    extern __shared__ __align__(16) unsigned char improve_smem[];
    __shared__ double red_g[kImproveWarps];
    __shared__ int red_i[kImproveWarps], red_o[kImproveWarps];
    __shared__ double sh_J;
    __shared__ int sh_n0;
    const int N = P.N, M = P.M, M1 = M + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double omega = P.omega;
    const bool p_smem = improve_p_in_smem(N, M);
    double *sd = reinterpret_cast<double *>(improve_smem);
    double *p = p_smem ? sd : io.workspace + (size_t)blockIdx.x * N * M;
    double *nh = sd + (p_smem ? (size_t)N * M : 0), *val = nh + M, *nhx = val + M, *cost = nhx + N;
    int32_t *t = reinterpret_cast<int32_t *>(cost + N), *ids = t + N;
    const int n_moves = N * M1, n_swaps = N * (N - 1) / 2;
    const int dq = kImproveThreads / M1, dr = kImproveThreads % M1;     // a thread's stride through the moves
    int s1 = 0, r0 = tid;                                                // its first swap (lexicographic index tid)
    while (s1 < N - 1 && r0 >= N - 1 - s1) { r0 -= N - 1 - s1; ++s1; }
    const int s2 = s1 + 1 + r0;

    for (int s = blockIdx.x; s < io.count; s += gridDim.x) {
        const int b = io.first_env + s * io.env_stride;
        const int slot = P.header(b).n(I_GEN) & 1;
        const UavRec *U = P.uav + P.uoff(slot, b);
        const TgtRec *T = P.tgt + P.toff(slot, b);
        for (int j = tid; j < M; j += kImproveThreads) { val[j] = T[j].value; ids[j] = T[j].id; }
        for (int k = tid; k < N; k += kImproveThreads) cost[k] = U[k].cost;
        fill_pair_matrix<kImproveWarps>(P, U, T, p, [](double x) { return x; });
        if (tid == 0) sh_n0 = 0;
        __syncthreads();
        const int32_t *row = io.assigned_in + (size_t)s * N;
        bool bad = false;
        for (int k = tid; k < N; k += kImproveThreads) {
            const int id = row[k];
            int pos = -1;
            if (id < -1) bad = true;
            else if (id >= 0) {
                for (int j = 0; j < M; ++j) if (ids[j] == id) { pos = j; break; }
                bad |= pos < 0;
            }
            t[k] = pos;
        }
        if (__syncthreads_or(bad)) {
            for (int k = tid; k < N; k += kImproveThreads) io.assigned_out[(size_t)s * N + k] = -1;
            if (tid == 0) {
                const double nan = quiet_nan();
                if (io.J_in) io.J_in[s] = nan;
                io.J_out[s] = nan; io.num_covered[s] = -1; io.moves[s] = -1; io.converged[s] = 0;
            }
            __syncthreads();
            continue;
        }
        for (int j = tid; j < M; j += kImproveThreads) nh[j] = improve_prod(p, t, N, M, j, -1, -1, 0, -1, 0);
        for (int k = tid; k < N; k += kImproveThreads)
            nhx[k] = t[k] >= 0 ? improve_prod(p, t, N, M, t[k], k, -1, 0, -1, 0) : 1.0;
        __syncthreads();
        if (tid == 0) {
            sh_J = improve_J(P, nh, val, cost, t, N, M);
            if (io.J_in) io.J_in[s] = sh_J;
        }
        __syncthreads();
        double J = sh_J;                                                     // running J: the threshold's scale
        int moves = 0;
        bool conv = false;
        for (;;) {
            double bg = -INFINITY;
            int bi = INT_MAX, bo = 0;                                        // gain, candidate index, packed old targets
            int k = tid / M1, r = tid % M1;
            for (int idx = tid; idx < n_moves; idx += kImproveThreads) {
                const int a = t[k], bt = r - 1;
                if (bt != a) {
                    double ga = 0.0, gb = 0.0;
                    if (a >= 0) ga = val[a] * (nh[a] - nhx[k]);
                    if (bt >= 0) gb = (val[bt] * nh[bt]) * p[(size_t)k * M + bt];
                    const double g = (ga + gb) + ((omega * cost[k]) * (double)((a >= 0) - (bt >= 0)));
                    if (g > bg) { bg = g; bi = idx; bo = a + 1; }
                }
                k += dq; r += dr;
                if (r >= M1) { r -= M1; ++k; }
            }
            int k1 = s1, k2 = s2;
            for (int idx = tid; idx < n_swaps; idx += kImproveThreads) {
                const int a1 = t[k1], a2 = t[k2];
                if (a1 != a2) {
                    double g1 = 0.0, g2 = 0.0;
                    if (a1 >= 0) g1 = val[a1] * (nh[a1] - (nhx[k1] * (1.0 - p[(size_t)k2 * M + a1])));
                    if (a2 >= 0) g2 = val[a2] * (nh[a2] - (nhx[k2] * (1.0 - p[(size_t)k1 * M + a2])));
                    const double g = (g1 + g2) + ((omega * (cost[k1] - cost[k2])) * (double)((a1 >= 0) - (a2 >= 0)));
                    if (g > bg) { bg = g; bi = n_moves + idx; bo = (a1 + 1) | ((a2 + 1) << 16); }
                }
                k2 += kImproveThreads;
                while (k2 >= N && k1 < N) { ++k1; k2 += k1 + 1 - N; }    // overflow into the next row, which starts at k1 + 1
            }
            // (not warp_argmax: its INT_MAX guard here and in the cross-warp pass cost 1.5-3 % of the kernel, B200 at 1000 W)
            for (int o = 16; o > 0; o >>= 1) {
                const double og = __shfl_xor_sync(kFullMask, bg, o);
                const int oi = __shfl_xor_sync(kFullMask, bi, o), oo = __shfl_xor_sync(kFullMask, bo, o);
                if (og > bg || (og == bg && oi < bi)) { bg = og; bi = oi; bo = oo; }
            }
            if (lane == 0) { red_g[warp] = bg; red_i[warp] = bi; red_o[warp] = bo; }
            __syncthreads();
            bg = red_g[0]; bi = red_i[0]; bo = red_o[0];
            for (int w = 1; w < kImproveWarps; ++w) {
                const double og = red_g[w];
                const int oi = red_i[w];
                if (og > bg || (og == bg && oi < bi)) { bg = og; bi = oi; bo = red_o[w]; }
            }
            if (!(bg > 1e-12 * fmax(1.0, fabs(J)))) { conv = true; break; }  // (uniform: every thread holds the winner)
            if (moves >= io.max_moves) break;
            ++moves;
            J += bg;
            int n1, n2 = 0, ja, jb;                                          // t'(k1) = n1, t'(k2) = n2; touched ja, jb
            if (bi < n_moves) {
                k1 = bi / M1; n1 = bi % M1 - 1; k2 = -1;
                ja = bo - 1; jb = n1;
            } else {
                int q = bi - n_moves;
                k1 = 0;
                while (q >= N - 1 - k1) { q -= N - 1 - k1; ++k1; }
                k2 = k1 + 1 + q;
                ja = (bo & 0xffff) - 1; jb = (bo >> 16) - 1;
                n1 = jb; n2 = ja;
            }
            for (int kk = tid; kk < N; kk += kImproveThreads) {
                const int tk = kk == k1 ? n1 : (kk == k2 ? n2 : t[kk]);
                if (tk < 0) nhx[kk] = 1.0;
                else if (tk == ja || tk == jb) nhx[kk] = improve_prod(p, t, N, M, tk, kk, k1, n1, k2, n2);
            }
            if (tid == kImproveThreads - 1 && ja >= 0) nh[ja] = improve_prod(p, t, N, M, ja, -1, k1, n1, k2, n2);
            if (tid == kImproveThreads - 2 && jb >= 0) nh[jb] = improve_prod(p, t, N, M, jb, -1, k1, n1, k2, n2);
            if (tid == 0) { t[k1] = n1; if (k2 >= 0) t[k2] = n2; }
            __syncthreads();
        }
        // outputs: t, nh are final (last written before the round's barrier)
        int first = 0;                                                       // UAVs that are the first on their target
        for (int kk = tid; kk < N; kk += kImproveThreads) {
            const int tk = t[kk];
            io.assigned_out[(size_t)s * N + kk] = tk >= 0 ? ids[tk] : -1;
            if (tk >= 0) {
                bool f = true;
                for (int i = 0; i < kk && f; ++i) f = t[i] != tk;
                first += f;
            }
        }
        if (first) atomicAdd(&sh_n0, first);
        if (tid == 0) {
            io.J_out[s] = improve_J(P, nh, val, cost, t, N, M);
            io.moves[s] = moves;
            io.converged[s] = conv ? 1 : 0;
        }
        __syncthreads();
        if (tid == 0) io.num_covered[s] = sh_n0;
        __syncthreads();                                                     // before the next scene reuses shared memory
    }
}

// ------------------------------------------------------------------------------------------------
// Upper bound on the best J of a scene (include/uavenv_b200.h, uavenv_upper_bound; the rule and its validity argument
// are stated there and in DESIGN §4.10): Frank-Wolfe on the concave relaxation of J.  Persistent CTAs, one scene at a
// time per CTA, with improve_kernel's launch shape and its home for the N x M matrix (a = min(-log1p(-p), A) in shared
// memory when improve_p_in_smem, else in the CTA's workspace slice).  An iteration:
//   1. nh_j = exp(-s_j) and w_j = v_j nh_j per target; barrier;
//   2. a warp per UAV row: g_kj = w_j a_kj - omega c_k, lanes keep their first maximum, warp_argmax; thread 0 then sums
//      F and sum_j w_j s_j in list order; barrier;
//   3. a thread per target: sigma_j over the picking UAVs in ascending k, d_j = sigma_j - s_j (into nh's storage); thread
//      0 sums the picked gradients and costs in ascending k and forms U_t; barrier;
//   4. the line search: each evaluation of phi' and phi'' is one block_sum2 (one barrier); s_j += gamma d_j.
// Every sum has a fixed order, so the bits depend on the scene alone.

constexpr int kBoundThreads = 256;
constexpr int kBoundWarps = kBoundThreads / 32;
constexpr double kBoundAmax = 40.0;   // a = min(-log1p(-p), A): finite where p = 1
constexpr int kBoundNewton = 10;      // safeguarded Newton steps of the line search

struct BoundIO {
    double *bound, *relaxed;   // [count]
    int32_t *iters;            // [count]
    double *workspace;         // [gridDim.x][N*M] when a does not fit shared memory, else NULL
    int32_t first_env, count, env_stride, max_iters;
};

__host__ __device__ __forceinline__ size_t bound_smem_bytes(int N, int M) {
    return (improve_p_in_smem(N, M) ? (size_t)N * M * sizeof(double) : 0) + (size_t)(4 * M + 2 * N) * sizeof(double) +
           (size_t)N * sizeof(int32_t);
}

// (sum of x1, sum of x2) over the CTA in a fixed order: each thread's strided share of targets (added in ascending j,
// from 0), warp_sum, then the warps' totals from warp 0 up, read by every thread.  red[2][2][kBoundWarps] alternates
// halves by `par`, so one barrier per call suffices (a half is rewritten only after the next call's barrier).
__device__ __forceinline__ void block_sum2(double x1, double x2, double (*red)[2][kBoundWarps], int &par, double &r1,
                                           double &r2) {
    const int warp = threadIdx.x >> 5;
    x1 = warp_sum(x1); x2 = warp_sum(x2);
    if ((threadIdx.x & 31) == 0) { red[par][0][warp] = x1; red[par][1][warp] = x2; }
    __syncthreads();
    r1 = red[par][0][0]; r2 = red[par][1][0];
    for (int w = 1; w < kBoundWarps; ++w) { r1 += red[par][0][w]; r2 += red[par][1][w]; }
    par ^= 1;
}

__global__ void __launch_bounds__(kBoundThreads) bound_kernel(const __grid_constant__ Params P, const BoundIO io) {
    extern __shared__ __align__(16) unsigned char bound_smem[];
    __shared__ double red[2][2][kBoundWarps];
    __shared__ double sh_F, sh_U, sh_dC, sh_margin;
    const int N = P.N, M = P.M;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double omega = P.omega;
    const bool a_smem = improve_p_in_smem(N, M);
    double *sd = reinterpret_cast<double *>(bound_smem);
    double *a = a_smem ? sd : io.workspace + (size_t)blockIdx.x * N * M;
    double *s = sd + (a_smem ? (size_t)N * M : 0), *w = s + M, *nh = w + M, *val = nh + M, *cost = val + M, *gp = cost + N;
    double *d = nh;                                                          // d_j replaces nh_j once F is summed
    int32_t *pick = reinterpret_cast<int32_t *>(gp + N);
    int par = 0;

    for (int sc = blockIdx.x; sc < io.count; sc += gridDim.x) {
        const int b = io.first_env + sc * io.env_stride;
        const int slot = P.header(b).n(I_GEN) & 1;
        const UavRec *U = P.uav + P.uoff(slot, b);
        const TgtRec *T = P.tgt + P.toff(slot, b);
        for (int j = tid; j < M; j += kBoundThreads) { val[j] = T[j].value; s[j] = 0.0; }
        for (int k = tid; k < N; k += kBoundThreads) cost[k] = U[k].cost;
        fill_pair_matrix<kBoundWarps>(P, U, T, a, [](double p) { return fmin(-log1p(-p), kBoundAmax); });
        __syncthreads();
        if (tid == 0) {
            double tv = 0.0, tc = 0.0;                                       // list order, UAV order
            for (int j = 0; j < M; ++j) tv += val[j];
            for (int k = 0; k < N; ++k) tc += cost[k];
            sh_margin = tv * exp(-kBoundAmax) + 1e-12 * (tv + omega * tc);
        }
        double C = 0.0, best = INFINITY, F = 0.0;
        int t = 0;
        for (;;) {
            ++t;
            for (int j = tid; j < M; j += kBoundThreads) {
                const double e = exp(-s[j]);
                nh[j] = e; w[j] = val[j] * e;
            }
            __syncthreads();
            for (int k = warp; k < N; k += kBoundWarps) {
                const double ock = omega * cost[k];
                const double *ak = a + (size_t)k * M;
                double bg = -INFINITY;
                int bj = INT_MAX;
                for (int j = lane; j < M; j += 32) {
                    const double g = w[j] * ak[j] - ock;
                    if (g > bg) { bg = g; bj = j; }
                }
                warp_argmax(bg, bj);
                if (lane == 0) { pick[k] = bg > 0.0 ? bj : -1; gp[k] = bg > 0.0 ? bg : 0.0; }
            }
            if (tid == 0) {
                double rev = 0.0, lin = 0.0;
                for (int j = 0; j < M; ++j) { rev += val[j] * (1.0 - nh[j]); lin += w[j] * s[j]; }
                sh_F = objective(P, rev, C);
                sh_U = lin;                                                  // sum_j w_j s_j until step 3
            }
            __syncthreads();
            for (int j = tid; j < M; j += kBoundThreads) {
                double sg = 0.0;
                for (int k = 0; k < N; ++k) if (pick[k] == j) sg += a[(size_t)k * M + j];
                d[j] = sg - s[j];
            }
            if (tid == 0) {
                double G = 0.0, Cs = 0.0;
                for (int k = 0; k < N; ++k) { G += gp[k]; if (pick[k] >= 0) Cs += cost[k]; }
                sh_U = (sh_F + G) - objective(P, sh_U, C);
                sh_dC = Cs - C;
            }
            __syncthreads();
            F = sh_F;
            const double Ut = sh_U, dC = sh_dC;
            best = fmin(best, Ut);
            if (Ut - F <= 1e-9 * fmax(1.0, fabs(Ut)) || t >= io.max_iters) break;   // (uniform)
            // line search on phi(gamma) = F(s + gamma d, C + gamma dC): phi' = sum_j (v_j e_j) d_j - omega dC and
            // phi'' = -sum_j ((v_j e_j) d_j) d_j with e_j = exp(-(s_j + gamma d_j))
            double gam = 1.0, p1, p2;
            auto eval = [&](double g) {
                double x1 = 0.0, x2 = 0.0;
                for (int j = tid; j < M; j += kBoundThreads) {
                    const double q = (val[j] * exp(-(s[j] + g * d[j]))) * d[j];
                    x1 += q; x2 += q * d[j];
                }
                double r1, r2;
                block_sum2(x1, x2, red, par, r1, r2);
                p1 = r1 - omega * dC; p2 = r2;                               // p2 = -phi''
            };
            eval(1.0);
            if (p1 < 0.0) {
                double lo = 0.0, hi = 1.0;
                for (int i = 0; i < kBoundNewton; ++i) {
                    double c = gam + p1 / p2;
                    if (c == gam) break;         // converged: a step below gamma's last bit (or phi' = 0 exactly)
                    if (!(c > lo && c < hi)) c = 0.5 * (lo + hi);
                    gam = c;
                    eval(gam);
                    if (p1 > 0.0) lo = gam; else hi = gam;
                }
            }
            for (int j = tid; j < M; j += kBoundThreads) s[j] = s[j] + gam * d[j];
            C = C + gam * dC;
        }
        if (tid == 0) {
            io.bound[sc] = best + sh_margin;
            io.relaxed[sc] = F;
            io.iters[sc] = t;
        }
        __syncthreads();                                                     // before the next scene reuses shared memory
    }
}

}  // namespace uavk
