// uavenv_device.cuh - device-side records and scalar building blocks of the batched
// UAV->target allocation environment (sm_100a).
//
// Reference semantics: envs/mechanics.py:11-241 (scores, observation row), envs/entities.py:13-61
// (entity state).  All score arithmetic is fp64 in the reference's operation order (this file is
// compiled with -fmad=false) because the Eq.21 accept test `new_r >= prev_r`
// (envs/uav_env.py:317) has to come out bit-identical to the reference's fp64 decision.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "philox.cuh"

namespace uavk {

constexpr int kStateDim = 14;  // configs/config.py:61
constexpr int kSeqLen = 5;     // configs/config.py:62
constexpr int kObsFloats = kStateDim * kSeqLen;

// ------------------------------------------------------------------------------------------------
// HBM layout.  Entities are 64-byte records, contiguous per env ("the env's tile"): a pointer pair
// (k, m) costs one 64 B gather per record, and the cooperative reset / scene generation /
// score-matrix paths stream the tile with fully coalesced accesses.

struct __align__(64) UavRec {  // envs/entities.py:13-36 (live fields) + per-scene derived values
    double x, y;               // sector 0: position
    double wx, wy;             //   unit heading velocity/||velocity||, (1,0) when ||velocity|| < 1e-6 (mechanics.py:31-36)
    double load, cost;         // sector 1
    double p_pen;              //   calc_penetration_prob(uav): target-independent (mechanics.py:118-163)
    double inv_speed;          //   1/||velocity||, or -1 when ||velocity|| < 1e-6 (mechanics.py:65)
};

struct __align__(64) TgtRec {  // envs/entities.py:39-49 + velocity norm (uav_env.py:141, mechanics.py:100)
    double x, y, speed, value; // sector 0: static
    double nh;                 // sector 1: prod(1 - p_final) over the lock list  ("target health")
    double nh_pure;            //           prod(1 - p_damage)
    double lock_cost;          //           sum of costs of the UAVs locked on it (chi_mc numerator)
    int32_t lock_tag;          //           len(locked_by_uavs) (bits 0..13; covered ("kill flag") <=> count > 0) | episode tag
                               //           (bits 14..31): the four dynamic fields are those of the env's CURRENT episode only
                               //           if the tag matches it - otherwise they read as cleared (see target_view)
    int32_t id;                //           Target.id (list position != id after the shuffle, uav_env.py:173)
};
static_assert(sizeof(UavRec) == 64 && sizeof(TgtRec) == 64, "records must be one 64 B line half");

// A restarted env (uav_env.py:175-182) does not touch its M target records: they carry the episode they were last
// written in, and a record of another episode is read as cleared.  (Aliasing needs a record left untouched for 2^18
// episodes; the step kernel wipes the arrays every 2^16 episodes, so it cannot happen.)
constexpr int kTagShift = 14;
constexpr uint32_t kEpochMask = 0x3ffffu;
__host__ __device__ __forceinline__ int32_t make_tag(int count, int episode) {
    return (int32_t)((uint32_t)count | (((uint32_t)episode & kEpochMask) << kTagShift));
}
__host__ __device__ __forceinline__ int tag_count(int32_t tag) { return (int)((uint32_t)tag & ((1u << kTagShift) - 1u)); }
__host__ __device__ __forceinline__ bool tag_current(int32_t tag, int episode) {
    return ((uint32_t)tag >> kTagShift) == ((uint32_t)episode & kEpochMask);
}
// the record as the env sees it in `episode`: returns the lock count, clears nh / nh_pure / lock_cost of a stale record
__host__ __device__ __forceinline__ int target_view(TgtRec &t, int episode) {
    if (tag_current(t.lock_tag, episode)) return tag_count(t.lock_tag);
    t.nh = 1.0; t.nh_pure = 1.0; t.lock_cost = 0.0;
    return 0;
}
// an empty lock list for record T[j] (indexed: a TgtRec & form changes reset_kernel's register allocation)
__host__ __device__ __forceinline__ void clear_locks(TgtRec *T, int j) {
    T[j].nh = 1.0; T[j].nh_pure = 1.0; T[j].lock_cost = 0.0; T[j].lock_tag = 0;
}

struct NfzRec { double x, y, radius; };            // envs/entities.py:52-55
struct IntRec { double x, y, vx, vy; };            // envs/entities.py:58-61 + velocity (uav_env.py:168)

// Scalar per-env state.  Tile-major structure-of-arrays: the 32 envs of a warp own one contiguous
// 4.75 KB tile [field][32 lanes] (f64 fields first, then i32 fields), so a warp reads its whole header
// with fully coalesced loads at immediate offsets from ONE base pointer, out of one DRAM neighbourhood.
enum F64Field {
    F_REV,            // sum_m (1 - nh_m) * value_m              envs/uav_env.py:264-265
    F_COST_SUM,       // sum of costs of assigned UAVs           envs/uav_env.py:262 / :195
    F_COVERED_VAL,    // sum of values of covered targets        envs/uav_env.py:199
    F_SUM_PD, F_SUM_PF,  // sums over locked pairs               envs/uav_env.py:370-408
    F_TOTAL_VAL,      // sum of target values (per scene)        envs/uav_env.py:198
    F_TOTAL_COST,     // total_swarm_cost (per scene)            envs/uav_env.py:118
    // the CURRENT pointer pair (k,m), captured when its observation row was computed, so that the
    // accept rule of the next step needs no gather:
    F_CUR_PF, F_CUR_PD,    // calc_advantage(uav_k, target_m)    mechanics.py:167-181
    F_CUR_VALUE,           // target_m.value
    F_CUR_NH, F_CUR_NHP,   // target_m products before this decision
    F_CUR_LOCK_COST,       // target_m lock cost
    F_CUR_UCOST,           // uav_k.cost
    NF64
};
enum I32Field {
    I_K, I_M,         // uav_idx / target_idx                    envs/uav_env.py:33-34
    I_NASSIGNED,      // number of locked (UAV,target) pairs A
    I_NCOVERED,       // N0                                      envs/uav_env.py:278-282
    I_AGE,            // valid rows of the observation window (0..5)
    I_EPISODE,        // 1-based episode counter                 main_train.py:77
    I_GEN,            // (index of the NEXT scene to generate << 1) | storage slot of the current scene.
                      // One word so the pre-generation service reads a consistent pair.  Written by the env's owner.
    I_CUR_LOCK_CNT,   // target_m lock count
    I_CUR_TID,        // target_m.id
    I_FINISHED,       // auto_reset = 0 only
    I_NEXT_TAG,       // scene index held complete in the OTHER slot (-1: none).   Written by the service only.
    I_SPARE,
    NI32
};
constexpr size_t kHdrTileBytes = (size_t)NF64 * 32 * sizeof(double) + (size_t)NI32 * 32 * sizeof(int32_t);
constexpr int kRingTileElems = 5 * 7 * 32;  // float2 elements of one warp tile of the observation ring
// header tile and ring tile of a warp are adjacent: one 13.75 KB neighbourhood (one TLB page) per warp for all of its
// streamed per-env state
constexpr size_t kEnvTileBytes = kHdrTileBytes + (size_t)kRingTileElems * sizeof(float2);

struct Hdr {  // view of one env's header: field x lives at d[x*32] / i[x*32]
    double *d;
    int32_t *i;
    __host__ __device__ __forceinline__ double &f(int x) const { return d[x * 32]; }
    __host__ __device__ __forceinline__ int32_t &n(int x) const { return i[x * 32]; }
};
__host__ __device__ __forceinline__ Hdr header_at(unsigned char *base, int b) {
    unsigned char *tile = base + (size_t)(b >> 5) * kEnvTileBytes;
    Hdr h;
    h.d = reinterpret_cast<double *>(tile) + (b & 31);
    h.i = reinterpret_cast<int32_t *>(tile + (size_t)NF64 * 32 * sizeof(double)) + (b & 31);
    return h;
}

struct Params {
    int32_t B, N, M, K1, K2;
    int32_t reset_episodes, auto_reset;
    double zeta_d, inv_zeta_d, k, c1, c2, c3, c4, omega, tie_band;
    double weather_speed, weather_load;
    double map_w, map_h, uav_x_lo, uav_x_hi, tgt_x_lo, tgt_x_hi, intercept_rad;
    uint32_t seed_lo, seed_hi;
    uint32_t env_id_base;
    // device arrays.  Scene storage is double-buffered ([2 slots]...): the current scene of an env lives in
    // slot (I_GEN & 1); the other slot receives the env's NEXT scene ahead of time (pre-generation service),
    // so the scheduled regeneration of main_train.py:79 is a slot flip on the step's critical path.
    UavRec *uav;        // [2][B][N]
    TgtRec *tgt;        // [2][B][M]
    int32_t *assigned;  // [B][N]  target id or -1     envs/entities.py:30
    int32_t *uav_type;  // [2][B][N]  cold
    double2 *uav_vel;   // [2][B][N]  cold (the records keep heading + speed)
    double2 *tgt_vel;   // [2][B][M]  cold
    NfzRec *nfz;        // [2][B][K1]
    IntRec *intc;       // [2][B][K2]
    // pre-generation service (uavenv_kernels.cuh): per-CTA launch counters and two alternating job queues
    uint32_t *svc_ctr;  // [service CTAs] launches seen by each service CTA (all equal: every CTA runs in every launch)
    uint32_t *q_count;  // [2] entries of each queue
    int32_t *q_env;     // [2][B] env of the entry
    int32_t *q_gen;     // [2][B] its I_GEN word when it was queued
    int32_t *q_done;    // [2][B] chunks finished
    uint32_t *step_ctr; // [0] = ring head (mod 5), [1] = CTA arrival counter of the running step
    unsigned char *hdr; // [B/32] env tiles (kEnvTileBytes each): header tile, then the observation ring tile
                        // [5 slots][7 feature pairs][32 lanes] float2
    __host__ __device__ __forceinline__ Hdr header(int b) const { return header_at(hdr, b); }
    __host__ __device__ __forceinline__ size_t uoff(int slot, int b) const { return ((size_t)slot * B + b) * N; }
    __host__ __device__ __forceinline__ size_t toff(int slot, int b) const { return ((size_t)slot * B + b) * M; }
    __host__ __device__ __forceinline__ size_t zoff(int slot, int b) const { return ((size_t)slot * B + b) * K1; }
    __host__ __device__ __forceinline__ size_t ioff(int slot, int b) const { return ((size_t)slot * B + b) * K2; }
    // ring element (slot, feature pair f) of env b: ring(b)[slot * 224 + f * 32]
    __host__ __device__ __forceinline__ float2 *ring(int b) const {
        return reinterpret_cast<float2 *>(hdr + (size_t)(b >> 5) * kEnvTileBytes + kHdrTileBytes) + (b & 31);
    }
};

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (philox.cuh): counter = (element, stream, scene index, global env id),
// key = seed.  (tests cross-check raw blocks and whole scenes against an independent CPU implementation)

__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {  // uniform [0,1) on the 2^-53 grid
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0);
}

enum Stream : uint32_t {  // draw list of envs/uav_env.py:65-173 (SURVEY.md §3.3)
    S_UAV_TYPE = 1, S_UAV_POS = 2, S_UAV_DYN = 3, S_N2 = 4, S_TGT_VAL = 5, S_TGT_POS = 6, S_TGT_VEL = 7,
    S_NFZ_A = 8, S_NFZ_B = 9, S_INT_A = 10, S_INT_B = 11, S_TGT_LIST = 12
};

// ------------------------------------------------------------------------------------------------
// Scores (fp64, reference operation order)

__device__ __forceinline__ double clip01(double v) { return v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v); }

// envs/mechanics.py:11-57 calc_angle_score (Eq.1) with the UAV's unit heading (wx,wy) precomputed.
// cos(sigma) is formed as (d . w)/|d| (one division) instead of (d/|d|) . w: <= 2 ulp apart.
__device__ __forceinline__ double angle_score(double ux, double uy, double wx, double wy, double tx, double ty,
                                              double &dist) {
    const double dx = tx - ux, dy = ty - uy;
    dist = sqrt(dx * dx + dy * dy);
    if (dist < 1e-6) return 1.0;                                   // :23
    double c = (dx * wx + dy * wy) / dist;                         // :28-39
    c = c < -1.0 ? -1.0 : (c > 1.0 ? 1.0 : c);
    const double sigma = acos(c);                                  // :40
    double b = 0.002 * dist;                                       // :44
    if (b < 1e-6) b = 1e-6;                                        // :51
    const double q = sigma / (b * 3.141592653589793);
    return exp(-(q * q));                                          // :55-56
}

// envs/mechanics.py:61-68 calc_speed_score (Eq.2); inv_speed < 0 encodes uav_speed < 1e-6
__device__ __forceinline__ double speed_score(double kparam, double inv_speed, double tgt_speed) {
    if (inv_speed < 0.0) return 0.0;
    return clip01(1.0 - (kparam * tgt_speed * inv_speed));
}

// envs/mechanics.py:72-89 calc_dist_score (Eq.3), D_mid = 0
__device__ __forceinline__ double dist_score(double dist, double inv_zeta) {
    const double q = dist * inv_zeta;
    return exp(-(q * q));
}

// envs/mechanics.py:93-114 calc_damage_prob (Eq.4)
__device__ __forceinline__ double damage_prob(const Params &P, const UavRec &u, double tx, double ty, double tspeed) {
    double dist;
    const double e_angle = angle_score(u.x, u.y, u.wx, u.wy, tx, ty, dist);
    const double e_dist = dist_score(dist, P.inv_zeta_d);
    const double e_speed = speed_score(P.k, u.inv_speed, tspeed);
    const double term = P.c1 * e_dist + P.c2 * e_speed;            // :111
    return clip01(e_angle * term * u.load);                        // :112-114
}

// envs/mechanics.py:167-181 calc_advantage: p_final of UAV u on the target at (tx, ty) moving at tspeed (*pd = p_damage)
__device__ __forceinline__ double pair_score(const Params &P, const UavRec &u, double tx, double ty, double tspeed,
                                             double *pd = nullptr) {
    const double d = damage_prob(P, u, tx, ty, tspeed);
    if (pd) *pd = d;
    return d * u.p_pen;                                            // :179
}

// envs/mechanics.py:118-163 calc_penetration_prob (Eq.5-6): depends on the UAV only
__device__ __forceinline__ double penetration_prob(const Params &P, const NfzRec *Z, const IntRec *I, const UavRec &u) {
    double p = 1.0;
    for (int i = 0; i < P.K1; ++i) {                               // :130-141
        double dist;
        const double ea = angle_score(u.x, u.y, u.wx, u.wy, Z[i].x, Z[i].y, dist);
        const double qd = dist / 10.0, ed = exp(-(qd * qd));       // zeta = 10 for obstacles (:78)
        p *= clip01((1.0 - ea) * (1.0 - ed));
    }
    for (int i = 0; i < P.K2; ++i) {                               // :144-161
        double dist;
        const double ea = angle_score(u.x, u.y, u.wx, u.wy, I[i].x, I[i].y, dist);
        const double qd = dist / 10.0, ed = exp(-(qd * qd));
        const double ispeed = sqrt(I[i].vx * I[i].vx + I[i].vy * I[i].vy);
        const double es = speed_score(P.k, u.inv_speed, ispeed);
        const double term = P.c3 * (1.0 - ed) + P.c4 * es;
        p *= clip01((1.0 - ea) * term);
    }
    return p;
}

// derived fields of a UAV record from its velocity (unit heading, 1/speed) ...
__device__ __forceinline__ void finish_uav_kinematics(UavRec &u, double vx, double vy) {
    const double speed = sqrt(vx * vx + vy * vy);
    if (speed < 1e-6) { u.wx = 1.0; u.wy = 0.0; u.inv_speed = -1.0; }
    else { u.wx = vx / speed; u.wy = vy / speed; u.inv_speed = 1.0 / speed; }
}
// ... and from the scene's obstacles Z[K1], I[K2] (any address space)
__device__ __forceinline__ void finish_uav(const Params &P, const NfzRec *Z, const IntRec *I, UavRec &u, double vx, double vy) {
    finish_uav_kinematics(u, vx, vy);
    u.p_pen = penetration_prob(P, Z, I, u);
}

// envs/mechanics.py:185-241 get_state_vector (Eq.15): fp64 features, cast to f32, then the power-of-two
// scalings applied in f32 exactly as the reference does (:235-239).
__device__ __forceinline__ void state_vector(double cost, double value, double chi_c, double chi_v, double chi_mc,
                                             double p_km, double p_km_dmg, double prev_joint_p, double prev_revenue,
                                             double prev_joint_p_pure, float *o) {
    const double hat_p = 1.0 - (1.0 - prev_joint_p) * (1.0 - p_km);            // :196
    const double hat_p_pure = 1.0 - (1.0 - prev_joint_p_pure) * (1.0 - p_km_dmg);  // :199
    const double hat_G = hat_p * value;                                        // :201
    o[0] = (float)cost * 0.5f;
    o[1] = (float)value * 0.0625f;
    o[2] = (float)chi_c;
    o[3] = (float)chi_v;
    o[4] = (float)chi_mc;
    o[5] = (float)p_km;
    o[6] = (float)prev_joint_p;
    o[7] = (float)hat_p;
    o[8] = (float)prev_revenue * 0.0625f;
    o[9] = (float)hat_G * 0.0625f;
    o[10] = (float)(p_km_dmg - p_km);                                          // :204
    o[11] = (float)(hat_p_pure - hat_p);                                       // :205
    o[12] = (float)((hat_p_pure * value) - hat_G) * 0.0625f;                   // :206
    o[13] = 1.0f;  // float(uav.available): the pointer UAV is always unassigned (uav_env.py:317-324)
}

// envs/uav_env.py:268 _calc_J_X: J from the revenue and the summed cost of the assigned UAVs (every J of the library)
__host__ __device__ __forceinline__ double objective(const Params &P, double rev, double cost) { return rev - (P.omega * cost); }

// envs/uav_env.py:271-293 _calculate_paper_reward (Eq.19) from the running aggregates
__device__ __forceinline__ double paper_reward(double J, int n0, int M) {
    return (n0 == M) ? 2.0 * J : J * ((double)n0 / (double)M);
}

// X' = X + (UAV -> target) (uav_env.py:308-313) from the carried aggregates: only the target's product nh, the revenue,
// the cost sum and N0 change.  (nh, value, lock_cnt: the target; pf: the pair's p_final; ucost: the UAV's cost)
struct Tentative { double nh2, rev2, cost2, new_r; int n02; };
__device__ __forceinline__ Tentative tentative_assign(const Params &P, double rev, double cost_sum, int n0, double nh,
                                                      double value, int lock_cnt, double pf, double ucost) {
    Tentative x;
    x.nh2 = nh * (1.0 - pf);
    x.rev2 = rev + ((1.0 - x.nh2) - (1.0 - nh)) * value;
    x.cost2 = cost_sum + ucost;
    x.n02 = n0 + (lock_cnt == 0);
    x.new_r = paper_reward(objective(P, x.rev2, x.cost2), x.n02, P.M);   // :313
    return x;
}

}  // namespace uavk
