// uavenv_capi.cu - the C ABI declared in include/uavenv_b200.h over the sm_100a kernels.
// Host side only: owns the device arrays, validates arguments, enqueues kernels on the caller's
// stream.  No exception leaves this file; every failure becomes a negative return + message.
#include "uavenv_b200.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "handle.cuh"
#include "uavenv_kernels.cuh"

using namespace uavk;
using capi::fail;

struct uavenv : capi::Handle {
    uavenv_cfg_t cfg;
    int32_t B = 0;
    uint64_t seed = 0, env_id_base = 0;
    Params P;
    float *obs_buf = nullptr;        // [B,5,14] handle-owned window buffer
    int64_t *d_actions = nullptr;    // staging for uavenv_step_host
    float *d_reward = nullptr;
    uint8_t *d_done = nullptr;
    double *d_scratch = nullptr;     // one double (recompute max diff)
    size_t reset_smem = 0;
    int n_service = 0;
    bool ready = false;              // reset() or load_scene() happened
};

extern "C" void uavenv_default_cfg(uavenv_cfg_t *c) {
    if (!c) return;
    std::memset(c, 0, sizeof *c);
    c->num_uavs = 30; c->num_targets = 10; c->num_nfz = 1; c->num_interceptors = 1;
    c->reset_episodes = 200; c->auto_reset = 1;
    c->param_zeta_d = 150.0; c->param_k = 1.2;
    c->param_c1 = 0.75; c->param_c2 = 0.25; c->param_c3 = 0.75; c->param_c4 = 0.25;
    c->cost_weight_omega = 0.0;
    c->weather_speed_factor = 1.0; c->weather_load_factor = 1.0;
    c->map_width = 180.0; c->map_height = 160.0;
    c->uav_gen_x_lo = 60.0; c->uav_gen_x_hi = 90.0;
    c->target_gen_x_lo = 160.0; c->target_gen_x_hi = 180.0;
    c->intercept_rad = 2.0;
    c->tie_band = 1e-12;
}

extern "C" int uavenv_abi_version(void) { return UAVENV_ABI_VERSION; }
extern "C" int32_t uavenv_num_envs(const uavenv_t *h) { return h ? h->B : 0; }
extern "C" const char *uavenv_last_error(const uavenv_t *h) { return capi::last_error(h); }
extern "C" float *uavenv_obs_buffer(uavenv_t *h) { return h ? h->obs_buf : nullptr; }

static int create_impl(uavenv *h) {
    const uavenv_cfg_t &c = h->cfg;
    const size_t B = (size_t)h->B, N = (size_t)c.num_uavs, M = (size_t)c.num_targets;
    const size_t K1 = (size_t)c.num_nfz, K2 = (size_t)c.num_interceptors;
    CU_TRY(h, cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CU_TRY(h, cudaGetDeviceProperties(&prop, h->device));
    if (prop.major < 10)
        return fail(h, UAVENV_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", h->device,
                    prop.major, prop.minor);
    Params &P = h->P;
    std::memset(&P, 0, sizeof P);
    P.B = h->B; P.N = c.num_uavs; P.M = c.num_targets; P.K1 = c.num_nfz; P.K2 = c.num_interceptors;
    P.reset_episodes = c.reset_episodes; P.auto_reset = c.auto_reset ? 1 : 0;
    P.zeta_d = c.param_zeta_d; P.inv_zeta_d = 1.0 / c.param_zeta_d; P.k = c.param_k; P.c1 = c.param_c1; P.c2 = c.param_c2; P.c3 = c.param_c3;
    P.c4 = c.param_c4; P.omega = c.cost_weight_omega; P.tie_band = c.tie_band;
    P.weather_speed = c.weather_speed_factor; P.weather_load = c.weather_load_factor;
    P.map_w = c.map_width; P.map_h = c.map_height;
    P.uav_x_lo = c.uav_gen_x_lo; P.uav_x_hi = c.uav_gen_x_hi;
    P.tgt_x_lo = c.target_gen_x_lo; P.tgt_x_hi = c.target_gen_x_hi; P.intercept_rad = c.intercept_rad;
    P.seed_lo = (uint32_t)h->seed; P.seed_hi = (uint32_t)(h->seed >> 32);
    P.env_id_base = (uint32_t)h->env_id_base;
    // scene storage is double-buffered (current scene + the pre-generated next one)
    CU_TRY(h, capi::alloc(h, &P.uav, 2 * B * N));
    CU_TRY(h, capi::alloc(h, &P.tgt, 2 * B * M));
    CU_TRY(h, capi::alloc(h, &P.assigned, B * N));
    CU_TRY(h, capi::alloc(h, &P.uav_type, 2 * B * N));
    CU_TRY(h, capi::alloc(h, &P.uav_vel, 2 * B * N));
    CU_TRY(h, capi::alloc(h, &P.tgt_vel, 2 * B * M));
    CU_TRY(h, capi::alloc(h, &P.nfz, 2 * B * K1));
    CU_TRY(h, capi::alloc(h, &P.intc, 2 * B * K2));
    // pre-generation service: one CTA per 1024 envs (only when scenes are ever regenerated, and when a warp's
    // shared-memory scratch holds the scene's obstacles)
    const size_t n_svc = (B + kServiceEnvsPerCta - 1) / kServiceEnvsPerCta;
    h->n_service = (c.auto_reset && c.reset_episodes > 0 &&
                    K1 * sizeof(NfzRec) + K2 * sizeof(IntRec) <= (size_t)kServiceScratchPerWarp) ? (int)n_svc : 0;
    CU_TRY(h, capi::alloc(h, &P.svc_ctr, n_svc));
    CU_TRY(h, cudaMemset(P.svc_ctr, 0, n_svc * sizeof(uint32_t)));
    CU_TRY(h, capi::alloc(h, &P.q_count, 2));
    CU_TRY(h, cudaMemset(P.q_count, 0, 2 * sizeof(uint32_t)));
    CU_TRY(h, capi::alloc(h, &P.q_env, 2 * B));
    CU_TRY(h, capi::alloc(h, &P.q_gen, 2 * B));
    CU_TRY(h, capi::alloc(h, &P.q_done, 2 * B));
    const size_t tiles = (B + 31) / 32;
    CU_TRY(h, capi::alloc(h, &P.step_ctr, 2));
    CU_TRY(h, capi::alloc(h, &P.hdr, tiles * kEnvTileBytes));
    {   // headers start zeroed, with "no scene prepared" in the service-owned words
        std::vector<unsigned char> init(tiles * kEnvTileBytes, 0);
        for (size_t b = 0; b < tiles * 32; ++b) {
            const Hdr hv = header_at(init.data(), (int)b);
            hv.n(I_NEXT_TAG) = -1;
        }
        CU_TRY(h, cudaMemcpy(P.hdr, init.data(), init.size(), cudaMemcpyHostToDevice));
    }
    CU_TRY(h, cudaMemset(P.step_ctr, 0, 2 * sizeof(uint32_t)));
    CU_TRY(h, cudaMemset(P.assigned, 0xff, B * N * sizeof(int32_t)));
    CU_TRY(h, capi::alloc(h, &h->obs_buf, B * kObsFloats));
    CU_TRY(h, capi::alloc(h, &h->d_actions, B));
    CU_TRY(h, capi::alloc(h, &h->d_reward, B));
    CU_TRY(h, capi::alloc(h, &h->d_done, B));
    CU_TRY(h, capi::alloc(h, &h->d_scratch, 1));
    // per-warp scratch of the scene generator: max(N,M) sort keys, for the 4 warps of a CTA
    h->reset_smem = (size_t)std::max(kWarpsPerCta, kResetThreads / 32) * std::max(N, M) * sizeof(uint32_t);
    if (h->reset_smem > 8 * 1024) {
        // process-wide function attributes: never lower what another handle (larger N, M) has already asked for
        static size_t attr_smem = 0;
        if (h->reset_smem > attr_smem) {
            CU_TRY(h, cudaFuncSetAttribute(step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->reset_smem));
            CU_TRY(h, cudaFuncSetAttribute(reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->reset_smem));
            attr_smem = h->reset_smem;
        }
    }
    CU_TRY(h, cudaDeviceSynchronize());
    return UAVENV_OK;
}

extern "C" int uavenv_create(const uavenv_cfg_t *cfg, int32_t num_envs, int32_t device, uint64_t seed,
                             uint64_t env_id_base, uavenv_t **out) {
    if (!cfg) return fail<uavenv>(nullptr, UAVENV_EINVAL, "uavenv_create: cfg is NULL");
    if (int rc = capi::check_create_args("uavenv_create", "num_envs", num_envs, out)) return rc;
    if (cfg->num_uavs <= 0 || cfg->num_targets <= 0 || cfg->num_nfz < 0 || cfg->num_interceptors < 0)
        return fail<uavenv>(nullptr, UAVENV_EINVAL, "uavenv_create: need num_uavs > 0, num_targets > 0, obstacles >= 0");
    if (cfg->num_uavs > 8192 || cfg->num_targets > 8192)
        return fail<uavenv>(nullptr, UAVENV_EINVAL, "uavenv_create: num_uavs / num_targets above 8192 are not supported");
    if (env_id_base + (uint64_t)num_envs > 0xffffffffull)
        return fail<uavenv>(nullptr, UAVENV_EINVAL, "uavenv_create: global env ids must fit 32 bits");
    uavenv *h;
    if (int rc = capi::new_handle("uavenv_create", device, h)) return rc;
    h->cfg = *cfg; h->B = num_envs; h->seed = seed; h->env_id_base = env_id_base;
    if (int rc = create_impl(h)) return capi::abandon_handle(h, rc);
    *out = h;
    return UAVENV_OK;
}

extern "C" int uavenv_destroy(uavenv_t *h) { return capi::destroy_handle(h); }

static int launch_check(uavenv *h, const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, UAVENV_ECUDA, "%s launch failed: %s", what, cudaGetErrorString(e));
    return UAVENV_OK;
}

static int check_ready(uavenv *h, const char *what) {
    return h->ready ? UAVENV_OK : fail(h, UAVENV_ESTATE, "%s before reset()/load_scene()", what);
}

// envs first_env + i * stride, i in [0, count), must exist; 64-bit arithmetic, so that no int32 argument wraps the test
static int check_env_range(uavenv *h, int64_t first_env, int64_t count, int64_t stride, const char *what) {
    const int64_t end = first_env + (count - 1) * stride + 1;
    if (count <= 0 || first_env < 0 || end > h->B)
        return fail(h, UAVENV_EINVAL, "%s: env range [%lld,%lld) empty or outside [0,%d)", what, (long long)first_env,
                    (long long)end, h->B);
    return UAVENV_OK;
}

extern "C" int uavenv_reset(uavenv_t *h, int32_t full_reset, const uint8_t *d_env_mask, float *d_obs, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!full_reset && !h->ready)
        return fail(h, UAVENV_ESTATE, "uavenv_reset(full_reset=0) before any scene exists (reset(full) or load_scene first)");
    if (d_env_mask && !h->ready)
        return fail(h, UAVENV_ESTATE, "uavenv_reset: the first reset must cover every env (d_env_mask = NULL)");
    CU_TRY(h, cudaSetDevice(h->device));
    const int grid = std::min((h->B + 3) / 4, 148 * 16);
    reset_kernel<<<grid, kResetThreads, h->reset_smem, (cudaStream_t)stream>>>(h->P, full_reset ? 1 : 0, d_env_mask, 0,
                                                                              h->B, d_obs);
    int rc = launch_check(h, "reset_kernel");
    if (rc == UAVENV_OK) h->ready = true;
    return rc;
}

static int launch_step(uavenv_t *h, const void *d_actions, int action_bytes, float *d_obs, float *d_reward,
                       uint8_t *d_done, const uavenv_info_t *info, void *stream, bool actions_in_host_memory = false) {
    if (!h) return UAVENV_EINVAL;
    if (!d_actions || !d_obs || !d_reward || !d_done)
        return fail(h, UAVENV_EINVAL, "uavenv_step: actions/obs/reward/done must be non-NULL device pointers");
    if (int rc = check_ready(h, "uavenv_step")) return rc;
    StepIO io;
    io.actions = d_actions; io.action_bytes = action_bytes; io.obs = d_obs; io.reward = d_reward; io.done = d_done;
    // actions that live in (mapped) host memory are fetched with ONE bulk copy per CTA instead of one 32 B read per warp
    io.actions_bulk = actions_in_host_memory && (reinterpret_cast<uintptr_t>(d_actions) & 15u) == 0 ? 1 : 0;
    io.J_val = info ? info->d_J_val : nullptr;
    io.num_assigned = info ? info->d_num_assigned : nullptr;
    io.is_valid = info ? info->d_is_valid_action : nullptr;
    io.avg_p_dmg = info ? info->d_avg_p_dmg : nullptr;
    io.avg_p_final = info ? info->d_avg_p_final : nullptr;
    io.reward_f64 = info ? info->d_reward_f64 : nullptr;
    const int n_main = (h->B + kStepThreads - 1) / kStepThreads;
    step_kernel<<<h->n_service + n_main, kStepThreads, h->reset_smem, (cudaStream_t)stream>>>(h->P, io, h->n_service);
    return launch_check(h, "step_kernel");
}

extern "C" int uavenv_step(uavenv_t *h, const int64_t *d_actions, float *d_obs, float *d_reward, uint8_t *d_done,
                           const uavenv_info_t *info, void *stream) {
    return launch_step(h, d_actions, 8, d_obs, d_reward, d_done, info, stream);
}

// device alias of a pinned + mapped host allocation (cudaHostAlloc / cudaHostRegister; torch pin_memory), or NULL
static void *mapped_alias(const void *host_ptr) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host_ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return attr.type == cudaMemoryTypeHost ? attr.devicePointer : nullptr;
}

static int step_host_impl(uavenv_t *h, const void *h_actions, int action_bytes, float *h_reward, uint8_t *h_done,
                          float *d_obs, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!h_actions || !h_reward || !h_done) return fail(h, UAVENV_EINVAL, "uavenv_step_host: NULL host buffer");
    cudaStream_t s = (cudaStream_t)stream;
    CU_TRY(h, cudaSetDevice(h->device));
    // Pinned, device-mapped host buffers are used in place: the fused kernel reads the actions and writes
    // reward / done straight over PCIe (no separate copy launches).  Pageable buffers go through staging copies.
    // (the aliases are looked up on every call: a pointer VALUE can be re-used by a different allocation)
    void *zc_a = mapped_alias(h_actions), *zc_r = mapped_alias(h_reward), *zc_d = mapped_alias(h_done);
    if (zc_a && zc_r && zc_d) {
        int rc = launch_step(h, zc_a, action_bytes, d_obs ? d_obs : h->obs_buf, (float *)zc_r, (uint8_t *)zc_d, nullptr,
                             stream, true);
        if (rc != UAVENV_OK) return rc;
        CU_TRY(h, cudaStreamSynchronize(s));
        return UAVENV_OK;
    }
    CU_TRY(h, cudaMemcpyAsync(h->d_actions, h_actions, (size_t)h->B * action_bytes, cudaMemcpyHostToDevice, s));
    int rc = launch_step(h, h->d_actions, action_bytes, d_obs ? d_obs : h->obs_buf, h->d_reward, h->d_done, nullptr, stream);
    if (rc != UAVENV_OK) return rc;
    CU_TRY(h, cudaMemcpyAsync(h_reward, h->d_reward, (size_t)h->B * sizeof(float), cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaMemcpyAsync(h_done, h->d_done, (size_t)h->B, cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaStreamSynchronize(s));
    return UAVENV_OK;
}

extern "C" int uavenv_step_host(uavenv_t *h, const int64_t *h_actions, float *h_reward, uint8_t *h_done, float *d_obs,
                                void *stream) {
    return step_host_impl(h, h_actions, 8, h_reward, h_done, d_obs, stream);
}

extern "C" int uavenv_step_host_i8(uavenv_t *h, const int8_t *h_actions, float *h_reward, uint8_t *h_done, float *d_obs,
                                   void *stream) {
    return step_host_impl(h, h_actions, 1, h_reward, h_done, d_obs, stream);
}

// ---- scene injection / readback ----------------------------------------------------------------

template <typename T>
static cudaError_t stage(std::vector<void *> &tmp, const T *host, size_t n, T **dev) {
    *dev = nullptr;
    if (!host || n == 0) return cudaSuccess;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) return e;
    tmp.push_back(q);
    *dev = static_cast<T *>(q);
    return cudaMemcpy(q, host, n * sizeof(T), cudaMemcpyHostToDevice);
}

// the checks both scene loads make before touching the GPU
static int check_scene_args(uavenv *h, const uavenv_scene_t *sc, int32_t num_scenes, int32_t copies, int32_t first_env,
                            const char *what) {
    if (num_scenes <= 0 || copies <= 0)
        return fail(h, UAVENV_EINVAL, "%s: need num_scenes > 0 and copies > 0 (got %d, %d)", what, num_scenes, copies);
    if (int rc = check_env_range(h, first_env, (int64_t)num_scenes * copies, 1, what)) return rc;
    const Params &P = h->P;
    if (!sc->uav_x || !sc->uav_y || !sc->uav_vx || !sc->uav_vy || !sc->uav_load || !sc->uav_cost || !sc->tgt_x ||
        !sc->tgt_y || !sc->tgt_vx || !sc->tgt_vy || !sc->tgt_value || !sc->tgt_id ||
        (P.K1 > 0 && (!sc->nfz_x || !sc->nfz_y)) || (P.K2 > 0 && (!sc->int_x || !sc->int_y || !sc->int_vx || !sc->int_vy)))
        return fail(h, UAVENV_EINVAL, "%s: a required scene array is NULL", what);
    return UAVENV_OK;
}

// the one packing path: device SoA of num_scenes scenes -> envs [first_env, first_env + num_scenes * copies), then the
// reset of a loaded scene; enqueued on `stream`
static int load_scene_impl(uavenv *h, const uavenv_scene_t &s, int32_t num_scenes, int32_t copies, int32_t first_env,
                           float *d_obs, cudaStream_t stream) {
    const int count = num_scenes * copies;
    const int grid = std::min((count + 3) / 4, 148 * 16);
    pack_scene_kernel<<<grid, kResetThreads, 0, stream>>>(h->P, s, first_env, count, copies);
    int rc = launch_check(h, "pack_scene_kernel");
    if (rc != UAVENV_OK) return rc;
    reset_kernel<<<grid, kResetThreads, h->reset_smem, stream>>>(h->P, 2, nullptr, first_env, count,
                                                                 d_obs ? d_obs : h->obs_buf);
    rc = launch_check(h, "reset_kernel");
    if (rc == UAVENV_OK) h->ready = true;  // envs outside the range keep whatever they had (zeros until reset)
    return rc;
}

extern "C" int uavenv_load_scene(uavenv_t *h, const uavenv_scene_t *sc, int32_t first_env, int32_t count,
                                  float *d_obs) {
    if (!h || !sc) return UAVENV_EINVAL;
    if (int rc = check_scene_args(h, sc, count, 1, first_env, "uavenv_load_scene")) return rc;
    const Params &P = h->P;
    CU_TRY(h, cudaSetDevice(h->device));
    std::vector<void *> tmp;
    uavenv_scene_t s{};
    const size_t n = (size_t)count * P.N, m = (size_t)count * P.M, k1 = (size_t)count * P.K1, k2 = (size_t)count * P.K2;
    cudaError_t e = cudaSuccess;
    auto S = [&](auto host, size_t cnt, auto dev) { if (e == cudaSuccess) e = stage(tmp, host, cnt, dev); };
    S(sc->uav_x, n, &s.uav_x); S(sc->uav_y, n, &s.uav_y); S(sc->uav_vx, n, &s.uav_vx); S(sc->uav_vy, n, &s.uav_vy);
    S(sc->uav_load, n, &s.uav_load); S(sc->uav_cost, n, &s.uav_cost); S(sc->uav_type, n, &s.uav_type);
    S(sc->tgt_x, m, &s.tgt_x); S(sc->tgt_y, m, &s.tgt_y); S(sc->tgt_vx, m, &s.tgt_vx); S(sc->tgt_vy, m, &s.tgt_vy);
    S(sc->tgt_value, m, &s.tgt_value); S(sc->tgt_id, m, &s.tgt_id);
    S(sc->nfz_x, k1, &s.nfz_x); S(sc->nfz_y, k1, &s.nfz_y); S(sc->nfz_radius, k1, &s.nfz_radius);
    S(sc->int_x, k2, &s.int_x); S(sc->int_y, k2, &s.int_y); S(sc->int_vx, k2, &s.int_vx); S(sc->int_vy, k2, &s.int_vy);
    int rc = UAVENV_OK;
    if (e == cudaSuccess) {
        rc = load_scene_impl(h, s, count, 1, first_env, d_obs, nullptr);
        e = cudaDeviceSynchronize();
    }
    for (void *p : tmp) cudaFree(p);
    if (rc != UAVENV_OK) return rc;
    if (e != cudaSuccess) return fail(h, UAVENV_ECUDA, "uavenv_load_scene: %s", cudaGetErrorString(e));
    return UAVENV_OK;
}

extern "C" int uavenv_load_scene_device(uavenv_t *h, const uavenv_scene_t *d_scene, int32_t num_scenes, int32_t copies,
                                         int32_t first_env, float *d_obs, void *stream) {
    if (!h || !d_scene) return UAVENV_EINVAL;
    if (int rc = check_scene_args(h, d_scene, num_scenes, copies, first_env, "uavenv_load_scene_device")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    return load_scene_impl(h, *d_scene, num_scenes, copies, first_env, d_obs, (cudaStream_t)stream);
}

extern "C" int uavenv_group_best(uavenv_t *h, int32_t first_env, int32_t num_groups, int32_t group_size, int32_t *d_best,
                                  double *d_J_best, int32_t *d_assigned_best, int32_t *d_num_covered, double *d_J_all,
                                  void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!d_best || !d_J_best || !d_assigned_best || !d_num_covered)
        return fail(h, UAVENV_EINVAL, "uavenv_group_best: best / J_best / assigned_best / num_covered must be non-NULL");
    if (num_groups <= 0 || group_size <= 0)
        return fail(h, UAVENV_EINVAL, "uavenv_group_best: need num_groups > 0 and group_size > 0 (got %d, %d)", num_groups,
                    group_size);
    if (int rc = check_env_range(h, first_env, (int64_t)num_groups * group_size, 1, "uavenv_group_best")) return rc;
    if (h->P.auto_reset)
        return fail(h, UAVENV_ESTATE, "uavenv_group_best: the handle restarts finished envs (auto_reset = 1); final "
                    "allocations are kept with auto_reset = 0 only");
    if (int rc = check_ready(h, "uavenv_group_best")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const int grid = (num_groups + 7) / 8;                               // a warp per group, 8 per CTA
    group_best_kernel<<<grid, kGroupBestThreads, 0, (cudaStream_t)stream>>>(h->P, first_env, num_groups, group_size, d_best,
                                                                           d_J_best, d_assigned_best, d_num_covered, d_J_all);
    return launch_check(h, "group_best_kernel");
}

template <typename T>
static cudaError_t fetch(std::vector<T> &v, const T *dev, size_t n) {
    v.resize(n);
    return n ? cudaMemcpy(v.data(), dev, n * sizeof(T), cudaMemcpyDeviceToHost) : cudaSuccess;
}

// the header tiles covering envs [first, first + count): env first + i's is header_at(tiles.data(), first % 32 + i)
static cudaError_t fetch_headers(const Params &P, size_t first, size_t count, std::vector<unsigned char> &tiles) {
    return fetch(tiles, P.hdr + first / 32 * kEnvTileBytes, ((first + count + 31) / 32 - first / 32) * kEnvTileBytes);
}

// envs [first, first + count) of a double-buffered [2 slots][B][per] array, each env's `per` elements taken from the
// storage slot of its current scene (I_GEN & 1; tiles from fetch_headers)
template <typename T>
static cudaError_t fetch_current(std::vector<T> &v, const T *dev, size_t per, const Params &P,
                                 std::vector<unsigned char> &tiles, size_t first, size_t count) {
    v.resize(count * per);
    std::vector<T> s;
    for (int slot = 0; slot < 2; ++slot) {
        const cudaError_t e = fetch(s, dev + ((size_t)slot * P.B + first) * per, count * per);
        if (e != cudaSuccess) return e;
        for (size_t i = 0; i < count; ++i)
            if ((header_at(tiles.data(), (int)(first % 32 + i)).n(I_GEN) & 1) == slot)
                std::copy(s.begin() + i * per, s.begin() + (i + 1) * per, v.begin() + i * per);
    }
    return cudaSuccess;
}

extern "C" int uavenv_get_scene(uavenv_t *h, uavenv_scene_t *sc, int32_t first_env, int32_t count) {
    if (!h || !sc) return UAVENV_EINVAL;
    if (int rc = check_env_range(h, first_env, count, 1, "uavenv_get_scene")) return rc;
    const Params &P = h->P;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());
    const size_t n = (size_t)count * P.N, m = (size_t)count * P.M, k1 = (size_t)count * P.K1, k2 = (size_t)count * P.K2;
    std::vector<unsigned char> tiles;
    CU_TRY(h, fetch_headers(P, first_env, count, tiles));
    std::vector<UavRec> U; std::vector<TgtRec> T; std::vector<int32_t> ty; std::vector<double2> tv, uv;
    std::vector<NfzRec> Z; std::vector<IntRec> I;
    CU_TRY(h, fetch_current(U, P.uav, P.N, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(T, P.tgt, P.M, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(ty, P.uav_type, P.N, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(tv, P.tgt_vel, P.M, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(uv, P.uav_vel, P.N, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(Z, P.nfz, P.K1, P, tiles, first_env, count));
    CU_TRY(h, fetch_current(I, P.intc, P.K2, P, tiles, first_env, count));
    for (size_t i = 0; i < n; ++i) {
        if (sc->uav_x) sc->uav_x[i] = U[i].x;
        if (sc->uav_y) sc->uav_y[i] = U[i].y;
        if (sc->uav_vx) sc->uav_vx[i] = uv[i].x;
        if (sc->uav_vy) sc->uav_vy[i] = uv[i].y;
        if (sc->uav_load) sc->uav_load[i] = U[i].load;
        if (sc->uav_cost) sc->uav_cost[i] = U[i].cost;
        if (sc->uav_type) sc->uav_type[i] = ty[i];
    }
    for (size_t j = 0; j < m; ++j) {
        if (sc->tgt_x) sc->tgt_x[j] = T[j].x;
        if (sc->tgt_y) sc->tgt_y[j] = T[j].y;
        if (sc->tgt_vx) sc->tgt_vx[j] = tv[j].x;
        if (sc->tgt_vy) sc->tgt_vy[j] = tv[j].y;
        if (sc->tgt_value) sc->tgt_value[j] = T[j].value;
        if (sc->tgt_id) sc->tgt_id[j] = T[j].id;
    }
    for (size_t i = 0; i < k1; ++i) {
        if (sc->nfz_x) sc->nfz_x[i] = Z[i].x;
        if (sc->nfz_y) sc->nfz_y[i] = Z[i].y;
        if (sc->nfz_radius) sc->nfz_radius[i] = Z[i].radius;
    }
    for (size_t i = 0; i < k2; ++i) {
        if (sc->int_x) sc->int_x[i] = I[i].x;
        if (sc->int_y) sc->int_y[i] = I[i].y;
        if (sc->int_vx) sc->int_vx[i] = I[i].vx;
        if (sc->int_vy) sc->int_vy[i] = I[i].vy;
    }
    return UAVENV_OK;
}

extern "C" int uavenv_get_state(uavenv_t *h, uavenv_state_t *st, int32_t first_env, int32_t count) {
    if (!h || !st) return UAVENV_EINVAL;
    if (int rc = check_env_range(h, first_env, count, 1, "uavenv_get_state")) return rc;
    const Params &P = h->P;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());
    const size_t c = (size_t)count, f = (size_t)first_env;
    auto D2H = [&](void *dst, const void *src, size_t bytes) -> cudaError_t {
        return dst ? cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) : cudaSuccess;
    };
    CU_TRY(h, D2H(st->assigned_target_id, P.assigned + f * P.N, c * P.N * 4));
    std::vector<unsigned char> tiles;
    CU_TRY(h, fetch_headers(P, f, c, tiles));
    for (size_t i = 0; i < c; ++i) {
        const Hdr hv = header_at(tiles.data(), (int)(f % 32 + i));
        if (st->uav_idx) st->uav_idx[i] = hv.n(I_K);
        if (st->target_idx) st->target_idx[i] = hv.n(I_M);
        if (st->episode) st->episode[i] = hv.n(I_EPISODE);
        if (st->scene_index) st->scene_index[i] = hv.n(I_GEN) >> 1;
        if (st->finished) st->finished[i] = (uint8_t)(hv.n(I_FINISHED) != 0);
        if (st->J_val) st->J_val[i] = objective(P, hv.f(F_REV), hv.f(F_COST_SUM));
        // UAV slots at / past the decision pointer have not decided in this episode (a restart does not clear them)
        if (st->assigned_target_id)
            for (int32_t k = std::max(hv.n(I_K), 0); k < P.N; ++k) st->assigned_target_id[i * P.N + k] = -1;
    }
    if (st->lock_count || st->not_hit || st->not_hit_pure) {
        std::vector<TgtRec> T;
        CU_TRY(h, fetch_current(T, P.tgt, P.M, P, tiles, f, c));
        for (size_t e = 0; e < c; ++e) {
            const int episode = header_at(tiles.data(), (int)(f % 32 + e)).n(I_EPISODE);
            for (size_t j = e * P.M; j < (e + 1) * P.M; ++j) {
                TgtRec t = T[j];                           // as the env sees it in its current episode
                const int cnt = target_view(t, episode);
                if (st->lock_count) st->lock_count[j] = cnt;
                if (st->not_hit) st->not_hit[j] = t.nh;
                if (st->not_hit_pure) st->not_hit_pure[j] = t.nh_pure;
            }
        }
    }
    return UAVENV_OK;
}

extern "C" int uavenv_set_episode_counters(uavenv_t *h, const int32_t *h_episode, int32_t first_env, int32_t count) {
    if (!h || !h_episode) return UAVENV_EINVAL;
    if (int rc = check_env_range(h, first_env, count, 1, "uavenv_set_episode_counters")) return rc;
    for (int32_t i = 0; i < count; ++i)
        if (h_episode[i] < 1) return fail(h, UAVENV_EINVAL, "uavenv_set_episode_counters: counters are 1-based");
    const Params &P = h->P;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());
    int32_t *d_ep = nullptr;
    CU_TRY(h, cudaMalloc(&d_ep, (size_t)count * sizeof(int32_t)));
    cudaError_t e = cudaMemcpy(d_ep, h_episode, (size_t)count * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        set_episode_kernel<<<std::min((count + 7) / 8, 148 * 8), 256>>>(P, d_ep, first_env, count);
        e = cudaDeviceSynchronize();
    }
    cudaFree(d_ep);
    if (e != cudaSuccess) return fail(h, UAVENV_ECUDA, "uavenv_set_episode_counters: %s", cudaGetErrorString(e));
    return UAVENV_OK;
}

// ---- score matrix / objective check / action stream ---------------------------------------------

template <typename OutT>
static int score_matrix_impl(uavenv *h, OutT *pf, OutT *pd, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!pf && !pd) return fail(h, UAVENV_EINVAL, "uavenv_score_matrix: both outputs NULL");
    if (int rc = check_ready(h, "uavenv_score_matrix")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t warps = (size_t)h->B * ((h->P.M + 31) / 32);          // one warp per (env, 32-target chunk)
    const int grid = (int)std::min<size_t>((warps + 7) / 8, (size_t)148 * 32);
    score_matrix_kernel<OutT><<<grid, 256, 0, (cudaStream_t)stream>>>(h->P, pf, pd);
    return launch_check(h, "score_matrix_kernel");
}
extern "C" int uavenv_score_matrix(uavenv_t *h, float *pf, float *pd, void *stream) {
    return score_matrix_impl<float>(h, pf, pd, stream);
}
extern "C" int uavenv_score_matrix_f64(uavenv_t *h, double *pf, double *pd, void *stream) {
    return score_matrix_impl<double>(h, pf, pd, stream);
}

extern "C" int uavenv_recompute_objective(uavenv_t *h, double *h_max_abs_diff, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (int rc = check_ready(h, "uavenv_recompute_objective")) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaMemsetAsync(h->d_scratch, 0, sizeof(double), s));
    const int grid = std::min((h->B + 7) / 8, 148 * 8);
    recompute_kernel<<<grid, 256, 0, s>>>(h->P, 1, h->d_scratch);
    int rc = launch_check(h, "recompute_kernel");
    if (rc != UAVENV_OK) return rc;
    double v = 0.0;
    CU_TRY(h, cudaMemcpyAsync(&v, h->d_scratch, sizeof(double), cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaStreamSynchronize(s));
    if (h_max_abs_diff) *h_max_abs_diff = v;
    return UAVENV_OK;
}

extern "C" int uavenv_random_actions(uavenv_t *h, uint64_t action_seed, uint64_t step, int64_t *d_actions, void *stream) {
    if (!h || !d_actions) return UAVENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    random_actions_kernel<<<(h->B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->P, (uint32_t)action_seed,
                                                                               (uint32_t)(action_seed >> 32), step, d_actions);
    return launch_check(h, "random_actions_kernel");
}

extern "C" int uavenv_best_target_actions(uavenv_t *h, int64_t *d_cache, int64_t *d_actions, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!d_cache || !d_actions) return fail(h, UAVENV_EINVAL, "uavenv_best_target_actions: cache/actions must be non-NULL device pointers");
    if (int rc = check_ready(h, "uavenv_best_target_actions")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    best_target_kernel<<<(h->B + kBestTargetThreads - 1) / kBestTargetThreads, kBestTargetThreads, 0, (cudaStream_t)stream>>>(
        h->P, d_cache, d_actions);
    return launch_check(h, "best_target_kernel");
}

// ---- local search on allocations ----------------------------------------------------------------

static int improve_sms(const uavenv *h) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device) != cudaSuccess) return 0;
    return sms;
}

extern "C" size_t uavenv_improve_workspace_bytes(const uavenv_t *h) {
    if (!h || improve_p_in_smem(h->P.N, h->P.M)) return 0;
    return (size_t)improve_sms(h) * h->P.N * h->P.M * sizeof(double);    // one p[N][M] slice per SM
}

extern "C" int uavenv_improve_allocation(uavenv_t *h, int32_t first_env, int32_t count, int32_t env_stride,
                                         const int32_t *d_assigned_in, int32_t max_moves, int32_t *d_assigned_out,
                                         double *d_J_in, double *d_J_out, int32_t *d_num_covered, int32_t *d_moves,
                                         uint8_t *d_converged, void *d_workspace, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!d_assigned_in || !d_assigned_out || !d_J_out || !d_num_covered || !d_moves || !d_converged)
        return fail(h, UAVENV_EINVAL, "uavenv_improve_allocation: assigned_in / assigned_out / J_out / num_covered / "
                    "moves / converged must be non-NULL");
    const bool p_smem = improve_p_in_smem(h->P.N, h->P.M);
    if (!p_smem && !d_workspace)
        return fail(h, UAVENV_EINVAL, "uavenv_improve_allocation: N*M = %d needs a workspace of "
                    "uavenv_improve_workspace_bytes() bytes", h->P.N * h->P.M);
    if (count <= 0 || env_stride <= 0 || max_moves < 0)
        return fail(h, UAVENV_EINVAL, "uavenv_improve_allocation: need count > 0, env_stride > 0 and max_moves >= 0 "
                    "(got %d, %d, %d)", count, env_stride, max_moves);
    if (int rc = check_env_range(h, first_env, count, env_stride, "uavenv_improve_allocation")) return rc;
    if (int rc = check_ready(h, "uavenv_improve_allocation")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const int sms = improve_sms(h);
    if (sms <= 0) return fail(h, UAVENV_ECUDA, "uavenv_improve_allocation: no multiprocessor count for device %d", h->device);
    const size_t smem = improve_smem_bytes(h->P.N, h->P.M);
    CU_TRY(h, cudaFuncSetAttribute(improve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;                          // the workspace holds one slice per SM: one CTA per SM on that path
    if (p_smem) CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, improve_kernel, kImproveThreads, smem));
    const int grid = std::min(count, sms * std::max(per_sm, 1));
    ImproveIO io;
    io.assigned_in = d_assigned_in; io.assigned_out = d_assigned_out; io.J_in = d_J_in; io.J_out = d_J_out;
    io.num_covered = d_num_covered; io.moves = d_moves; io.converged = d_converged;
    io.workspace = p_smem ? nullptr : static_cast<double *>(d_workspace);
    io.first_env = first_env; io.count = count; io.env_stride = env_stride; io.max_moves = max_moves;
    improve_kernel<<<grid, kImproveThreads, smem, (cudaStream_t)stream>>>(h->P, io);
    return launch_check(h, "improve_kernel");
}

// ---- upper bound on the best allocation ----------------------------------------------------------------------------

extern "C" int uavenv_upper_bound(uavenv_t *h, int32_t first_env, int32_t count, int32_t env_stride, int32_t iters,
                                  double *d_bound, double *d_relaxed, int32_t *d_iters, void *d_workspace, void *stream) {
    if (!h) return UAVENV_EINVAL;
    if (!d_bound || !d_relaxed || !d_iters)
        return fail(h, UAVENV_EINVAL, "uavenv_upper_bound: bound / relaxed / iters must be non-NULL");
    const bool a_smem = improve_p_in_smem(h->P.N, h->P.M);
    if (!a_smem && !d_workspace)
        return fail(h, UAVENV_EINVAL, "uavenv_upper_bound: N*M = %d needs a workspace of "
                    "uavenv_improve_workspace_bytes() bytes", h->P.N * h->P.M);
    if (count <= 0 || env_stride <= 0 || iters < 1)
        return fail(h, UAVENV_EINVAL, "uavenv_upper_bound: need count > 0, env_stride > 0 and iters >= 1 (got %d, %d, %d)",
                    count, env_stride, iters);
    if (int rc = check_env_range(h, first_env, count, env_stride, "uavenv_upper_bound")) return rc;
    if (int rc = check_ready(h, "uavenv_upper_bound")) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const int sms = improve_sms(h);
    if (sms <= 0) return fail(h, UAVENV_ECUDA, "uavenv_upper_bound: no multiprocessor count for device %d", h->device);
    const size_t smem = bound_smem_bytes(h->P.N, h->P.M);
    CU_TRY(h, cudaFuncSetAttribute(bound_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;                          // the workspace holds one slice per SM: one CTA per SM on that path
    if (a_smem) CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bound_kernel, kBoundThreads, smem));
    const int grid = std::min(count, sms * std::max(per_sm, 1));
    BoundIO io;
    io.bound = d_bound; io.relaxed = d_relaxed; io.iters = d_iters;
    io.workspace = a_smem ? nullptr : static_cast<double *>(d_workspace);
    io.first_env = first_env; io.count = count; io.env_stride = env_stride; io.max_iters = iters;
    bound_kernel<<<grid, kBoundThreads, smem, (cudaStream_t)stream>>>(h->P, io);
    return launch_check(h, "bound_kernel");
}
