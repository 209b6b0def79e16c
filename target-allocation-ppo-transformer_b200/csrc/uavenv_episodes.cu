// uavenv_episodes.cu - per-episode records of an evaluation run (sm_100a).
//
// One launch per env step folds the step's outputs into per-env running sums and writes a record when an episode ends.
// The same statistics as torch ops would take about a dozen elementwise launches per step, against an env step of
// 12-20 us.  Records land at [env, episode index]: the layout is in env order and does not depend on scheduling.
#include "uavenv_b200.h"

#include <cstdint>
#include <cuda_runtime.h>

#include "handle.cuh"

static_assert(sizeof(uavenv_episode_t) == 40, "uavenv_episode_t layout");

namespace {

struct InfoIn {
    const double *reward;
    const float *J_val, *avg_p_dmg, *avg_p_final;
    const int32_t *num_assigned;
    const int8_t *is_valid;
};

__global__ void __launch_bounds__(256) episode_accumulate_kernel(int B, const int64_t *__restrict__ actions,
                                                                 const uint8_t *__restrict__ done, InfoIn in, int quota,
                                                                 uavenv_episode_acc_t acc, uavenv_episode_t *__restrict__ records) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int k = acc.d_episodes[b];
    if (k >= quota) return;                         // quota reached: the env's later episodes are not recorded
    const double ret = acc.d_ret[b] + in.reward[b];
    const int length = acc.d_length[b] + 1;
    const int assigns = acc.d_assigns[b] + (actions[b] == 1 ? 1 : 0);
    const int valid = acc.d_valid[b] + (in.is_valid[b] == 1 ? 1 : 0);
    if (done[b]) {
        uavenv_episode_t r;
        r.ret = ret;
        r.J_val = in.J_val[b]; r.avg_p_dmg = in.avg_p_dmg[b]; r.avg_p_final = in.avg_p_final[b];
        r.length = length; r.num_assigned = in.num_assigned[b]; r.assigns = assigns; r.valid = valid;
        records[(size_t)b * quota + k] = r;
        acc.d_episodes[b] = k + 1;
        if (k + 1 == quota) atomicAdd(acc.d_envs_complete, 1);
        acc.d_ret[b] = 0.0; acc.d_length[b] = 0; acc.d_assigns[b] = 0; acc.d_valid[b] = 0;
    } else {
        acc.d_ret[b] = ret; acc.d_length[b] = length; acc.d_assigns[b] = assigns; acc.d_valid[b] = valid;
    }
}

}  // namespace

extern "C" int uavenv_episode_accumulate(int32_t B, const int64_t *d_actions, const uint8_t *d_done, const uavenv_info_t *info,
                                         int32_t episodes_per_env, const uavenv_episode_acc_t *acc, uavenv_episode_t *d_records,
                                         int32_t device, void *stream) {
    if (B <= 0 || episodes_per_env <= 0)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: need B > 0 and episodes_per_env > 0 (got %d, %d)", __func__, B,
                                  episodes_per_env);
    if (!d_actions || !d_done || !info || !acc || !d_records)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: actions / done / info / acc / records must be non-NULL", __func__);
    if (!info->d_reward_f64 || !info->d_J_val || !info->d_avg_p_dmg || !info->d_avg_p_final || !info->d_num_assigned ||
        !info->d_is_valid_action)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: every array of info must be non-NULL", __func__);
    if (!acc->d_ret || !acc->d_length || !acc->d_assigns || !acc->d_valid || !acc->d_episodes || !acc->d_envs_complete)
        return capi::fail<uavenv>(nullptr, UAVENV_EINVAL, "%s: every array of acc must be non-NULL", __func__);
    if (int rc = capi::check_cuda<uavenv>(cudaSetDevice(device), __func__, "cudaSetDevice")) return rc;
    const InfoIn in = {info->d_reward_f64, info->d_J_val, info->d_avg_p_dmg, info->d_avg_p_final, info->d_num_assigned,
                       info->d_is_valid_action};
    episode_accumulate_kernel<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(B, d_actions, d_done, in, episodes_per_env, *acc,
                                                                                  d_records);
    return capi::check_cuda<uavenv>(cudaGetLastError(), __func__, "episode_accumulate_kernel launch");
}
