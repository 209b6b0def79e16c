"""Batched evaluation of a policy checkpoint: per-episode results over a fixed set of held-out scenes.

    res = ub.evaluate("runs/final_model.pth", num_envs=16384)
    res["summary"]["J_mean"], res["summary"]["J_sem"], res["J"]            # [num_envs * world, episodes_per_env]

Every step is three launches on the current stream: the actor-only tcgen05 forward (greedy or sampled,
include/uavpolicy_eval_b200.h), the fused env step, and uavenv_episode_accumulate, which folds the step into per-env
sums and writes a record when an episode ends.  The only host synchronisation is a poll of the completed-env counter
every POLL_STEPS steps.

ub.evaluate_baseline("best_target" | "random", ...) plays the same scenes with a rule in place of the network (the
best-target heuristic's kernel, or the Bernoulli(1/2) action stream): reference points for a checkpoint's numbers.

Scenes: the env runs with RESET_EPISODES = 1, so every episode is a fresh scene keyed (seed, global env id, scene
index).  The default seed is not the training seed, so the evaluation plays scenes the training envs do not; two
checkpoints evaluated with the same seed play the same scenes, and their records can be compared episode by episode.
"""
import copy
import ctypes as C
import os
import time
from collections.abc import Mapping

import numpy as np
import torch

from . import _capi, parallel
from .configs.config import cfg as _global_cfg

DEFAULT_SEED = 20240917          # held out: differs from the training default cfg.SEED = 42
POLL_STEPS = 32
EPISODE_KEYS = ("return", "J", "num_assigned", "coverage", "length", "assigns", "valid", "avg_p_dmg", "avg_p_final")
_RECORD_DTYPE = np.dtype(_capi.EPISODE_FIELDS + [("_pad", "<i4")])


def load_checkpoint(policy, cfg=None):
    """A TransformerActorCritic from a module (returned as it is), a state_dict, or the path of a checkpoint written by
    train() or by the reference (`policy.state_dict()`, loaded with weights_only=True).  Raises ValueError on a
    state_dict whose keys or shapes are not those of the network."""
    from .networks.transformer_net import TransformerActorCritic
    if isinstance(policy, TransformerActorCritic):
        return policy
    if isinstance(policy, torch.nn.Module):
        raise TypeError("expected a TransformerActorCritic, got %s" % type(policy).__name__)
    if isinstance(policy, (str, os.PathLike)):
        policy = torch.load(os.fspath(policy), map_location="cpu", weights_only=True)
    if not isinstance(policy, Mapping):
        raise TypeError("policy must be a TransformerActorCritic, a state_dict or a checkpoint path")
    net = TransformerActorCritic(cfg)
    try:
        net.load_state_dict(policy, strict=True)
    except RuntimeError as exc:
        raise ValueError("not a TransformerActorCritic state_dict: %s" % exc) from exc
    return net


class EpisodeRecorder:
    """Per-episode records of a UAVEnvBatched (built with_info=True), one uavenv_episode_accumulate launch per step.

        rec = EpisodeRecorder(env, episodes_per_env)
        obs, _, _, _ = env.step(actions); rec.record(actions)        # after every step, on the same stream
        rec.complete() == env.num_envs;  rec.records() -> dict of numpy [num_envs, episodes_per_env]

    Records are kept on the device in env order, at [env, episode index]; an env's episodes past the quota are not
    recorded."""

    def __init__(self, env, episodes_per_env):
        if env._info_c is None:
            raise ValueError("the env must be built with with_info=True")
        self.env, self.quota, self.num_envs = env, int(episodes_per_env), env.num_envs
        if self.quota <= 0:
            raise ValueError("episodes_per_env must be positive")
        B, dev = self.num_envs, env.device
        self._lib = _capi.load()
        self._ret = torch.zeros(B, dtype=torch.float64, device=dev)
        self._ints = torch.zeros(4, B, dtype=torch.int32, device=dev)       # length, assigns, valid, episodes
        self._complete = torch.zeros(1, dtype=torch.int32, device=dev)
        self.raw = torch.zeros(B * self.quota * _capi.EPISODE_BYTES, dtype=torch.uint8, device=dev)
        self._acc = _capi.UavenvEpisodeAcc(self._ret.data_ptr(), *(t.data_ptr() for t in self._ints),
                                           self._complete.data_ptr())

    def record(self, actions):
        """Fold the env's last step, taken with `actions` (int64 [B] on the device), into the records."""
        _capi.check(self._lib.uavenv_episode_accumulate(
            self.num_envs, C.c_void_p(actions.data_ptr()), C.c_void_p(self.env._done_u8.data_ptr()), C.byref(self.env._info_c),
            self.quota, C.byref(self._acc), C.c_void_p(self.raw.data_ptr()), self.env.device.index, self.env._stream()))

    def complete(self):
        """Envs that have recorded all their episodes (synchronises)."""
        return int(self._complete.item())

    def records(self, raw=None):
        """Per-episode numpy arrays [envs, episodes_per_env] (keys EPISODE_KEYS) of `raw` (default: this recorder's)."""
        return records_from_raw(self.raw if raw is None else raw, self.quota, self.env.M)


def records_from_raw(raw, quota, num_targets):
    host = raw.cpu().numpy() if isinstance(raw, torch.Tensor) else np.asarray(raw, np.uint8)
    rec = host.view(_RECORD_DTYPE).reshape(-1, quota)
    return {"return": rec["ret"].copy(), "J": rec["J_val"].copy(), "num_assigned": rec["num_assigned"].copy(),
            "coverage": rec["num_assigned"] / float(num_targets), "length": rec["length"].copy(),
            "assigns": rec["assigns"].copy(), "valid": rec["valid"].copy(), "avg_p_dmg": rec["avg_p_dmg"].copy(),
            "avg_p_final": rec["avg_p_final"].copy()}


def _world():
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        return torch.distributed.get_rank(), torch.distributed.get_world_size()
    return 0, 1


def _stats(x):
    """(mean, sample std, standard error of the mean) of all values of x."""
    x = np.asarray(x, np.float64).reshape(-1)
    std = float(x.std(ddof=1)) if x.size > 1 else 0.0
    return float(x.mean()), std, std / np.sqrt(x.size)


def _summary(res, env_steps, wall):
    s = {}
    for key in ("return", "J", "coverage"):
        s[key + "_mean"], s[key + "_std"], s[key + "_sem"] = _stats(res[key])
    s["valid_assign_rate"] = float(res["valid"].sum()) / max(int(res["assigns"].sum()), 1)
    s["length_mean"] = float(res["length"].mean())
    s["episodes"] = int(res["length"].size)
    s["env_steps"] = int(env_steps)
    s["wall_s"] = float(wall)
    s["episodes_per_s"] = s["episodes"] / wall
    s["env_steps_per_s"] = env_steps / wall
    return s


def _eval_setup(num_envs, episodes_per_env, config, device, env_id_base):
    """(device, num_envs, quota, cfg, rank's first global env id, world size) of an evaluation run, arguments checked."""
    num_envs, quota = int(num_envs), int(episodes_per_env)
    if num_envs <= 0 or quota <= 0:
        raise ValueError("num_envs and episodes_per_env must be positive")
    device = _capi.cuda_device(device, "evaluate")
    cfg = (config if config is not None else _global_cfg).copy(RESET_EPISODES=1)   # a fresh scene every episode
    rank, world = _world()
    base = rank * num_envs if env_id_base is None else int(env_id_base)
    return device, num_envs, quota, cfg, base, world


def _play(env, quota, act, world):
    """Play `quota` episodes in every env of `env` with actions act(obs, step) (int64 [B] on the device); returns the
    records of all ranks in global env order, the steps taken and the wall seconds."""
    num_envs, device = env.num_envs, env.device
    rec = EpisodeRecorder(env, quota)
    max_steps = quota * env.N * env.M        # every step moves the (UAV, target) pointer: an episode ends within N * M
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    obs = env.reset(full_reset=True)
    steps = 0
    while steps < max_steps:
        action = act(obs, steps)
        obs, _, _, _ = env.step(action)
        rec.record(action)
        steps += 1
        if steps % POLL_STEPS == 0 and rec.complete() == num_envs:
            break
    # summed over the ranks, so that all of them raise together instead of some waiting in the all-gather
    missing = int(parallel.reduce_scalar(num_envs - rec.complete(), "sum", device))
    if missing:
        raise RuntimeError("%d of %d envs did not finish %d episodes within %d steps" % (
            missing, num_envs * world, quota, max_steps))
    raw = rec.raw
    if world > 1:
        parts = [torch.empty_like(raw) for _ in range(world)]
        torch.distributed.all_gather(parts, raw)
        raw = torch.cat(parts)
    res = records_from_raw(raw, quota, env.M)
    return res, steps, time.perf_counter() - t0


def evaluate(policy, num_envs=4096, episodes_per_env=1, greedy=True, seed=DEFAULT_SEED, config=None, device=None,
             env_id_base=None):
    """Play `episodes_per_env` episodes in each of `num_envs` envs (per rank) and return per-episode numpy arrays
    [num_envs * world, episodes_per_env] in global env order (keys EPISODE_KEYS; coverage = num_assigned / M) and a
    `summary` dict (mean / std / standard error of return, J and coverage; valid-assign rate = sum(valid) /
    sum(assigns); mean length; episode count; env-steps; wall seconds; episodes and env-steps per second).

    policy: a TransformerActorCritic (left unchanged, on its own device), its state_dict, or a checkpoint path.  greedy: argmax actions; otherwise actions
    sampled keyed (seed, step, global env id).  env_id_base: global id of this rank's first env (None: rank *
    num_envs, as train() shards).  Under an initialised process group every rank calls this with the same num_envs and
    episodes_per_env, and the records of all ranks are all-gathered."""
    from .envs.uav_env import UAVEnvBatched
    from .networks.fused_forward import FusedPolicyForward
    device, num_envs, quota, cfg, base, world = _eval_setup(num_envs, episodes_per_env, config, device, env_id_base)
    net = load_checkpoint(policy, cfg)
    if net is policy:                            # the caller's module stays where it is: evaluate a copy on the device
        net = copy.deepcopy(net)
    net = net.to(device)
    env = fused = None
    try:
        env = UAVEnvBatched(num_envs, device=device, seed=seed, config=cfg, env_id_base=base)
        fused = FusedPolicyForward(num_envs, device, seed=seed, env_id_base=base)
        fused.sync(net)
        res, steps, wall = _play(env, quota, lambda obs, step: fused.act(obs, step, greedy=greedy)[0], world)
    finally:
        if fused is not None:
            fused.close()
        if env is not None:
            env.close()
    res["summary"] = _summary(res, parallel.reduce_scalar(steps * num_envs, "sum", device), wall)
    return res


BASELINES = ("best_target", "random")


def evaluate_baseline(kind, num_envs=4096, episodes_per_env=1, seed=DEFAULT_SEED, config=None, device=None,
                      env_id_base=None):
    """Reference points for evaluate(): the same scenes played by a rule instead of a network.  Returns the same dict as
    evaluate() (records in global env order, all-gathered under a process group, and `summary`); with an equal seed its
    records pair episode by episode with those of evaluate(checkpoint).

    kind "best_target": each UAV Assigns the target whose tentative assignment gives the highest paper reward (Eq.19),
    if that reward is not below the current one (UAVEnvBatched.best_target_actions, one kernel per step).
    kind "random": Bernoulli(1/2) actions keyed (seed + 1, step, global env id) - UAVEnvBatched.random_actions with
    action_seed = seed + 1, so the action stream is not drawn with the scenes' key."""
    from .envs.uav_env import UAVEnvBatched
    if kind not in BASELINES:
        raise ValueError("kind must be one of %s, got %r" % (", ".join(BASELINES), kind))
    device, num_envs, quota, cfg, base, world = _eval_setup(num_envs, episodes_per_env, config, device, env_id_base)
    env = None
    try:
        env = UAVEnvBatched(num_envs, device=device, seed=seed, config=cfg, env_id_base=base)

        def act(obs, step):
            return env.best_target_actions() if kind == "best_target" else env.random_actions(step, action_seed=seed + 1)

        res, steps, wall = _play(env, quota, act, world)
    finally:
        if env is not None:
            env.close()
    res["summary"] = _summary(res, parallel.reduce_scalar(steps * num_envs, "sum", device), wall)
    return res
