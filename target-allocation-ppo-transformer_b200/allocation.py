"""Target allocation for given scenes with a trained policy: best-of-K sampled episodes per scene.

    res = ub.allocate("runs/final_model.pth", scenes=my_scenes, samples=16)
    res["assigned_target_id"]       # int32 [S, N]: Target.id each UAV of scene s is sent to in its best episode, -1 = none
    res["J"], res["J_samples"]      # f64 [S] the best episode's J,  [S, K] every episode's J

    pol = ub.improve_allocation(my_scenes, res["assigned_target_id"])   # local search from any allocation
    pol["assigned_target_id"], pol["J"], pol["J_before"]

    ub_ = ub.upper_bound(my_scenes)     # certified: no allocation of scene s beats ub_["bound"][s]
    gap = ub_["bound"] - pol["J"]       # how far an allocation can be from the optimum, at most

Each scene is played K times in K envs of one UAVEnvBatched built with auto_reset=False, so a finished episode keeps its
final allocation on the device.  Per chunk of scenes: uavenv_load_scene_device puts every scene into its K envs (no host
round trip), the loop act -> step runs until all of the chunk's envs are done (a poll every POLL_STEPS steps), and
uavenv_group_best picks each scene's best episode and reads out its allocation.  Only the results cross to the host.

Sampling: the actions of sample c of scene s are drawn with the key (seed, step, s*K + c) - the fused forward's
env_id_base is set to each chunk's first sample id - so the result does not depend on how the scenes are chunked.

Local search (improve_allocation, allocate(improve=True)): uavenv_improve_allocation moves one UAV or swaps two while J
rises (steepest ascent; the rule is in include/uavenv_b200.h), on the device, a scene per CTA.  allocate runs it on the
first env of each scene's group right after group_best - every member holds the same scene - so no second scene load
is needed.

Upper bound (upper_bound, allocate(bound=True)): uavenv_upper_bound runs Frank-Wolfe on the concave relaxation of J and
returns min_t of its duality bound plus a stated margin, a value no allocation of the scene exceeds (the rule and its
proof are in include/uavenv_b200.h).  allocate runs it on the same env as the local search.
"""
import copy
import time

import torch

from . import _capi
from .configs.config import cfg as _global_cfg
from .evaluation import DEFAULT_SEED, POLL_STEPS, _eval_setup, _stats, load_checkpoint


def _scene_count(scenes, N):
    if not hasattr(scenes, "get") or scenes.get("uav_x") is None:
        raise ValueError("scenes must be a get_scene()-style dict of arrays (uav_x [S, N], ...)")
    n = torch.as_tensor(scenes["uav_x"]).numel()
    if n == 0 or n % N:
        raise ValueError("scenes['uav_x'] has %d elements, not a positive multiple of NUM_UAVS = %d" % (n, N))
    return n // N


def _device_scenes(scenes, S, device):
    """The scene arrays on the device as [S, ...] tensors (one move; chunks are row slices of them)."""
    fields = {name for name, _, _ in _capi.SCENE_FIELDS}
    return {k: torch.as_tensor(v).to(device).reshape(S, -1) for k, v in scenes.items()
            if k in fields and v is not None and torch.as_tensor(v).numel() > 0}


def _max_moves(max_moves):
    if max_moves is not None and int(max_moves) < 0:
        raise ValueError("max_moves must be >= 0 (or None: 16 * NUM_UAVS)")
    return None if max_moves is None else int(max_moves)


def allocate(policy, scenes=None, num_scenes=None, samples=1, greedy=None, seed=DEFAULT_SEED, config=None, device=None,
             max_envs=65536, improve=False, bound=False):
    """Allocate the targets of S scenes: play each scene `samples` (K) times with the policy and return the best
    episode's allocation per scene.

    policy: a TransformerActorCritic, its state_dict or a checkpoint path (see load_checkpoint), or "best_target" (the
    best-target heuristic, deterministic: K must be 1).  scenes: a get_scene()-style dict of arrays [S, N] / [S, M] /
    [S, K1] / [S, K2] (numpy or torch, host or device; list order, targets after the shuffle), or None with num_scenes:
    the first-episode scenes of evaluate(..., seed=seed), scene s keyed (seed, global env id s).  greedy: argmax actions
    (default when K == 1); otherwise actions sampled keyed (seed, step, s*K + c).  config: sizes and constants (default
    the global cfg).  max_envs: the most envs played at once; scenes go through in chunks of max_envs // K.
    improve: polish each scene's best allocation with the local search of improve_allocation (cap 16 * N moves).
    bound: also compute each scene's certified upper bound on J (upper_bound, 256 iterations).

    Returns numpy arrays: "assigned_target_id" int32 [S, N], "J" f64 [S] (the value get_state reports as J_val),
    "num_covered" int32 [S] (N0), "best_sample" int32 [S] (the first sample with the highest J), "J_samples" f64 [S, K];
    and "summary": J mean / std / standard error over the scenes, mean J of all samples, K, scenes, env-steps (steps
    times envs played), wall seconds, scenes/s and env-steps/s.  With improve=True, "assigned_target_id", "J" and
    "num_covered" are those of the improved allocation, and "J_before_improve" f64 [S] (the best episode's J), "moves"
    int32 [S] and "converged" bool [S] (False: the move cap stopped the search) are added; "best_sample" and "J_samples"
    stay those of the episodes.  With bound=True, "J_bound" f64 [S] (upper_bound's "bound") is added, and the summary
    gains "J_bound_mean" and "gap_mean" (the mean of J_bound - J)."""
    K = int(samples)
    if K <= 0:
        raise ValueError("samples must be positive")
    if greedy is None:
        greedy = K == 1
    if greedy and K > 1:
        raise ValueError("greedy=True with samples > 1: every sample of a scene would be the same episode")
    if isinstance(policy, str) and policy == "best_target" and K > 1:
        raise ValueError("the best_target heuristic is deterministic: samples must be 1")
    max_envs = int(max_envs)
    if K > max_envs:
        raise ValueError("samples (%d) > max_envs (%d): one scene's samples must fit one chunk" % (K, max_envs))
    if (scenes is None) == (num_scenes is None):
        raise ValueError("give exactly one of scenes and num_scenes")
    N = int((config if config is not None else _global_cfg).NUM_UAVS)
    S = _scene_count(scenes, N) if scenes is not None else int(num_scenes)
    if S <= 0:
        raise ValueError("num_scenes must be positive")
    device, S, _, cfg, _, _ = _eval_setup(S, 1, config, device, 0)

    from .envs.uav_env import UAVEnvBatched
    from .networks.fused_forward import FusedPolicyForward
    heuristic = isinstance(policy, str) and policy == "best_target"
    net = None
    if not heuristic:
        net = load_checkpoint(policy, cfg)
        if net is policy:                        # the caller's module stays where it is
            net = copy.deepcopy(net)
        net = net.to(device)
    per = min(max_envs // K, S)                  # scenes per chunk
    E = per * K
    dev_scenes = None
    if scenes is not None:                       # one move to the device; chunks are row slices of it
        dev_scenes = _device_scenes(scenes, S, device)
    env = fused = None
    parts = []
    env_steps = 0
    try:
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        env = UAVEnvBatched(E, device=device, seed=seed, config=cfg, auto_reset=False)
        if heuristic:
            def act(obs, step):
                return env.best_target_actions()
        else:
            fused = FusedPolicyForward(E, device, seed=seed)
            fused.sync(net)

            def act(obs, step):
                return fused.act(obs, step, greedy=greedy)[0]
        limit = env.N * env.M                    # every step moves the (UAV, target) pointer: an episode ends within N * M
        for c0 in range(0, S, per):
            n = min(per, S - c0)
            if dev_scenes is not None:
                chunk = {k: v[c0:c0 + n] for k, v in dev_scenes.items()}
            else:
                chunk = _generated_scenes(n, c0, seed, cfg, device)
            env.load_scene_device(chunk, copies=K, first_env=0)
            obs = env.obs
            if fused is not None:
                fused.env_id_base = c0 * K       # the sample key (seed, step, global sample id)
            done = env.done[:n * K]              # (envs past n*K hold finished episodes of the previous chunk: inert)
            steps = 0
            while steps < limit:
                obs, _, _, _ = env.step(act(obs, steps))
                steps += 1
                if steps % POLL_STEPS == 0 and bool(done.all()):
                    break
            if not bool(done.all()):
                raise RuntimeError("%d of %d envs did not finish their episode within %d steps" % (
                    int((~done).sum()), n * K, limit))
            env_steps += steps * E
            part = env.group_best(K, 0, n)
            if improve:                          # on env g*K of each group: the scene, bit for bit, of every member
                pol = env.improve_allocation(part["assigned_target_id"], first_env=0, env_stride=K)
                part["J_before_improve"] = part["J"]
                for k in ("assigned_target_id", "J", "num_covered", "moves", "converged"):
                    part[k] = pol[k]
            if bound:
                part["J_bound"] = env.upper_bound(first_env=0, count=n, env_stride=K)["bound"]
            parts.append(part)
        res = {k: torch.cat([p[k] for p in parts]).cpu().numpy() for k in parts[0]}
        wall = time.perf_counter() - t0
    finally:
        if fused is not None:
            fused.close()
        if env is not None:
            env.close()
    out = {"assigned_target_id": res["assigned_target_id"], "J": res["J"], "num_covered": res["num_covered"],
           "best_sample": res["best"], "J_samples": res["J_all"]}
    if improve:
        for k in ("J_before_improve", "moves", "converged"):
            out[k] = res[k]
    if bound:
        out["J_bound"] = res["J_bound"]
    s = {}
    s["J_mean"], s["J_std"], s["J_sem"] = _stats(out["J"])
    s["J_samples_mean"] = float(out["J_samples"].mean())
    if improve:
        s["J_before_improve_mean"] = float(out["J_before_improve"].mean())
        s["moves_mean"] = float(out["moves"].mean())
    if bound:
        s["J_bound_mean"] = float(out["J_bound"].mean())
        s["gap_mean"] = float((out["J_bound"] - out["J"]).mean())
    s["samples"], s["scenes"], s["env_steps"], s["wall_s"] = K, S, int(env_steps), float(wall)
    s["scenes_per_s"], s["env_steps_per_s"] = S / wall, env_steps / wall
    out["summary"] = s
    return out


def improve_allocation(scenes, assigned_target_id, max_moves=None, config=None, device=None, max_envs=65536):
    """Polish given allocations of S scenes to a local optimum of J: steepest ascent over single-UAV moves (to another
    target or to none) and swaps of two UAVs' targets, one applied per round, until no candidate raises J by more than
    1e-12 * max(1, |J|) or max_moves moves have been applied (the exact rule is in include/uavenv_b200.h).

    scenes: a get_scene()-style dict of arrays (as allocate takes them).  assigned_target_id: int [S, N], the Target.id
    each UAV is sent to (-1 = none): a user's allocation, the reference's, or allocate's.  max_moves: cap on applied
    moves per scene (None: 16 * N).  config: sizes and omega (default the global cfg).  max_envs: scenes per launch.

    Returns numpy arrays: "assigned_target_id" int32 [S, N], "J" f64 [S] after and "J_before" f64 [S] before the search,
    "num_covered" int32 [S] (N0 after), "moves" int32 [S] (moves applied), "converged" bool [S] (True: the result is a
    local optimum; False: the cap was reached first); and "summary": mean J before and after, mean moves, converged
    fraction, scenes, wall seconds and scenes/s.  A row holding an id that is not a Target.id of its scene comes back
    as a row of -1 with J NaN, num_covered -1 and moves -1."""
    max_moves = _max_moves(max_moves)
    max_envs = int(max_envs)
    if max_envs <= 0:
        raise ValueError("max_envs must be positive")
    N = int((config if config is not None else _global_cfg).NUM_UAVS)
    S = _scene_count(scenes, N)
    asg = torch.as_tensor(assigned_target_id)
    if asg.dtype.is_floating_point or asg.dtype == torch.bool or asg.dtype.is_complex:
        raise ValueError("assigned_target_id must be an integer array of Target.ids")
    if asg.numel() != S * N:
        raise ValueError("assigned_target_id has %d elements, scenes hold %d x NUM_UAVS = %d" % (asg.numel(), S, S * N))
    device, S, _, cfg, _, _ = _eval_setup(S, 1, config, device, 0)
    from .envs.uav_env import UAVEnvBatched
    dev_scenes = _device_scenes(scenes, S, device)
    asg = asg.to(device=device, dtype=torch.int32).reshape(S, N)
    per = min(max_envs, S)
    env = None
    parts = []
    try:
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        env = UAVEnvBatched(per, device=device, seed=0, config=cfg, auto_reset=False, with_info=False)
        for c0 in range(0, S, per):
            n = min(per, S - c0)
            env.load_scene_device({k: v[c0:c0 + n] for k, v in dev_scenes.items()}, copies=1, first_env=0)
            parts.append(env.improve_allocation(asg[c0:c0 + n], first_env=0, env_stride=1, max_moves=max_moves))
        res = {k: torch.cat([p[k] for p in parts]).cpu().numpy() for k in parts[0]}
        wall = time.perf_counter() - t0
    finally:
        if env is not None:
            env.close()
    ok = res["moves"] >= 0                       # rows with valid ids (the means skip the flagged ones)
    mean = (lambda x: float(x[ok].mean())) if ok.any() else (lambda x: float("nan"))
    res["summary"] = {"J_before_mean": mean(res["J_before"]), "J_mean": mean(res["J"]), "moves_mean": mean(res["moves"]),
                      "converged_frac": float(res["converged"].mean()), "scenes": S, "invalid_rows": int((~ok).sum()),
                      "wall_s": float(wall), "scenes_per_s": S / wall}
    return res


def upper_bound(scenes, iters=256, config=None, device=None, max_envs=65536):
    """Certified upper bound on the best J of each of S scenes: no allocation of scene s has J above "bound"[s], so
    bound - J is at most how far an allocation's J is from the optimum.  Frank-Wolfe on the concave relaxation of J for
    at most `iters` iterations (fewer when the relaxation is solved first); the rule, and why the bound holds whatever
    the iteration does, are in include/uavenv_b200.h (uavenv_upper_bound).

    scenes: a get_scene()-style dict of arrays (as allocate takes them).  iters: iteration cap (>= 1).  config: sizes
    and omega (default the global cfg).  max_envs: scenes per launch.

    Returns numpy arrays: "bound" f64 [S], "relaxed" f64 [S] (the relaxation's value at the last iterate: bound -
    relaxed shows whether more iterations would tighten the bound), "iters" int32 [S] (iterations run); and "summary":
    mean bound, mean relaxed value, mean iterations, scenes, wall seconds and scenes/s."""
    iters = int(iters)
    if iters < 1:
        raise ValueError("iters must be >= 1")
    max_envs = int(max_envs)
    if max_envs <= 0:
        raise ValueError("max_envs must be positive")
    N = int((config if config is not None else _global_cfg).NUM_UAVS)
    S = _scene_count(scenes, N)
    device, S, _, cfg, _, _ = _eval_setup(S, 1, config, device, 0)
    from .envs.uav_env import UAVEnvBatched
    dev_scenes = _device_scenes(scenes, S, device)
    per = min(max_envs, S)
    env = None
    parts = []
    try:
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        env = UAVEnvBatched(per, device=device, seed=0, config=cfg, auto_reset=False, with_info=False)
        for c0 in range(0, S, per):
            n = min(per, S - c0)
            env.load_scene_device({k: v[c0:c0 + n] for k, v in dev_scenes.items()}, copies=1, first_env=0)
            parts.append(env.upper_bound(first_env=0, count=n, iters=iters))
        res = {k: torch.cat([p[k] for p in parts]).cpu().numpy() for k in parts[0]}
        wall = time.perf_counter() - t0
    finally:
        if env is not None:
            env.close()
    res["summary"] = {"bound_mean": float(res["bound"].mean()), "relaxed_mean": float(res["relaxed"].mean()),
                      "iters_mean": float(res["iters"].mean()), "scenes": S, "wall_s": float(wall),
                      "scenes_per_s": S / wall}
    return res


def _generated_scenes(n, first, seed, cfg, device):
    """The first-episode scenes of evaluate(..., seed) for global env ids [first, first + n): a full reset of envs keyed
    (seed, global env id) (cfg carries RESET_EPISODES = 1, as evaluate's)."""
    from .envs.uav_env import UAVEnvBatched
    gen = UAVEnvBatched(n, device=device, seed=seed, config=cfg, auto_reset=False, env_id_base=first, with_info=False)
    try:
        gen.reset(full_reset=True)
        return gen.get_scene()
    finally:
        gen.close()
