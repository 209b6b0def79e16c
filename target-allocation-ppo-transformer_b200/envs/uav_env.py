"""Host-side mirror of the reference environment (envs/uav_env.py) over the sm_100a C ABI.

`UAVEnvBatched` is the batched drop-in for the rollout path: the same reset/step contract
(envs/uav_env.py:42,295), the same [5,14] observation window and {0,1} actions, for B independent
envs resident in HBM, one fused kernel launch per step.  `UAVEnv` is the B=1 wrapper with the
reference's exact single-env signatures (numpy window, Python scalars, info dict).

PyTorch is used for device memory and streams only; every computation happens in
lib/libuavenv_b200.so.  There is no CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from .. import _capi
from ..configs.config import Config, cfg as _global_cfg
from .entities import build_entities

_NP = {"f8": np.float64, "i4": np.int32, "u1": np.uint8}
_TORCH = {"f8": torch.float64, "i4": torch.int32}


class _Discrete:           # stand-in for gym.spaces.Discrete (envs/uav_env.py:18); gym is not a dependency
    def __init__(self, n):
        self.n = n
        self.shape = ()
        self.dtype = np.int64

    def sample(self):
        return int(np.random.randint(self.n))

    def contains(self, x):
        return 0 <= int(x) < self.n


class _Box:                # stand-in for gym.spaces.Box (envs/uav_env.py:21-24)
    def __init__(self, shape):
        self.low, self.high, self.shape, self.dtype = -np.inf, np.inf, tuple(shape), np.float32


class UAVEnvBatched(_capi.Handle):
    """B independent UAV->target allocation envs on one B200.

    reset(full_reset=True) -> obs[B,5,14] f32 (CUDA)
    step(actions[B] int64) -> (obs[B,5,14], reward[B] f32, done[B] bool, info dict of [B] tensors)

    The returned tensors are owned by the env and overwritten by the next call (no allocation on the
    step path); clone what must outlive a step.  With auto_reset (default) a finished env restarts
    inside the same launch following main_train.py:79 (new scene every cfg.RESET_EPISODES episodes,
    counter-based RNG keyed on (seed, env_id_base + b, scene index)), and `obs` of a finished env is
    the first window of its next episode.
    """

    def __init__(self, num_envs, device=None, seed=None, config=None, auto_reset=True, env_id_base=0,
                 with_info=True, tie_band=1e-12):
        super().__init__(_capi.load, "uavenv", device, "UAVEnvBatched")
        self.cfg = (config if config is not None else _global_cfg).copy()
        self.num_envs = int(num_envs)
        self.seed = int(self.cfg.SEED if seed is None else seed)
        self.env_id_base = int(env_id_base)
        self.auto_reset = bool(auto_reset)
        self.N, self.M = int(self.cfg.NUM_UAVS), int(self.cfg.NUM_TARGETS)
        self.K1, self.K2 = int(self.cfg.NUM_NFZ), int(self.cfg.NUM_INTERCEPTORS)
        self.action_space = _Discrete(self.cfg.ACTION_DIM)
        self.observation_space = _Box((self.cfg.SEQ_LEN, self.cfg.STATE_DIM))
        ccfg = self.cfg.to_c(auto_reset=self.auto_reset, tie_band=tie_band)
        self._create(C.byref(ccfg), self.num_envs, self.device.index, self.seed, self.env_id_base)
        B, dev = self.num_envs, self.device
        self.obs = torch.zeros(B, _capi.SEQ_LEN, _capi.STATE_DIM, dtype=torch.float32, device=dev)
        # per-step outputs are carved out of ONE allocation (8-byte aligned slices): fewer distinct pages per launch
        Bp = (B + 7) // 8 * 8
        self._io = torch.zeros(Bp * 30, dtype=torch.uint8, device=dev)
        off = [0]

        def carve(dtype, nbytes_per):
            t = self._io[off[0]:off[0] + B * nbytes_per].view(dtype)
            off[0] += Bp * nbytes_per
            return t

        reward_f64 = carve(torch.float64, 8)
        self.reward = carve(torch.float32, 4)
        j_val, n_asg = carve(torch.float32, 4), carve(torch.int32, 4)
        avg_pd, avg_pf = carve(torch.float32, 4), carve(torch.float32, 4)
        self._done_u8 = carve(torch.uint8, 1)
        valid = carve(torch.int8, 1)
        self.done = self._done_u8.view(torch.bool)
        self.info = {}
        self._info_c = None
        if with_info:
            self.info = {"J_val": j_val, "num_assigned": n_asg,
                         "is_valid_action": valid,                     # -1 None / 0 False / 1 True
                         "avg_p_dmg": avg_pd, "avg_p_final": avg_pf, "reward_f64": reward_f64}
            ic = _capi.UavenvInfo()
            ic.d_J_val = self.info["J_val"].data_ptr()
            ic.d_num_assigned = self.info["num_assigned"].data_ptr()
            ic.d_is_valid_action = self.info["is_valid_action"].data_ptr()
            ic.d_avg_p_dmg = self.info["avg_p_dmg"].data_ptr()
            ic.d_avg_p_final = self.info["avg_p_final"].data_ptr()
            ic.d_reward_f64 = self.info["reward_f64"].data_ptr()
            self._info_c = ic
        self._actions = torch.zeros(B, dtype=torch.int64, device=dev)
        self._h_reward = self._h_done = None
        self._best_target_cache = None        # best_target_actions' per-env entries, allocated on first use
        self._improve_workspace = None        # improve_allocation's / upper_bound's N x M slices (large N*M only), on first use

    # ------------------------------------------------------------------ reset / step
    def reset(self, full_reset=True, env_mask=None):
        """envs/uav_env.py:42-63 for every env (or those with env_mask[b] != 0)."""
        mask_ptr = None
        if env_mask is not None:
            env_mask = torch.as_tensor(env_mask).to(device=self.device, dtype=torch.uint8).contiguous()
            if env_mask.numel() != self.num_envs:
                raise ValueError("env_mask must have num_envs elements")
            mask_ptr = C.c_void_p(env_mask.data_ptr())
        self._chk(self._lib.uavenv_reset(self._h, int(bool(full_reset)), mask_ptr, C.c_void_p(self.obs.data_ptr()),
                                         self._stream()))
        self._forget_best_targets()
        return self.obs

    def _forget_best_targets(self):
        # a full reset or a scene load restarts the episode counter at 1: the cache key alone cannot tell the new episode 1
        # from the old one when the first call after it comes later than the first step
        if self._best_target_cache is not None:
            self._best_target_cache.zero_()

    def _as_actions(self, actions):
        if isinstance(actions, torch.Tensor) and actions.device == self.device and actions.dtype == torch.int64 \
                and actions.is_contiguous():
            a = actions
        else:
            self._actions.copy_(torch.as_tensor(actions).reshape(-1).to(torch.int64), non_blocking=True)
            a = self._actions
        if a.numel() != self.num_envs:
            raise ValueError("expected %d actions, got %d" % (self.num_envs, a.numel()))
        return a

    def step(self, actions):
        """envs/uav_env.py:295-435 for all envs in one fused launch.  1 = Assign, anything else = Skip."""
        a = self._as_actions(actions)
        self._chk(self._lib.uavenv_step(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(self.obs.data_ptr()),
                                        C.c_void_p(self.reward.data_ptr()), C.c_void_p(self._done_u8.data_ptr()),
                                        C.byref(self._info_c) if self._info_c is not None else None, self._stream()))
        return self.obs, self.reward, self.done, self.info

    def step_host(self, actions_cpu, reward_out=None, done_out=None, obs_out=None):
        """The same step driven from HOST buffers (the reference's caller lives on the host):
        actions (int64, or one byte each as int8/uint8) travel host->device, reward/done device->host, inside the
        call - in place over PCIe when the tensors are pinned, through staging copies otherwise.  The observation
        window stays in self.obs on the device for the policy; with obs_out (a pinned host [B,5,14] f32 tensor) it is
        ALSO copied to the host inside the call, i.e. the reference's full (obs, reward, done) crosses the boundary
        (envs/uav_env.py:435).  Returns (reward_cpu, done_cpu)."""
        if self._h_reward is None:
            self._h_reward = torch.zeros(self.num_envs, dtype=torch.float32).pin_memory()
            self._h_done = torch.zeros(self.num_envs, dtype=torch.uint8).pin_memory()
        r = self._h_reward if reward_out is None else reward_out
        d = self._h_done if done_out is None else done_out
        if actions_cpu.is_cuda or actions_cpu.numel() != self.num_envs or not actions_cpu.is_contiguous() \
                or actions_cpu.dtype not in (torch.int64, torch.int8, torch.uint8):
            raise ValueError("actions_cpu must be a contiguous host int64 / int8 / uint8 tensor with num_envs elements")
        fn = self._lib.uavenv_step_host if actions_cpu.dtype == torch.int64 else self._lib.uavenv_step_host_i8
        self._chk(fn(self._h, C.c_void_p(actions_cpu.data_ptr()), C.c_void_p(r.data_ptr()), C.c_void_p(d.data_ptr()),
                     C.c_void_p(self.obs.data_ptr()), self._stream()))
        if obs_out is not None:
            if obs_out.is_cuda or obs_out.dtype != torch.float32 or obs_out.numel() != self.obs.numel() \
                    or not obs_out.is_contiguous():
                raise ValueError("obs_out must be a contiguous host float32 tensor of [num_envs,5,14]")
            obs_out.copy_(self.obs, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        return r, d

    def random_actions(self, step, action_seed=1, out=None):
        """Bernoulli(1/2) actions keyed (action_seed, step, global env id) - the benchmark action stream."""
        out = self._actions if out is None else out
        self._chk(self._lib.uavenv_random_actions(self._h, int(action_seed), int(step), C.c_void_p(out.data_ptr()),
                                                  self._stream()))
        return out

    def best_target_actions(self, out=None):
        """Actions [B] int64 (device) of the best-target heuristic at the current pointers: UAV k Assigns iff the pointer
        target is the one whose tentative assignment gives the highest paper reward (Eq.19; lowest index on a tie) and
        that reward is not below the current one.  The best target is computed once per UAV row and cached on the device
        (keyed by episode and UAV pointer); call after reset() / a step, on the env's stream."""
        out = self._actions if out is None else out
        if not (isinstance(out, torch.Tensor) and out.device == self.device and out.dtype == torch.int64
                and out.is_contiguous() and out.numel() == self.num_envs):
            raise ValueError("out must be a contiguous int64 tensor of num_envs elements on the env's device")
        if self._best_target_cache is None:
            self._best_target_cache = torch.zeros(self.num_envs, dtype=torch.int64, device=self.device)
        self._chk(self._lib.uavenv_best_target_actions(self._h, C.c_void_p(self._best_target_cache.data_ptr()),
                                                       C.c_void_p(out.data_ptr()), self._stream()))
        return out

    # ------------------------------------------------------------------ scene / state access
    def _dims(self):
        return {"N": self.N, "M": self.M, "K1": self.K1, "K2": self.K2, "1": 1}

    def _scene_struct(self, scene, array):
        """(scene count, the arrays to keep alive, a UavenvScene of their addresses) of a scene dict named as
        _capi.SCENE_FIELDS; array(value, kind) -> (contiguous array, element count, address)."""
        dims = self._dims()
        count = None
        keep, sc = [], _capi.UavenvScene()
        for name, kind, dim in _capi.SCENE_FIELDS:
            if name not in scene or scene[name] is None:
                if name in ("uav_type", "nfz_radius") or dims[dim] == 0:
                    continue
                raise KeyError("scene is missing %r" % name)
            if dims[dim] == 0:
                continue
            a, n, ptr = array(scene[name], kind)
            c = n // dims[dim]
            if n != c * dims[dim] or c == 0:
                raise ValueError("scene[%r] has %d elements, not a multiple of %d" % (name, n, dims[dim]))
            if count is None:
                count = c
            elif c != count:
                raise ValueError("scene arrays disagree on the number of scenes")
            keep.append(a)
            setattr(sc, name, ptr)
        return count, keep, sc

    def load_scene(self, scene, first_env=0):
        """Inject scenes (dict of arrays named as include/uavenv_b200.h:uavenv_scene, list order; one env
        ([N]) or several ([count,N])) into envs [first_env, first_env+count); they are left reset
        (episode 1).  Returns their first observation windows (a view of self.obs)."""
        def host(v, kind):
            a = np.ascontiguousarray(np.asarray(v, dtype=_NP[kind]))
            return a, a.size, a.ctypes.data

        count, keep, sc = self._scene_struct(scene, host)
        self._chk(self._lib.uavenv_load_scene(self._h, C.byref(sc), int(first_env), int(count),
                                              C.c_void_p(self.obs.data_ptr())))
        self._forget_best_targets()
        return self.obs[first_env:first_env + count]

    def load_scene_device(self, scene, copies=1, first_env=0):
        """Inject S scenes given as device tensors (dict named as _capi.SCENE_FIELDS, shapes [S,N] / [S,M] / [S,K1] /
        [S,K2]; host tensors or numpy arrays are moved to the env's device first) into envs [first_env, first_env +
        S*copies): scene s goes to envs first_env + s*copies + c, c in [0, copies), left reset (episode 1).  No host
        round trip and no synchronisation: the packing runs on the env's stream.  Returns the loaded envs' first
        observation windows (a view of self.obs)."""
        def device(v, kind):
            t = torch.as_tensor(v).to(device=self.device, dtype=_TORCH[kind]).contiguous()
            return t, t.numel(), t.data_ptr()

        # (a copy made here is freed in stream order when `keep` goes: the packing has read it by then)
        count, keep, sc = self._scene_struct(scene, device)
        self._chk(self._lib.uavenv_load_scene_device(self._h, C.byref(sc), int(count), int(copies), int(first_env),
                                                     C.c_void_p(self.obs.data_ptr()), self._stream()))
        self._forget_best_targets()
        return self.obs[first_env:first_env + count * int(copies)]

    def group_best(self, group_size, first_env=0, num_groups=None):
        """The best member of each group of `group_size` consecutive envs from first_env (an env built with
        auto_reset=False, after its episodes have finished): highest J (= get_state()["J_val"], bit for bit), lowest
        member index on a tie.  Returns device tensors {"best": int32 [G] member index (-1: a member has not finished),
        "J": f64 [G], "assigned_target_id": int32 [G,N] (Target.id, -1 = unassigned), "num_covered": int32 [G],
        "J_all": f64 [G, group_size] every member's J}.  One launch on the env's stream."""
        group_size = int(group_size)
        if num_groups is None:
            num_groups = (self.num_envs - int(first_env)) // max(group_size, 1)
        G, dev = int(num_groups), self.device
        out = {"best": torch.empty(G, dtype=torch.int32, device=dev), "J": torch.empty(G, dtype=torch.float64, device=dev),
               "assigned_target_id": torch.empty(G, self.N, dtype=torch.int32, device=dev),
               "num_covered": torch.empty(G, dtype=torch.int32, device=dev),
               "J_all": torch.empty(G, group_size, dtype=torch.float64, device=dev)}
        self._chk(self._lib.uavenv_group_best(self._h, int(first_env), G, group_size,
                                              *(C.c_void_p(out[k].data_ptr()) for k in ("best", "J", "assigned_target_id",
                                                                                        "num_covered", "J_all")),
                                              self._stream()))
        return out

    def improve_allocation(self, assigned, first_env=0, env_stride=1, max_moves=None):
        """Steepest-ascent local search (single-UAV moves and two-UAV swaps, include/uavenv_b200.h:
        uavenv_improve_allocation) on the allocations assigned [S, N] (Target.id, -1 = none; moved to the device) of the
        scenes held by envs first_env + s * env_stride.  max_moves: cap on applied moves per scene (None: 16 * N).
        Returns device tensors {"assigned_target_id": int32 [S,N], "J": f64 [S], "J_before": f64 [S], "num_covered":
        int32 [S] (N0), "moves": int32 [S], "converged": bool [S] (False: the cap stopped the search before a local
        optimum)}.  A row with an id that is not a Target.id of its scene gets moves -1, J NaN, N0 -1 and a row of -1.
        One launch on the env's stream."""
        a = torch.as_tensor(assigned).to(device=self.device, dtype=torch.int32).contiguous()
        if a.numel() == 0 or a.numel() % self.N:
            raise ValueError("assigned has %d elements, not a positive multiple of N = %d" % (a.numel(), self.N))
        S, dev = a.numel() // self.N, self.device
        max_moves = 16 * self.N if max_moves is None else int(max_moves)
        ws = self._workspace()
        out = {"assigned_target_id": torch.empty(S, self.N, dtype=torch.int32, device=dev),
               "J": torch.empty(S, dtype=torch.float64, device=dev),
               "J_before": torch.empty(S, dtype=torch.float64, device=dev),
               "num_covered": torch.empty(S, dtype=torch.int32, device=dev),
               "moves": torch.empty(S, dtype=torch.int32, device=dev),
               "converged": torch.empty(S, dtype=torch.uint8, device=dev)}
        self._chk(self._lib.uavenv_improve_allocation(
            self._h, int(first_env), S, int(env_stride), C.c_void_p(a.data_ptr()), max_moves,
            *(C.c_void_p(out[k].data_ptr()) for k in ("assigned_target_id", "J_before", "J", "num_covered", "moves",
                                                      "converged")),
            C.c_void_p(ws.data_ptr() if ws is not None else None), self._stream()))
        out["converged"] = out["converged"].view(torch.bool)
        return out

    def _workspace(self):
        """The workspace of improve_allocation and upper_bound (uavenv_improve_workspace_bytes), or None when 0."""
        ws = int(self._lib.uavenv_improve_workspace_bytes(self._h))
        if ws and (self._improve_workspace is None or self._improve_workspace.numel() < ws):
            self._improve_workspace = torch.empty(ws, dtype=torch.uint8, device=self.device)
        return self._improve_workspace if ws else None

    def upper_bound(self, first_env=0, count=None, env_stride=1, iters=256):
        """Certified upper bound on the best J of the scenes held by envs first_env + s * env_stride, s in [0, count)
        (count None: as many as fit): Frank-Wolfe on the concave relaxation of J for at most `iters` iterations
        (include/uavenv_b200.h: uavenv_upper_bound states the rule and why the bound is valid).  Returns device tensors
        {"bound": f64 [S] (no allocation of the scene has a higher J), "relaxed": f64 [S] (the relaxation's value at the
        last iterate), "iters": int32 [S] (iterations run)}.  One launch on the env's stream."""
        first_env, env_stride = int(first_env), int(env_stride)
        if count is None:
            count = (self.num_envs - first_env + env_stride - 1) // max(env_stride, 1)
        S, dev = int(count), self.device
        out = {"bound": torch.empty(max(S, 0), dtype=torch.float64, device=dev),
               "relaxed": torch.empty(max(S, 0), dtype=torch.float64, device=dev),
               "iters": torch.empty(max(S, 0), dtype=torch.int32, device=dev)}
        ws = self._workspace()
        self._chk(self._lib.uavenv_upper_bound(
            self._h, first_env, S, env_stride, int(iters), *(C.c_void_p(out[k].data_ptr()) for k in ("bound", "relaxed", "iters")),
            C.c_void_p(ws.data_ptr() if ws is not None else None), self._stream()))
        return out

    def get_scene(self, first_env=0, count=None):
        count = self.num_envs - first_env if count is None else count
        dims = self._dims()
        out, sc = {}, _capi.UavenvScene()
        for name, kind, dim in _capi.SCENE_FIELDS:
            out[name] = np.zeros((count, dims[dim]), dtype=_NP[kind])
            if dims[dim]:
                setattr(sc, name, out[name].ctypes.data)
        self._chk(self._lib.uavenv_get_scene(self._h, C.byref(sc), int(first_env), int(count)))
        return out

    def get_state(self, first_env=0, count=None):
        count = self.num_envs - first_env if count is None else count
        dims = self._dims()
        out, st = {}, _capi.UavenvState()
        for name, kind, dim in _capi.STATE_FIELDS:
            shape = (count,) if dim == "1" else (count, dims[dim])
            out[name] = np.zeros(shape, dtype=_NP[kind])
            setattr(st, name, out[name].ctypes.data)
        self._chk(self._lib.uavenv_get_state(self._h, C.byref(st), int(first_env), int(count)))
        return out

    def set_episode_counters(self, episode, first_env=0):
        """Restore the 1-based per-env episode counters behind the main_train.py:79 schedule."""
        ep = np.ascontiguousarray(np.asarray(episode, dtype=np.int32).reshape(-1))
        self._chk(self._lib.uavenv_set_episode_counters(self._h, C.c_void_p(ep.ctypes.data), int(first_env), ep.size))

    def scene(self, b):
        """(uavs, targets, nfz_list, interceptors) of env b as reference-style entity objects."""
        sc = {k: v[0] for k, v in self.get_scene(b, 1).items()}
        st = self.get_state(b, 1)
        return build_entities(sc, st["assigned_target_id"][0], self.cfg.INTERCEPT_RAD)

    @property
    def uav_idx(self):
        return self.get_state()["uav_idx"]

    @property
    def target_idx(self):
        return self.get_state()["target_idx"]

    def score_matrix(self, dtype=torch.float32):
        """p_final, p_damage [B,N,M] - the main.py:38-45 double loop over mechanics.calc_advantage."""
        pf = torch.empty(self.num_envs, self.N, self.M, dtype=dtype, device=self.device)
        pd = torch.empty_like(pf)
        fn = self._lib.uavenv_score_matrix if dtype == torch.float32 else self._lib.uavenv_score_matrix_f64
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be float32 or float64")
        self._chk(fn(self._h, C.c_void_p(pf.data_ptr()), C.c_void_p(pd.data_ptr()), self._stream()))
        return pf, pd

    def recompute_objective(self):
        """Re-derive the running objective from the per-target products (warp per env); returns the
        largest |carried J - fresh J| found, and re-anchors the running sums."""
        v = C.c_double(0.0)
        self._chk(self._lib.uavenv_recompute_objective(self._h, C.byref(v), self._stream()))
        return v.value


class UAVEnv:
    """Single-env drop-in with the reference's signatures (envs/uav_env.py:13-63,295-435):
    reset(full_reset=True) -> np.float32[5,14];  step(action) -> (obs, reward: float, done: bool, info: dict).
    Sizes and constants are read from the module-level `cfg` when the env is constructed."""

    def __init__(self, device=None, seed=None, config=None):
        self._env = UAVEnvBatched(1, device=device, seed=seed, config=config, auto_reset=False)
        self.cfg = self._env.cfg
        self.action_space = self._env.action_space
        self.observation_space = self._env.observation_space
        self._done = True
        self._entities = None

    def reset(self, full_reset=True):
        obs = self._env.reset(full_reset=full_reset)
        self._done = False
        self._entities = None
        return obs[0].cpu().numpy()

    def load_scene(self, scene):
        obs = self._env.load_scene(scene, 0)
        self._done = False
        self._entities = None
        return obs[0].cpu().numpy()

    def step(self, action):
        if self._done:
            raise IndexError("step() on a finished episode - call reset() (envs/uav_env.py:296)")
        obs, _, done, info = self._env.step(torch.tensor([int(action)], dtype=torch.int64))
        self._entities = None
        done_b = bool(done[0].item())
        self._done = done_b
        v = int(info["is_valid_action"][0].item())
        out_info = {
            "J_val": float(info["J_val"][0].item()),
            "num_assigned": int(info["num_assigned"][0].item()),
            "is_valid_action": None if v < 0 else bool(v),
            "avg_p_dmg": float(info["avg_p_dmg"][0].item()),
            "avg_p_final": float(info["avg_p_final"][0].item()),
        }
        obs_np = np.zeros(self.cfg.STATE_DIM, np.float32) if done_b else obs[0].cpu().numpy()  # uav_env.py:188-189
        return obs_np, float(info["reward_f64"][0].item()), done_b, out_info

    def _ents(self):
        if self._entities is None:
            self._entities = self._env.scene(0)
        return self._entities

    uavs = property(lambda self: self._ents()[0])
    targets = property(lambda self: self._ents()[1])
    nfz_list = property(lambda self: self._ents()[2])
    interceptors = property(lambda self: self._ents()[3])
    uav_idx = property(lambda self: int(self._env.get_state(0, 1)["uav_idx"][0]))
    target_idx = property(lambda self: int(self._env.get_state(0, 1)["target_idx"][0]))

    def close(self):
        self._env.close()
