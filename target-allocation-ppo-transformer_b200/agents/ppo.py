"""PPO rollout post-processing on the device (agents/ppo.py:77-94 of the reference).

compute_gae runs the chunked warp-scan GAE kernel + advantage normalisation of csrc/ppo_gae.cu on a
time-major [T,B] rollout.  With a torch.distributed process group the three normalisation
statistics {count, sum, sum of squares} are all-reduced so every rank normalises with the global
mean / unbiased std, as one big single-GPU batch would (SURVEY.md §8e).
"""
import ctypes as C

import torch

from .. import _capi


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def compute_gae(rewards, values, dones, last_value=None, gamma=0.998, lam=0.95, normalize=True, group=None):
    """rewards, values: f32 [T,B]; dones: bool/uint8 [T,B]; last_value: f32 [B] or None (episodic, V_T = 0).
    Returns (returns [T,B], advantages [T,B]).  Defaults are cfg.GAMMA / cfg.GAE_LAMBDA."""
    if rewards.dim() == 1:
        rewards, values, dones = rewards[:, None], values[:, None], dones[:, None]
        squeeze = True
    else:
        squeeze = False
    if not rewards.is_cuda:
        raise RuntimeError("compute_gae runs on the GPU only (no CPU fallback)")
    T, B = rewards.shape
    dev = rewards.device
    rewards = rewards.contiguous().float()
    values = values.contiguous().float()
    dones_u8 = dones.contiguous().view(torch.uint8) if dones.dtype == torch.bool else dones.contiguous().to(torch.uint8)
    if last_value is not None:
        last_value = last_value.contiguous().float()
    returns = torch.empty_like(rewards)
    adv = torch.empty_like(rewards)
    stats = torch.zeros(3, dtype=torch.float64, device=dev)
    lib = _capi.load()
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    distributed = group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()
                                        and torch.distributed.get_world_size() > 1)
    local_norm = int(bool(normalize) and not distributed)
    _capi.check(lib.ppo_gae_advantages(_ptr(rewards), _ptr(values), _ptr(dones_u8), _ptr(last_value), T, B, float(gamma),
                                       float(lam), _ptr(returns), _ptr(adv), local_norm, _ptr(stats), dev.index, stream))
    if normalize and distributed:
        torch.distributed.all_reduce(stats, group=group)
        _capi.check(lib.ppo_normalize_advantages(_ptr(adv), T * B, _ptr(stats), dev.index, stream))
    if squeeze:
        returns, adv = returns[:, 0], adv[:, 0]
    return returns, adv


def normalize_advantages(adv, stats):
    lib = _capi.load()
    stream = C.c_void_p(torch.cuda.current_stream(adv.device).cuda_stream)
    _capi.check(lib.ppo_normalize_advantages(_ptr(adv), adv.numel(), _ptr(stats), adv.device.index, stream))
    return adv


# ------------------------------------------------------------------------------------------------------------
# Batched PPO agent (agents/ppo.py:12-183 of the reference, for a [T,B] device-resident rollout)

class PPOAgent:
    """select_action / store_transition / update with the reference's losses and optimiser
    (ppo.py:17-22 four Adam groups; :131-153 clipped surrogate, max-of-means clipped value loss, entropy bonus;
    :160 global-norm clip), over a fixed-horizon rollout of B envs instead of a Python list of single steps.

    Differences forced by batching (SURVEY.md section 7): the rollout is cut at a fixed horizon T, so V(s_T)
    bootstraps the last step (the reference only updates at episode ends, where it is 0, ppo.py:77); the
    minibatch is `minibatch_size` transitions (default T*B/4; cfg.BATCH_SIZE = 64 suits the reference's
    ~300-sample buffers).  With a process group, gradients are summed over ranks in ONE flat NCCL all-reduce
    per minibatch (the parameters' .grad are views into one buffer), then averaged, clipped and applied.
    """

    def __init__(self, num_envs, horizon, device, cfg=None, group=None, minibatch_size=None, seed=0,
                 fused_rollout=False, env_id_base=0, update_precision="tf32", graph_update=False, optimizer="fused"):
        from ..configs.config import cfg as global_cfg
        from ..networks.transformer_net import TransformerActorCritic
        self.cfg = cfg or global_cfg
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.B, self.T = int(num_envs), int(horizon)
        self.group = group
        self.world = torch.distributed.get_world_size(group) if (
            torch.distributed.is_available() and torch.distributed.is_initialized()) else 1
        # identical initial weights on every rank, without touching the caller's global RNG stream
        devs = [self.device] if self.device.type == "cuda" else []
        with torch.random.fork_rng(devices=devs):
            torch.manual_seed(seed)
            self.policy = TransformerActorCritic(self.cfg).to(self.device)
            self.policy_old = TransformerActorCritic(self.cfg).to(self.device)
        self.policy_old.load_state_dict(self.policy.state_dict())
        c = self.cfg
        # graph_update: after three eager minibatch steps the whole step is captured once and replayed as one CUDA
        # graph launch (Adam's step counter lives on the device)
        self.graph_update = bool(graph_update) and self.device.type == "cuda"
        if optimizer not in ("fused", "torch"):
            raise ValueError("optimizer must be 'fused' (csrc/ppo_optim.cu) or 'torch' (torch.optim.Adam, A/B reference)")
        groups = [                                                                # ppo.py:17-22
            {"params": list(self.policy.actor_head.parameters()), "lr": c.LR_ACTOR},
            {"params": list(self.policy.actor_net.parameters()), "lr": c.LR_ACTOR},
            {"params": list(self.policy.critic_head.parameters()), "lr": c.LR_CRITIC},
            {"params": list(self.policy.critic_net.parameters()), "lr": c.LR_CRITIC},
        ]
        params = list(self.policy.parameters())
        self.num_params = sum(p.numel() for p in params)
        # parameters and their .grad are views of ONE flat buffer each (state_dict order): the library reads the
        # weights in place, the all-reduce is one call, and clip + Adam run over the flat buffers (csrc/ppo_optim.cu)
        self._flat_params = torch.empty(self.num_params, device=self.device)
        self._flat_grad = torch.zeros(self.num_params, device=self.device)
        lr_of = {id(p): g["lr"] for g in groups for p in g["params"]}
        off, seg_end, seg_lr = 0, [], []
        for p in params:
            n = p.numel()
            self._flat_params[off:off + n].copy_(p.detach().reshape(-1))
            p.data = self._flat_params[off:off + n].view_as(p)
            p.grad = self._flat_grad[off:off + n].view_as(p)
            off += n
            if seg_lr and seg_lr[-1] == lr_of[id(p)]:
                seg_end[-1] = off
            else:
                seg_end.append(off); seg_lr.append(lr_of[id(p)])
        self.optimizer_kind = optimizer if self.device.type == "cuda" else "torch"
        if self.optimizer_kind == "torch":
            self.optimizer = torch.optim.Adam(groups, capturable=self.graph_update)
        else:
            self.optimizer = None
            self._seg_end = (C.c_int64 * len(seg_end))(*seg_end)
            self._seg_lr = (C.c_float * len(seg_lr))(*seg_lr)
            self._exp_avg = torch.zeros(self.num_params, device=self.device)
            self._exp_avg_sq = torch.zeros(self.num_params, device=self.device)
            self._adam_step = torch.zeros(1, dtype=torch.int64, device=self.device)
            self._norm_partials = torch.zeros(_capi.load().ppo_optim_partials(), dtype=torch.float64, device=self.device)
            self.grad_norm = torch.zeros(1, device=self.device)      # pre-clip norm of the last step
        T, B, dev = self.T, self.B, self.device
        self.buf_obs = torch.zeros(T, B, c.SEQ_LEN, c.STATE_DIM, device=dev)
        self.buf_action = torch.zeros(T, B, dtype=torch.int64, device=dev)
        self.buf_logp = torch.zeros(T, B, device=dev)
        self.buf_value = torch.zeros(T, B, device=dev)
        self.buf_reward = torch.zeros(T, B, device=dev)
        self.buf_done = torch.zeros(T, B, dtype=torch.bool, device=dev)
        self.t = 0
        self.minibatch_size = int(minibatch_size) if minibatch_size else max(c.BATCH_SIZE, (T * B) // 4)
        mb = min(self.minibatch_size, T * B)
        self._mb_idx = torch.zeros(mb, dtype=torch.int64, device=dev)             # persistent inputs of a minibatch step
        self._ret = torch.zeros(T * B, device=dev)
        self._adv = torch.zeros(T * B, device=dev)
        self._mb_sums = torch.zeros(3, device=dev)
        self._mb_stats = torch.zeros(3, device=dev)
        self._graph, self._graph_warm = None, 0
        self._side = torch.cuda.Stream(device=dev) if self.graph_update else None
        self._gen = torch.Generator(device=dev).manual_seed(seed + 1 + (
            torch.distributed.get_rank(group) if self.world > 1 else 0))
        # the update's GEMMs (PyTorch autograd on the mirror network): "tf32" tensor-core math or strict "fp32"
        # or "fused": the hand-written sm_100a forward + backward of both trunks (csrc/policy_train.cu; bf16 operands,
        # fp32 accumulation and gradients), PyTorch only for the two small heads and the loss
        if update_precision not in ("tf32", "fp32", "fused"):
            raise ValueError("update_precision must be 'fused', 'tf32' or 'fp32'")
        self.update_precision = update_precision
        self.trunks = None
        if update_precision == "fused":
            from ..networks.fused_train import FusedTrunks
            self.trunks = FusedTrunks(min(self.minibatch_size, T * B), dev)
        # rollout forward on the tensor cores (csrc/policy_forward.cu) instead of the fp32 PyTorch mirror
        self.fused = None
        self._rollout_step = 0
        if fused_rollout:
            from ..networks.fused_forward import FusedPolicyForward
            self.fused = FusedPolicyForward(self.B, dev, seed=seed, env_id_base=env_id_base)
            self.fused.sync(self.policy_old)

    def close(self):
        """Release the captured update graph (it holds NCCL kernels: destroy it BEFORE destroy_process_group())."""
        if self._graph is not None:
            torch.cuda.synchronize(self.device)
            self._graph = None
            import gc
            gc.collect()
            torch.cuda.synchronize(self.device)

    # -- rollout ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def select_action(self, obs):
        """ppo.py:52-62 for a batch: sample from policy_old, remember (state, action, log-prob, value)."""
        if self.fused is not None:
            action, logp, value, _ = self.fused.get_action(obs, self._rollout_step)
            self._rollout_step += 1
        else:
            action, logp, value, _ = self.policy_old.get_action(obs, generator=self._gen)
        t = self.t
        self.buf_obs[t].copy_(obs); self.buf_action[t].copy_(action)
        self.buf_logp[t].copy_(logp); self.buf_value[t].copy_(value.squeeze(-1))
        return action

    def store_transition(self, reward, done):
        """ppo.py:64-66"""
        self.buf_reward[self.t].copy_(reward); self.buf_done[self.t].copy_(done)
        self.t += 1

    def full(self):
        return self.t >= self.T

    def clear_buffer(self):
        """ppo.py:183: drop the collected transitions (update() does this itself)."""
        self.t = 0

    # -- update -------------------------------------------------------------------------------------------
    def update(self, last_obs):
        """ppo.py:68-181.  Returns the mean losses like the reference ({"loss_actor","loss_critic","entropy"})."""
        c = self.cfg
        assert self.t == self.T, "update() needs a full rollout"
        tf32_before = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = self.update_precision != "fp32"
        try:
            return self._update(last_obs)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = tf32_before

    def _minibatch_step(self):
        """One optimiser step (ppo.py:117-168) on the minibatch whose buffer indices sit in self._mb_idx.  Touches only
        persistent tensors, so that the whole step - gather, evaluate, losses, backward, gradient all-reduce, clip,
        Adam - can be replayed as one CUDA graph."""
        c = self.cfg
        n = self.T * self.B
        idx = self._mb_idx
        obs = self.buf_obs.view(n, c.SEQ_LEN, c.STATE_DIM)
        act, old_logp, old_val = self.buf_action.view(n), self.buf_logp.view(n), self.buf_value.view(n)
        if self.trunks is not None:                                         # forward, loss and backward in the library
            self.trunks.ppo_step(self._flat_params, obs[idx], act[idx], old_logp[idx], self._adv[idx], self._ret[idx],
                                 old_val[idx], c.EPS_CLIP, 0.5, 0.01, self._flat_grad, self._mb_stats)
            self._apply_gradient()
            self._mb_sums += self._mb_stats
            return
        logp, value, entropy = self.policy.evaluate(obs[idx], act[idx])
        value = value.squeeze(-1)
        ratio = torch.exp(logp - old_logp[idx])                             # :131
        a = self._adv[idx]
        loss_actor = -torch.min(ratio * a, torch.clamp(ratio, 1 - c.EPS_CLIP, 1 + c.EPS_CLIP) * a).mean()
        v_clip = old_val[idx] + torch.clamp(value - old_val[idx], -c.EPS_CLIP, c.EPS_CLIP)     # :141
        r = self._ret[idx]
        loss_critic = torch.max(((value - r) ** 2).mean(), ((v_clip - r) ** 2).mean())           # :143-147
        ent = entropy.mean()
        loss = loss_actor + 0.5 * loss_critic - 0.01 * ent                  # :153
        self._flat_grad.zero_()
        loss.backward()
        self._apply_gradient()
        self._mb_sums += torch.stack([loss_actor.detach(), loss_critic.detach(), ent.detach()])

    def _apply_gradient(self):
        """all-reduce (the only collective of training), then averaging over ranks + global-norm clip (ppo.py:160) + the
        four-group Adam step (ppo.py:17-22,162) as two launches over the flat buffers (csrc/ppo_optim.cu)"""
        c = self.cfg
        if self.world > 1:
            torch.distributed.all_reduce(self._flat_grad, group=self.group)
        if self.optimizer_kind == "torch":                                  # A/B reference: eager tensor ops + torch Adam
            if self.world > 1:
                self._flat_grad.div_(self.world)
            norm = self._flat_grad.norm()
            self._flat_grad.mul_(torch.clamp(c.GRAD_NORM_CLIP / (norm + 1e-6), max=1.0))
            self.optimizer.step()
            return
        _capi.check(_capi.load().ppo_clip_adam_step(
            _ptr(self._flat_params), _ptr(self._flat_grad), _ptr(self._exp_avg), _ptr(self._exp_avg_sq), self.num_params,
            self._seg_end, self._seg_lr, len(self._seg_lr), 1.0 / self.world, float(c.GRAD_NORM_CLIP), 0.9, 0.999, 1e-8,
            _ptr(self._adam_step), _ptr(self._norm_partials), _ptr(self.grad_norm), self.device.index,
            C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def launches_per_minibatch(self):
        """Own kernels launched by one minibatch step (bench.py's gpu_launches claim)."""
        n = 79 if self.trunks is not None else 0      # 32 tcgen05 GEMMs, 16 weight-gradient, 29 LN / attention / embedding / head, 2 loss
        return n + (2 if self.optimizer_kind == "fused" else 0)

    def time_gradient_allreduce(self, iters=50):
        """Microseconds per NCCL all-reduce of a buffer shaped like the flat gradient (CUDA events around `iters`
        back-to-back calls on the current stream); 0.0 on one rank."""
        if self.world == 1:
            return 0.0
        buf = torch.zeros_like(self._flat_grad)
        for _ in range(5):
            torch.distributed.all_reduce(buf, group=self.group)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(self.device)
        e0.record()
        for _ in range(iters):
            torch.distributed.all_reduce(buf, group=self.group)
        e1.record()
        torch.cuda.synchronize(self.device)
        return 1e3 * e0.elapsed_time(e1) / iters

    def _run_minibatch(self):
        """Eager for the first steps (they double as the warm-up torch wants before a capture), then ONE graph launch."""
        if not self.graph_update:
            return self._minibatch_step()
        if self._graph is not None:
            return self._graph.replay()
        cur = torch.cuda.current_stream(self.device)
        if self._graph_warm < 3:
            self._graph_warm += 1
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self._minibatch_step()
            cur.wait_stream(self._side)
            return
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self._side):
            self._minibatch_step()
        self._graph = g
        g.replay()

    def _update(self, last_obs):
        c = self.cfg
        if self.fused is not None:          # V(s_T) from the same tcgen05 forward that produced the rollout's values
            last_value = self.fused.get_action(last_obs, self._rollout_step)[2].clone()
        else:
            with torch.no_grad():
                _, last_value = self.policy_old.logits_and_value(last_obs)
        returns, adv = compute_gae(self.buf_reward, self.buf_value, self.buf_done, last_value.squeeze(-1), c.GAMMA,
                                   c.GAE_LAMBDA, normalize=True, group=self.group if self.world > 1 else None)
        n = self.T * self.B
        self._ret.copy_(returns.view(n)); self._adv.copy_(adv.view(n))
        self._mb_sums.zero_()
        count = 0
        mb = min(self.minibatch_size, n)
        for _ in range(c.K_EPOCHS):                                                # ppo.py:112
            perm = torch.randperm(n, device=self.device, generator=self._gen)
            for i in range(0, n - mb + 1, mb):                                     # drop_last=True (:115)
                self._mb_idx.copy_(perm[i:i + mb])
                self._run_minibatch()
                count += 1
        sums = self._mb_sums
        self.policy_old.load_state_dict(self.policy.state_dict())                  # ppo.py:172
        if self.fused is not None:
            self.fused.sync(self.policy_old)
        self.t = 0
        if count == 0:
            return None
        m = (sums / count).tolist()
        return {"loss_actor": m[0], "loss_critic": m[1], "entropy": m[2]}
