"""The two transformer trunks of the PPO update - forward AND backward - on sm_100a (csrc/policy_train.cu,
policy_wgrad.cu, policy_gemm.cu) as one autograd function behind `TransformerActorCritic.evaluate`
(networks/transformer_net.py:124-143, called from agents/ppo.py:126).

    trunks = FusedTrunks(max_samples, device)
    logp, value, entropy = trunks.evaluate(policy, obs, action)      # differentiable w.r.t. policy.parameters()

bf16 activations / GEMM operands with fp32 accumulation; LayerNorm, softmax, reductions and all parameter gradients
in fp32.  The MLP heads and the loss run in PyTorch on the two [n,128] feature matrices this op returns."""
import ctypes as C

import torch

from .. import _capi
from .fused_forward import flatten_params


class _TrunkFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, owner, obs, flat):
        n = obs.shape[0]
        feat = torch.empty(n, 2, 128, device=obs.device, dtype=torch.float32)
        owner._chk(owner._lib.uavtrain_forward(owner._h, C.c_void_p(flat.data_ptr()), C.c_void_p(obs.data_ptr()), n,
                                               C.c_void_p(feat.data_ptr()), owner._stream()))
        ctx.owner = owner
        ctx.keep = (obs, flat)              # the backward re-reads both in place
        owner._pending = n
        return feat

    @staticmethod
    def backward(ctx, dfeat):
        owner = ctx.owner
        if owner._pending != dfeat.shape[0]:
            raise RuntimeError("FusedTrunks keeps the activations of ONE forward: backward must follow its forward")
        dfeat = dfeat.contiguous().float()
        grad = torch.empty(_capi.NUM_PARAMS, device=dfeat.device, dtype=torch.float32)
        owner._chk(owner._lib.uavtrain_backward(owner._h, C.c_void_p(dfeat.data_ptr()), C.c_void_p(grad.data_ptr()),
                                                owner._stream()))
        owner._pending = 0
        return None, None, grad


class _PolicyFn(torch.autograd.Function):
    """trunks + heads: (obs, flat parameters) -> (logits [n,2], value [n,1])"""

    @staticmethod
    def forward(ctx, owner, obs, flat):
        n = obs.shape[0]
        logits = torch.empty(n, 2, device=obs.device, dtype=torch.float32)
        value = torch.empty(n, 1, device=obs.device, dtype=torch.float32)
        owner._chk(owner._lib.uavtrain_forward_heads(owner._h, C.c_void_p(flat.data_ptr()), C.c_void_p(obs.data_ptr()), n,
                                                     C.c_void_p(logits.data_ptr()), C.c_void_p(value.data_ptr()), owner._stream()))
        ctx.owner = owner
        ctx.keep = (obs, flat)
        owner._pending = n
        return logits, value

    @staticmethod
    def backward(ctx, dlogits, dvalue):
        owner = ctx.owner
        if owner._pending != dlogits.shape[0]:
            raise RuntimeError("FusedTrunks keeps the activations of ONE forward: backward must follow its forward")
        dlogits, dvalue = dlogits.contiguous().float(), dvalue.contiguous().float()
        grad = torch.empty(_capi.NUM_PARAMS, device=dlogits.device, dtype=torch.float32)
        owner._chk(owner._lib.uavtrain_backward_heads(owner._h, C.c_void_p(dlogits.data_ptr()), C.c_void_p(dvalue.data_ptr()),
                                                      C.c_void_p(grad.data_ptr()), owner._stream()))
        owner._pending = 0
        return None, None, grad


class FusedTrunks(_capi.Handle):
    def __init__(self, max_samples, device):
        super().__init__(_capi.load_policy, "uavtrain", device, "the fused PPO update")
        self._create(self.device.index, int(max_samples))
        self.max_samples = int(max_samples)
        self._pending = 0
        self._work = None

    def features(self, module, obs):
        """[n,2,128] fp32: last-token features of actor_net / critic_net; differentiable w.r.t. module.parameters()."""
        return _TrunkFn.apply(self, obs.contiguous().float(), self._fp32_params(module))

    def logits_and_value(self, module, obs):
        """== module.logits_and_value(obs): trunks and heads in the library, differentiable w.r.t. module.parameters()."""
        return _PolicyFn.apply(self, obs.contiguous().float(), self._fp32_params(module))

    @staticmethod
    def _fp32_params(module):
        flat = flatten_params(module)
        if flat.dtype != torch.float32:
            raise ValueError("expected the fp32 parameters of TransformerActorCritic")
        return flat

    def evaluate(self, module, obs, action):
        """== module.evaluate(obs, action) (transformer_net.py:124-143): (log_prob [n], value [n,1], entropy [n])."""
        logits, value = self.logits_and_value(module, obs)
        logp_all = torch.log_softmax(logits, dim=-1)
        entropy = -(logp_all.exp() * logp_all).sum(-1)
        return logp_all.gather(-1, action[:, None]).squeeze(-1), value, entropy

    @torch.no_grad()
    def ppo_step(self, flat_params, obs, action, old_logp, adv, ret, old_value, eps_clip, c_value, c_entropy, grad_out, stats_out=None):
        """One PPO minibatch gradient without autograd: forward (trunks + heads) -> PPO loss value and gradient
        (agents/ppo.py:126-153) -> backward, all in the library.  grad_out [NUM_PARAMS] fp32 is OVERWRITTEN with dL/dparams;
        stats_out (optional, [3]) receives {actor loss, critic loss, mean entropy}.  Inputs are [n]-shaped device tensors."""
        n = obs.shape[0]
        if self._work is None or self._work.shape[0] < n:
            self._work = torch.empty(self.max_samples, 6, device=self.device, dtype=torch.float32)
        w = self._work
        p = lambda t: C.c_void_p(t.data_ptr())
        obs, action = obs.contiguous().float(), action.contiguous()
        old_logp, adv, ret, old_value = (t.contiguous().float() for t in (old_logp, adv, ret, old_value))
        base, n6 = w.data_ptr(), self.max_samples * 4      # [logits 2n | value n | dlogits 2n | dvalue n] carved from one buffer
        logits, value, dlogits, dvalue = base, base + 2 * n6, base + 3 * n6, base + 5 * n6
        s = self._stream()
        self._chk(self._lib.uavtrain_forward_heads(self._h, p(flat_params), p(obs), n, C.c_void_p(logits), C.c_void_p(value), s))
        self._chk(self._lib.uavtrain_ppo_loss(self._h, C.c_void_p(logits), C.c_void_p(value), p(action), p(old_logp), p(adv), p(ret),
                                              p(old_value), n, float(eps_clip), float(c_value), float(c_entropy),
                                              C.c_void_p(dlogits), C.c_void_p(dvalue), p(stats_out) if stats_out is not None else None, s))
        self._chk(self._lib.uavtrain_backward_heads(self._h, C.c_void_p(dlogits), C.c_void_p(dvalue), p(grad_out), s))
        self._pending = 0
