"""Rollout forward of the policy on the 5th-gen tensor cores (csrc/policy_fused.cu + policy_forward.cu) behind the
`get_action` contract of networks/transformer_net.py:96-122.

    fused = FusedPolicyForward(max_batch, device); fused.sync(policy_old)
    action, logp, value, entropy = fused.get_action(obs, step)
    action, logp = fused.act(obs, step, greedy=True)      # actor only: evaluation

bf16 operands / fp32 accumulation: outputs agree with the fp32 network to ~1e-2 absolute (tested); gradients are
never taken through this path - PPO's update evaluates the network again (networks/fused_train.py or the PyTorch
mirror, by PPOAgent's update_precision)."""
import ctypes as C

import torch

from .. import _capi


def flatten_params(module):
    """A TransformerActorCritic's parameters as the library's flat vector (named_parameters order); differentiable."""
    flat = torch.cat([p.reshape(-1) for p in module.parameters()])
    if flat.numel() != _capi.NUM_PARAMS:
        raise ValueError("expected the %d parameters of TransformerActorCritic" % _capi.NUM_PARAMS)
    return flat


class FusedPolicyForward(_capi.Handle):
    def __init__(self, max_batch, device, seed=0, env_id_base=0):
        super().__init__(_capi.load_policy, "uavpolicy", device, "the fused policy forward")
        self._create(self.device.index, int(max_batch))
        self.max_batch, self.seed, self.env_id_base = int(max_batch), int(seed), int(env_id_base)
        dev = self.device
        self.action = torch.zeros(max_batch, dtype=torch.int64, device=dev)
        self.logp = torch.zeros(max_batch, device=dev)
        self.value = torch.zeros(max_batch, 1, device=dev)
        self.entropy = torch.zeros(max_batch, device=dev)
        self.logits = torch.zeros(max_batch, 2, device=dev)
        self._flat = None

    def sync(self, module):
        """Copy the weights of a TransformerActorCritic (named_parameters order == the reference's state_dict order)."""
        flat = flatten_params(module).detach().float()
        if flat.device != self.device:
            raise ValueError("expected the parameters of TransformerActorCritic on %s" % self.device)
        self._flat = flat
        self._chk(self._lib.uavpolicy_set_weights(self._h, C.c_void_p(flat.data_ptr()), self._stream()))

    def get_action(self, obs, step):
        """(action int64 [B], log_prob [B], value [B,1], entropy [B]); tensors are reused by the next call."""
        B = obs.shape[0]
        obs = obs.contiguous()
        self._chk(self._lib.uavpolicy_get_action(
            self._h, C.c_void_p(obs.data_ptr()), B, self.seed, int(step), self.env_id_base,
            C.c_void_p(self.action.data_ptr()), C.c_void_p(self.logp.data_ptr()), C.c_void_p(self.value.data_ptr()),
            C.c_void_p(self.entropy.data_ptr()), C.c_void_p(self.logits.data_ptr()), self._stream()))
        return self.action[:B], self.logp[:B], self.value[:B], self.entropy[:B]

    def act(self, obs, step=0, greedy=True):
        """(action int64 [B], log_prob [B]) from the actor alone (include/uavpolicy_eval_b200.h): the critic is not run,
        and value / entropy are left as they were.  greedy: argmax of the logits (a tie goes to 0); otherwise a sample
        bit-identical to get_action's for the same (seed, step, env).  self.logits is filled as by get_action."""
        B = obs.shape[0]
        obs = obs.contiguous()
        self._chk(self._lib.uavpolicy_act(
            self._h, C.c_void_p(obs.data_ptr()), B, 1 if greedy else 0, self.seed, int(step), self.env_id_base,
            C.c_void_p(self.action.data_ptr()), C.c_void_p(self.logp.data_ptr()), C.c_void_p(self.logits.data_ptr()),
            self._stream()))
        return self.action[:B], self.logp[:B]
