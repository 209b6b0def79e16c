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


class _PolicyHandle:
    """One handle of the policy library on a CUDA device: created with <_api>_create, every call checked through
    <_api>_last_error, work enqueued on the device's current stream, <_api>_destroy on close.  _api is "uavpolicy"
    (FusedPolicyForward) or "uavtrain" (networks/fused_train.py: FusedTrunks)."""
    _api = None

    def __init__(self, size, device, what):
        self._h = None
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("%s runs on a CUDA device (sm_100a) only" % what)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = _capi.load_policy()
        h = C.c_void_p()
        self._chk(getattr(self._lib, self._api + "_create")(self.device.index, int(size), C.byref(h)))
        self._h = h

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, rc):
        if rc != 0:
            raise _capi.UavenvError(rc, (getattr(self._lib, self._api + "_last_error")(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            getattr(self._lib, self._api + "_destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FusedPolicyForward(_PolicyHandle):
    _api = "uavpolicy"

    def __init__(self, max_batch, device, seed=0, env_id_base=0):
        super().__init__(max_batch, device, "the fused policy forward")
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
