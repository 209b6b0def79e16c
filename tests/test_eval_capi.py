"""CPU-side checks of the evaluation path: the actor-only forward (include/uavpolicy_eval_b200.h) and the episode
accumulator (uavenv_episode_accumulate) are exported and validate their arguments before touching a GPU; evaluate()
refuses a CPU device; the checkpoint loader takes a module, a state_dict or a path."""
import ctypes as C
import os
import re

import pytest
import torch

from conftest import ROOT

import uavenv_b200 as ub


def _declared(header, prefix):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:%s)_[a-z0-9_]+)\s*\(" % prefix, text)))


def test_policy_library_exports_the_evaluation_header():
    from target_allocation_ppo_transformer_b200 import _capi
    L = _capi.load_policy()
    names = _declared("uavpolicy_eval_b200.h", "uavpolicy")
    assert names == ["uavpolicy_act"]
    for name in names:
        assert hasattr(L, name), "libuavpolicy_b200.so does not export %s" % name


def test_env_library_exports_the_episode_accumulator():
    assert hasattr(ub.load_library(), "uavenv_episode_accumulate")


def test_act_validates_arguments_without_gpu():
    from target_allocation_ppo_transformer_b200 import _capi
    L = _capi.load_policy()
    buf = C.c_void_p(64)              # never dereferenced: validation fails first

    def act(B=8, mode=1, obs=buf, action=buf, h=None):
        return L.uavpolicy_act(h, obs, B, mode, 0, 0, 0, action, None, None, None)

    assert act(B=0) == -1 and b"B=0" in L.uavpolicy_last_error(None)
    assert act(B=-3) == -1
    assert act(mode=2) == -1 and b"mode 2" in L.uavpolicy_last_error(None)
    assert act(mode=-1) == -1
    assert act(action=None) == -1 and b"non-NULL" in L.uavpolicy_last_error(None)
    assert act(obs=None) == -1
    assert act() == -1 and b"handle is NULL" in L.uavpolicy_last_error(None)


def test_episode_accumulate_validates_arguments_without_gpu():
    from target_allocation_ppo_transformer_b200 import _capi
    L = ub.load_library()
    p = 64                            # never dereferenced: validation fails first
    info_fields = [n for n, _ in _capi.UavenvInfo._fields_]
    acc_fields = [n for n, _ in _capi.UavenvEpisodeAcc._fields_]

    def call(B=8, quota=2, actions=p, done=p, records=p, info_null=None, acc_null=None, info=True, acc=True):
        ic = _capi.UavenvInfo(*[None if n == info_null else p for n in info_fields])
        ac = _capi.UavenvEpisodeAcc(*[None if n == acc_null else p for n in acc_fields])
        return L.uavenv_episode_accumulate(B, actions, done, C.byref(ic) if info else None, quota,
                                           C.byref(ac) if acc else None, records, 0, None)

    def rejected(**kw):               # -1, with a message for uavenv_last_error(NULL) that names the function
        assert L.ppo_normalize_advantages(None, 1, None, 0, None) == -1       # another message in between
        rc, msg = call(**kw), L.uavenv_last_error(None)
        return rc == -1 and msg.startswith(b"uavenv_episode_accumulate: ")

    assert rejected(B=0)
    assert rejected(quota=0) and rejected(quota=-1)
    assert rejected(actions=None) and rejected(done=None) and rejected(records=None)
    assert rejected(info=False) and rejected(acc=False)
    for name in info_fields:
        assert rejected(info_null=name), name
    for name in acc_fields:
        assert rejected(acc_null=name), name
    if not torch.cuda.is_available():
        assert call() == -2           # valid arguments: the device is needed
        assert L.uavenv_last_error(None).startswith(b"uavenv_episode_accumulate: cudaSetDevice failed")


def test_evaluate_refuses_a_cpu_device():
    net = ub.TransformerActorCritic()
    with pytest.raises(RuntimeError):
        ub.evaluate(net, num_envs=4, device="cpu")


def test_checkpoint_loader_takes_a_module_a_state_dict_and_a_path(tmp_path):
    torch.manual_seed(0)
    net = ub.TransformerActorCritic()
    assert ub.load_checkpoint(net) is net
    sd = net.state_dict()
    from_sd = ub.load_checkpoint(sd)
    path = tmp_path / "final_model.pth"
    torch.save(sd, path)
    for loaded in (from_sd, ub.load_checkpoint(str(path)), ub.load_checkpoint(path)):
        got = loaded.state_dict()
        assert list(got) == list(sd)
        assert all(torch.equal(got[k], sd[k]) for k in sd)
    bad = dict(sd)
    bad["actor_head.9.weight"] = bad.pop("actor_head.2.weight")
    with pytest.raises(ValueError):
        ub.load_checkpoint(bad)
    with pytest.raises(ValueError):
        ub.load_checkpoint({k: v for k, v in sd.items() if not k.startswith("critic_head")})
    with pytest.raises(TypeError):
        ub.load_checkpoint(torch.nn.Linear(2, 2))
