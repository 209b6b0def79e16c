"""The policy / value network mirror against golden vectors recorded from the reference network
(oracle/gen_golden_policy.py -> tests/golden/policy_net.npz): identical state_dict keys and shapes,
fp32 outputs within 2e-5 (same math, different kernel association)."""
import numpy as np
import torch

from helpers import policy_fixture

import uavenv_b200  # noqa: F401
from target_allocation_ppo_transformer_b200.networks.transformer_net import TransformerActorCritic


def _load():
    fx, sd = policy_fixture()
    return fx, {k: torch.from_numpy(v) for k, v in sd.items()}


def test_state_dict_is_interchangeable_with_the_reference():
    fx, sd = _load()
    net = TransformerActorCritic()
    own = net.state_dict()
    assert list(own.keys()) == [str(k) for k in fx["keys"]]          # same names, same order
    for k, v in own.items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    assert sum(p.numel() for p in net.parameters()) == 419267        # SURVEY.md section 2
    net.load_state_dict(sd, strict=True)


def test_forward_matches_reference_outputs():
    fx, sd = _load()
    net = TransformerActorCritic()
    net.load_state_dict(sd)
    net.eval()
    obs = torch.from_numpy(fx["obs"])
    act = torch.from_numpy(fx["actions"])
    with torch.no_grad():
        logp, value, ent = net.evaluate(obs, act)
        logits, _ = net.logits_and_value(obs)
    np.testing.assert_allclose(logits.numpy(), fx["logits"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(logp.numpy(), fx["logp"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(value.numpy(), fx["value"], rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(ent.numpy(), fx["entropy"], rtol=2e-5, atol=2e-6)


def test_get_action_contract():
    net = TransformerActorCritic()
    obs = torch.rand(7, 5, 14)
    g = torch.Generator().manual_seed(0)
    a, lp, v, e = net.get_action(obs, generator=g)
    assert a.shape == (7,) and a.dtype == torch.int64 and set(a.tolist()) <= {0, 1}
    assert lp.shape == (7,) and v.shape == (7, 1) and e.shape == (7,)      # transformer_net.py:118-122
    lp2, v2, e2 = net.evaluate(obs, a)
    assert torch.allclose(lp, lp2) and torch.allclose(v, v2) and torch.allclose(e, e2)
    a1, _, _, _ = net.get_action(obs[0])                                    # a single [5,14] window (:98)
    assert a1.shape == (1,)


def test_last_token_formulation_equals_full_forward():
    _, sd = _load()
    net = TransformerActorCritic()
    net.load_state_dict(sd)
    x = torch.rand(33, 5, 14)
    x[::3, :2] = 0.0
    with torch.no_grad():
        for block in (net.actor_net, net.critic_net):
            assert torch.allclose(block.forward_last(x), block(x)[:, -1], rtol=1e-5, atol=1e-6)
