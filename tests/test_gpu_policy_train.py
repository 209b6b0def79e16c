"""The hand-written sm_100a forward + backward of the PPO update (csrc/policy_train.cu, policy_wgrad.cu) against
PyTorch autograd on the fp32 mirror network, and against one update of the UNMODIFIED reference agent
(tests/golden/ppo_update.npz).  bf16 operands / fp32 accumulation: tolerances are stated per test."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from helpers import policy_fixture

pytestmark = pytest.mark.gpu


def _cos(a, b):
    return torch.nn.functional.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


@pytest.mark.parametrize("rows,n_out,k_in,ld_x", [(128, 128, 128, 128), (1000, 128, 128, 128), (4099, 384, 128, 128),
                                                  (3000, 256, 128, 640), (5000, 128, 256, 256), (200000, 256, 128, 128)])
def test_tcgen05_weight_gradient_kernel(rows, n_out, k_in, ld_x):
    """dW += dY^T X with both operands read MN-major from row-major activations; ragged tails; strided X; the
    accumulator stays in TMEM across all slabs of a CTA.  fp32 accumulation of exact bf16 products: 1e-5 relative."""
    import uavenv_b200  # noqa: F401
    from target_allocation_ppo_transformer_b200 import _capi
    L = _capi.load_policy()
    g = torch.Generator(device="cuda").manual_seed(rows)
    dy = (torch.randn(rows, n_out, device="cuda", generator=g) * 0.5).bfloat16()
    xfull = (torch.randn(rows, ld_x, device="cuda", generator=g) * 0.5).bfloat16()
    dw = torch.full((n_out, k_in), 0.25, device="cuda")                       # the kernel ACCUMULATES
    db = torch.full((n_out,), -1.0, device="cuda") if k_in == 128 else None   # bias gradient = dY^T 1, same tensor-core pass
    rc = L.uavpolicy_selftest_wgrad(C.c_void_p(dy.data_ptr()), n_out, C.c_void_p(xfull.data_ptr()), ld_x, rows, n_out, k_in,
                                    C.c_void_p(dw.data_ptr()), C.c_void_p(db.data_ptr()) if db is not None else None, None)
    torch.cuda.synchronize()
    assert rc == 0
    ref = dy.double().t() @ xfull[:, :k_in].double() + 0.25
    assert (dw.double() - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    if db is not None:
        ref_b = dy.double().sum(0) - 1.0
        assert (db.double() - ref_b).abs().max().item() <= 1e-5 * max(1.0, ref_b.abs().max().item())


def _perturbed_net(seed=0):
    import uavenv_b200 as ub
    torch.manual_seed(seed)
    net = ub.TransformerActorCritic().cuda()
    with torch.no_grad():                    # biases / LayerNorm parameters start at 0 / 1: make every one of them matter
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    return net


@pytest.mark.parametrize("n", [1000, 4096 + 37])
def test_trunk_features_and_every_parameter_gradient_match_fp32_autograd(n):
    """features: 5e-2 absolute at a scale of ~5 (bf16 activations); gradients, per parameter tensor: relative L2 error
    <= 8e-2 and cosine >= 0.997 (the loosest are linear1.{weight,bias}, where bf16 rounding flips a few ReLU masks;
    everything else is ~1e-2 / 0.9998); parameters the trunks do not own (the heads) get exactly zero from this op."""
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    net = _perturbed_net()
    obs = torch.rand(n, 5, 14, device="cuda")
    obs[: n // 3, :3] = 0                    # padded windows as at the start of an episode
    obs[n // 3: n // 2, :1] = 0
    trunks = FusedTrunks(n, "cuda")
    feat = trunks.features(net, obs)
    ref = torch.stack([net.actor_net.forward_last(obs), net.critic_net.forward_last(obs)], 1)
    assert feat.shape == ref.shape and (feat - ref).abs().max().item() < 5e-2
    dfeat = torch.randn_like(ref) / n
    net.zero_grad()
    feat.backward(dfeat)
    got = {k: p.grad.clone() for k, p in net.named_parameters()}
    net.zero_grad()
    ref.backward(dfeat)
    for k, p in net.named_parameters():
        if "head" in k:
            assert p.grad is None and not got[k].any()
            continue
        rel = ((got[k] - p.grad).norm() / p.grad.norm()).item()
        assert rel <= 8e-2 and _cos(got[k], p.grad) >= 0.997, (k, rel, _cos(got[k], p.grad))


def test_logits_value_and_all_gradients_with_heads_inside():
    """uavtrain_forward_heads / _backward_heads: logits / value within 3e-2 / 5e-2 of the fp32 network.  Through the heads'
    ReLU a bf16 forward flips a few masks, which moves every upstream gradient: PyTorch's own bf16 autocast of the same
    network is the yardstick.  Per parameter tensor: relative L2 error <= 0.15, cosine >= 0.99, and not more than
    1.5x (+1e-2) the error autocast makes on the same inputs."""
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    net = _perturbed_net(2)
    n = 3001
    obs = torch.rand(n, 5, 14, device="cuda")
    obs[: n // 4, :2] = 0
    trunks = FusedTrunks(n, "cuda")
    logits, value = trunks.logits_and_value(net, obs)
    ref_l, ref_v = net.logits_and_value(obs)
    assert logits.shape == (n, 2) and value.shape == (n, 1)
    assert (logits - ref_l).abs().max() < 3e-2 and (value - ref_v).abs().max() < 5e-2
    dl, dv = torch.randn_like(ref_l) / n, torch.randn_like(ref_v) / n

    def grads(fn):
        net.zero_grad()
        l, v = fn()
        torch.autograd.backward([l.float(), v.float()], [dl, dv])
        return {k: p.grad.clone() for k, p in net.named_parameters()}

    def autocast():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return net.logits_and_value(obs)

    ref = grads(lambda: net.logits_and_value(obs))
    got = grads(lambda: trunks.logits_and_value(net, obs))
    lib = grads(autocast)
    for k in ref:
        rel = ((got[k] - ref[k]).norm() / ref[k].norm()).item()
        rel_lib = ((lib[k] - ref[k]).norm() / ref[k].norm()).item()
        assert rel <= 0.15 and _cos(got[k], ref[k]) >= 0.99 and rel <= 1.5 * rel_lib + 1e-2, (k, rel, rel_lib)


def test_evaluate_contract_and_repeatability():
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    net = _perturbed_net(1)
    n = 777
    obs = torch.rand(n, 5, 14, device="cuda")
    act = torch.randint(0, 2, (n,), device="cuda")
    trunks = FusedTrunks(1024, "cuda")
    lp, v, e = trunks.evaluate(net, obs, act)
    lp_ref, v_ref, e_ref = net.evaluate(obs, act)
    assert lp.shape == (n,) and v.shape == (n, 1) and e.shape == (n,)
    assert (lp - lp_ref).abs().max() < 3e-2 and (v - v_ref).abs().max() < 5e-2 and (e - e_ref).abs().max() < 3e-2
    (lp.mean() + v.mean()).backward()
    g1 = torch.cat([p.grad.flatten() for p in net.parameters()])
    net.zero_grad()
    lp2, v2, _ = trunks.evaluate(net, obs, act)
    assert torch.equal(lp, lp2) and torch.equal(v, v2)          # the forward is deterministic
    (lp2.mean() + v2.mean()).backward()
    g2 = torch.cat([p.grad.flatten() for p in net.parameters()])
    assert _cos(g1, g2) > 0.999999                               # backward: fp32 atomics reorder sums, nothing more
    with pytest.raises(Exception):
        trunks.features(net, torch.rand(2048, 5, 14, device="cuda"))   # more windows than the workspace holds


def test_fused_update_against_the_reference_agents_update():
    """Same buffer and initial weights as one update of the unmodified reference agent (ppo_update.npz): losses within
    2e-2 relative / absolute, clipped gradient direction cosine >= 0.99 on the recorded stride-5 sample."""
    import uavenv_b200 as ub
    fx = np.load(os.path.join(GOLDEN, "ppo_update.npz"))
    T = len(fx["rewards"])
    agent = ub.PPOAgent(num_envs=1, horizon=T, device="cuda", cfg=ub.Config(K_EPOCHS=1), minibatch_size=T, update_precision="fused")
    sd = {k: torch.from_numpy(v) for k, v in policy_fixture()[1].items()}
    agent.policy.load_state_dict(sd); agent.policy_old.load_state_dict(sd)
    obs = torch.from_numpy(fx["obs"]).cuda()
    agent.buf_obs.copy_(obs[:, None]); agent.buf_action.copy_(torch.from_numpy(fx["actions"]).cuda()[:, None])
    agent.buf_logp.copy_(torch.from_numpy(fx["logps"]).cuda()[:, None])
    agent.buf_value.copy_(torch.from_numpy(fx["values"]).cuda()[:, None])
    agent.buf_reward.copy_(torch.from_numpy(fx["rewards"]).cuda()[:, None])
    agent.buf_done.copy_(torch.from_numpy(fx["done"]).cuda()[:, None])
    agent.t = T
    out = agent.update(last_obs=obs[-1:].clone())
    assert abs(out["loss_critic"] - float(fx["loss_critic"])) <= 2e-2 * abs(float(fx["loss_critic"]))
    assert abs(out["loss_actor"] - float(fx["loss_actor"])) <= 2e-2
    assert abs(out["entropy"] - float(fx["entropy"])) <= 2e-2
    g = agent._flat_grad.cpu().numpy()[::5].astype(np.float64)
    ref = fx["grad_clipped_stride5"].astype(np.float64)
    assert (g * ref).sum() / np.sqrt((g * g).sum() * (ref * ref).sum()) >= 0.99


def test_fused_update_trains_like_the_tf32_update():
    """Two agents, same seed, same rollout: after one multi-epoch update the reported losses agree and the fused agent's
    parameters moved in the same direction."""
    import uavenv_b200 as ub
    B, T = 512, 16
    agents = [ub.PPOAgent(B, T, "cuda", minibatch_size=2048, seed=3, update_precision=p) for p in ("fused", "tf32")]
    env = ub.UAVEnvBatched(B, seed=1)
    obs = env.reset()
    w0 = torch.cat([p.detach().flatten() for p in agents[0].policy.parameters()]).clone()
    while not agents[1].full():
        a = agents[1].select_action(obs)
        agents[0].buf_obs[agents[0].t].copy_(obs)
        obs, reward, done, _ = env.step(a)
        for ag in agents:
            ag.store_transition(reward, done)
    for name in ("buf_action", "buf_logp", "buf_value"):
        getattr(agents[0], name).copy_(getattr(agents[1], name))
    agents[0]._gen.set_state(agents[1]._gen.get_state())         # same minibatch permutations
    stats = [ag.update(obs) for ag in agents]
    for k in ("loss_actor", "loss_critic", "entropy"):
        assert np.isfinite(stats[0][k]) and abs(stats[0][k] - stats[1][k]) <= 2e-2 * max(1.0, abs(stats[1][k])), (k, stats)
    d = [torch.cat([p.detach().flatten() for p in ag.policy.parameters()]) - w0 for ag in agents]
    assert _cos(d[0], d[1]) > 0.8            # Adam's first steps are sign-like: small gradients may flip, the bulk agrees


def test_graph_replayed_update_matches_the_eager_update():
    """graph_update=True: three eager minibatch steps, then the whole step (gather, forward, loss, backward, clip, Adam) is
    captured once and replayed (77 of the 80 steps here).  Same weights, rollout and permutations => the same losses
    (5e-3: Adam runs with device-side step counters in the captured variant, and fp32 atomics reorder the gradient sums)
    and the same parameter movement (cosine of the deltas)."""
    import uavenv_b200 as ub
    B, T = 256, 16
    agents = [ub.PPOAgent(B, T, "cuda", minibatch_size=256, seed=5, update_precision="fused", graph_update=g) for g in (True, False)]
    env = ub.UAVEnvBatched(B, seed=2)
    obs = env.reset()
    w0 = torch.cat([p.detach().flatten() for p in agents[0].policy.parameters()]).clone()
    while not agents[1].full():
        a = agents[1].select_action(obs)
        agents[0].buf_obs[agents[0].t].copy_(obs)
        obs, reward, done, _ = env.step(a)
        for ag in agents:
            ag.store_transition(reward, done)
    for name in ("buf_action", "buf_logp", "buf_value"):
        getattr(agents[0], name).copy_(getattr(agents[1], name))
    agents[0]._gen.set_state(agents[1]._gen.get_state())         # (sampling the actions advanced agent 1's generator)
    stats = [ag.update(obs) for ag in agents]
    for k in stats[0]:
        assert abs(stats[0][k] - stats[1][k]) <= 5e-3 * max(1.0, abs(stats[1][k])), (k, stats)
    assert agents[0]._graph is not None and agents[1]._graph is None
    d = [torch.cat([p.detach().flatten() for p in ag.policy.parameters()]) - w0 for ag in agents]
    assert _cos(d[0], d[1]) > 0.95
    agents[0].close()
    assert agents[0]._graph is None


@pytest.mark.parametrize("n", [1, 257, 5000])
def test_ppo_loss_kernel_value_and_gradient_match_autograd(n):
    """uavtrain_ppo_loss against the PyTorch expression of agents/ppo.py:126-153 (both value-loss branches are hit by
    scaling old_value): the three statistics to 1e-5, dL/dlogits and dL/dvalue to 1e-6 absolute at a scale of 1/n."""
    import uavenv_b200 as ub
    from target_allocation_ppo_transformer_b200 import _capi
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    L = _capi.load_policy()
    tr = FusedTrunks(8, "cuda")
    g = torch.Generator(device="cuda").manual_seed(n)
    p = lambda t: C.c_void_p(t.data_ptr())
    for spread in (0.05, 1.0):
        logits = torch.randn(n, 2, device="cuda", generator=g).requires_grad_()
        value = torch.randn(n, device="cuda", generator=g).requires_grad_()
        act = torch.randint(0, 2, (n,), device="cuda", generator=g)
        old_logp = torch.log_softmax(logits.detach() + 0.3 * torch.randn(n, 2, device="cuda", generator=g), -1).gather(-1, act[:, None]).squeeze(-1)
        adv = torch.randn(n, device="cuda", generator=g)
        ret = torch.randn(n, device="cuda", generator=g)
        old_v = value.detach() + spread * torch.randn(n, device="cuda", generator=g)
        eps = 0.2
        logp_all = torch.log_softmax(logits, -1)
        logp = logp_all.gather(-1, act[:, None]).squeeze(-1)
        ratio = torch.exp(logp - old_logp)
        la = -torch.min(ratio * adv, torch.clamp(ratio, 1 - eps, 1 + eps) * adv).mean()
        vclip = old_v + torch.clamp(value - old_v, -eps, eps)
        lc = torch.max(((value - ret) ** 2).mean(), ((vclip - ret) ** 2).mean())
        ent = (-(logp_all.exp() * logp_all).sum(-1)).mean()
        (la + 0.5 * lc - 0.01 * ent).backward()
        dl, dv, st = torch.empty(n, 2, device="cuda"), torch.empty(n, device="cuda"), torch.empty(3, device="cuda")
        rc = L.uavtrain_ppo_loss(tr._h, p(logits.detach()), p(value.detach()), p(act), p(old_logp), p(adv), p(ret), p(old_v), n, eps, 0.5, 0.01,
                                 p(dl), p(dv), p(st), None)
        torch.cuda.synchronize()
        assert rc == 0
        ref = torch.stack([la, lc, ent]).detach()
        assert torch.allclose(st, ref, rtol=1e-5, atol=1e-6), (st, ref)
        assert (dl - logits.grad).abs().max().item() <= 1e-6 + 1e-5 / n and (dv - value.grad).abs().max().item() <= 1e-6 + 1e-5 / n
