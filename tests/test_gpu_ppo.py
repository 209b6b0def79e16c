"""Batched PPO agent on the GPU against one full-batch update of the UNMODIFIED reference agent
(tests/golden/ppo_update.npz from oracle/gen_golden_policy.py): same buffer, same initial weights ->
same losses and the same clipped gradient (fp32, 1e-4 relative to the gradient scale)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from helpers import assert_logits_close, policy_fixture

pytestmark = pytest.mark.gpu


def test_single_update_matches_reference_agent():
    import uavenv_b200 as ub
    fx = np.load(os.path.join(GOLDEN, "ppo_update.npz"))
    T = len(fx["rewards"])
    cfg = ub.Config(K_EPOCHS=1)
    agent = ub.PPOAgent(num_envs=1, horizon=T, device="cuda", cfg=cfg, minibatch_size=T, update_precision="fp32")
    sd = {k: torch.from_numpy(v) for k, v in policy_fixture()[1].items()}
    agent.policy.load_state_dict(sd); agent.policy_old.load_state_dict(sd)
    obs = torch.from_numpy(fx["obs"]).cuda()
    # the buffer the reference filled (its own sampled actions / log-probs / values, ppo.py:52-66)
    agent.buf_obs.copy_(obs[:, None]); agent.buf_action.copy_(torch.from_numpy(fx["actions"]).cuda()[:, None])
    agent.buf_logp.copy_(torch.from_numpy(fx["logps"]).cuda()[:, None])
    agent.buf_value.copy_(torch.from_numpy(fx["values"]).cuda()[:, None])
    agent.buf_reward.copy_(torch.from_numpy(fx["rewards"]).cuda()[:, None])
    agent.buf_done.copy_(torch.from_numpy(fx["done"]).cuda()[:, None])
    # our own forward of those states reproduces the reference's stored values / log-probs
    with torch.no_grad():
        lp, v, _ = agent.policy.evaluate(obs, agent.buf_action[:, 0])
    assert torch.allclose(lp, agent.buf_logp[:, 0], atol=2e-5) and torch.allclose(v[:, 0], agent.buf_value[:, 0], atol=5e-5)
    agent.t = T
    out = agent.update(last_obs=obs[-1:].clone())        # the buffer ends on a terminal step: bootstrap is masked
    assert abs(out["loss_critic"] - float(fx["loss_critic"])) <= 1e-4 * abs(float(fx["loss_critic"]))
    assert abs(out["loss_actor"] - float(fx["loss_actor"])) <= 1e-5
    assert abs(out["entropy"] - float(fx["entropy"])) <= 1e-5
    g = agent._flat_grad.cpu().numpy()                    # clipped gradient of the single minibatch step
    ref = fx["grad_clipped_stride5"]
    scale = np.abs(ref).max()
    np.testing.assert_allclose(g[::5], ref, rtol=1e-3, atol=1e-4 * scale)
    assert abs((g.astype(np.float64) ** 2).sum() - float(fx["grad_clipped_sumsq"])) <= 1e-3 * float(fx["grad_clipped_sumsq"])


def test_rollout_and_update_run_end_to_end():
    """A short batched rollout + update with the real env (BASELINE.json config 4 shape, scaled down)."""
    import uavenv_b200 as ub
    B, T = 512, 16
    env = ub.UAVEnvBatched(B, seed=1)
    agent = ub.PPOAgent(B, T, "cuda", minibatch_size=2048)
    obs = env.reset()
    w0 = agent.policy.actor_head[2].weight.detach().clone()
    for it in range(2):
        while not agent.full():
            a = agent.select_action(obs)
            obs, reward, done, _ = env.step(a)
            agent.store_transition(reward, done)
        stats = agent.update(obs)
        assert stats is not None and all(np.isfinite(v) for v in stats.values())
        assert 0.0 < stats["entropy"] <= np.log(2.0) + 1e-4
    assert not torch.equal(w0, agent.policy.actor_head[2].weight)
    sd_old, sd_new = agent.policy_old.state_dict(), agent.policy.state_dict()
    assert all(torch.equal(sd_old[k], sd_new[k]) for k in sd_new)          # ppo.py:172
    env.close()


def test_train_loop_logs_reference_columns_and_saves_reference_loadable_checkpoint(tmp_path):
    import csv
    import uavenv_b200 as ub
    from target_allocation_ppo_transformer_b200 import train as tr
    hist = tr.train(num_envs=256, horizon=40, iterations=2, log_dir=str(tmp_path), minibatch_size=4096, verbose=False)
    assert len(hist) == 2 and hist[-1]["samples_per_sec"] > 0 and hist[-1]["Episode"] > 0
    rows = list(csv.reader(open(tmp_path / "training_stats.csv")))
    assert rows[0] == ["Episode", "Avg_Reward", "Avg_Q0", "Avg_J_Value", "Max_Coverage", "Action1_Ratio",      # main_train.py:57-63
                       "Valid_Assign_Rate", "Avg_P_Dmg", "Avg_P_Final", "Loss_Critic", "Loss_Actor", "Entropy"]
    assert np.isfinite(hist[-1]["Avg_Q0"]) and hist[-1]["Max_Coverage"] >= 1
    assert len(rows) == 3
    sd = torch.load(tmp_path / "final_model.pth", map_location="cpu")
    ref = policy_fixture()[1]
    assert list(sd.keys()) == list(ref)                                  # the keys the reference network expects
    assert all(tuple(sd[k].shape) == ref[k].shape for k in ref)


def test_fused_rollout_forward_drives_training():
    """The tcgen05 rollout forward inside the PPO loop: buffers hold its actions / log-probs / values, the update
    runs on the fp32 mirror, the weights are re-synchronised afterwards."""
    import uavenv_b200 as ub
    B, T = 384, 12
    env = ub.UAVEnvBatched(B, seed=2)
    agent = ub.PPOAgent(B, T, "cuda", minibatch_size=1152, fused_rollout=True)
    obs = env.reset()
    while not agent.full():
        a = agent.select_action(obs)
        # log-prob / value stored by the fused forward agree with the fp32 network on the same states
        with torch.no_grad():
            lp, v, _ = agent.policy_old.evaluate(obs, a)
        assert_logits_close(agent.buf_logp[agent.t], lp, agent.policy_old, logprobs=True)
        assert float((v.squeeze(-1) - agent.buf_value[agent.t]).abs().max()) < 5e-2
        obs, reward, done, _ = env.step(a)
        agent.store_transition(reward, done)
    stats = agent.update(obs)
    assert stats is not None and np.isfinite(stats["loss_critic"])
    a2 = agent.select_action(obs)                       # runs with the re-synchronised weights
    assert set(a2.tolist()) <= {0, 1}
    env.close()


@pytest.mark.parametrize("nq", [5, 1])
def test_fused_attention_forward_and_gradients_match_tensor_ops(nq):
    """csrc/ppo_attn.cu against the plain tensor-op attention of the mirror network (fp32, 1e-5)."""
    import uavenv_b200  # noqa: F401
    from target_allocation_ppo_transformer_b200.networks import attn_op
    torch.manual_seed(nq)
    n = 777
    packed = torch.randn(n, 5, 384, device="cuda", requires_grad=True)
    qsrc = torch.randn(n, 1, 128, device="cuda", requires_grad=True)
    pad = torch.rand(n, 5, device="cuda") < 0.3
    pad[:, -1] = False

    def run(fused):
        pk = packed.detach().clone().requires_grad_(True)
        qs = qsrc.detach().clone().requires_grad_(True)
        q = pk[..., :128] if nq == 5 else qs
        k, v = pk[..., 128:256], pk[..., 256:]
        if fused:
            assert attn_op.usable(q, k, v)
            out = attn_op.attention5(q, k, v, pad)
        else:
            qh, kh, vh = (t.reshape(n, -1, 8, 16).transpose(1, 2) for t in (q, k, v))
            sc = (qh @ kh.transpose(-1, -2)) / 4.0
            sc = sc.masked_fill(pad[:, None, None, :], float("-inf"))
            out = (torch.softmax(sc, -1) @ vh).transpose(1, 2).reshape(n, -1, 128)
        w = torch.linspace(-1, 1, out.numel(), device="cuda").view_as(out)
        (out * w).sum().backward()
        return out.detach(), pk.grad, (qs.grad if nq == 1 else None)

    o1, g1, q1 = run(True)
    o0, g0, q0 = run(False)
    assert torch.allclose(o1, o0, rtol=1e-5, atol=1e-6)
    if nq == 5:
        assert torch.allclose(g1, g0, rtol=1e-4, atol=1e-6)
    else:
        assert torch.allclose(g1[..., 128:], g0[..., 128:], rtol=1e-4, atol=1e-6)
        assert torch.allclose(q1, q0, rtol=1e-4, atol=1e-6)


def test_fused_clip_adam_matches_torch_clip_and_adam():
    """csrc/ppo_optim.cu against clip_grad_norm_-style scaling + torch.optim.Adam with the reference's four groups
    (agents/ppo.py:17-22,160-162): same parameters after 5 steps (1e-6), same clipped gradient, same pre-clip norm."""
    import uavenv_b200 as ub
    a = ub.PPOAgent(4, 4, "cuda", seed=5, optimizer="fused")
    b = ub.PPOAgent(4, 4, "cuda", seed=5, optimizer="torch")
    assert torch.equal(a._flat_params, b._flat_params)
    assert a._flat_params.data_ptr() == next(a.policy.parameters()).data_ptr()      # parameters are views of the flat buffer
    g = torch.Generator(device="cuda").manual_seed(3)
    for step in range(5):
        grad = torch.randn(a.num_params, device="cuda", generator=g) * (0.01 if step % 2 else 0.0005)   # clipped and unclipped
        a._flat_grad.copy_(grad); b._flat_grad.copy_(grad)
        a._apply_gradient(); b._apply_gradient()
        assert abs(float(a.grad_norm) - float(grad.norm())) <= 1e-5 * float(grad.norm())
        assert torch.allclose(a._flat_grad, b._flat_grad, rtol=1e-5, atol=1e-9)
        assert torch.allclose(a._flat_params, b._flat_params, rtol=1e-6, atol=2e-7), step
    assert int(a._adam_step) == 5
    # the two learning rates really differ by segment: actor params moved ~5x less than critic params
    w0 = ub.PPOAgent(4, 4, "cuda", seed=5)._flat_params
    moved = (a._flat_params - w0).abs()
    n_actor = sum(p.numel() for p in a.policy.actor_net.parameters()) + sum(p.numel() for p in a.policy.actor_head.parameters())
    assert float(moved[:n_actor].mean()) * 3 < float(moved[n_actor:].mean())
