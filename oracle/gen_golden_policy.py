#!/usr/bin/env python
"""Golden vectors of the reference policy network (networks/transformer_net.py) and PPO maths (agents/ppo.py).
TEST INFRASTRUCTURE ONLY; run in the build container:  python oracle/gen_golden_policy.py
Writes tests/golden/policy_net.npz: the reference TransformerActorCritic's state_dict (seeded init, then perturbed
so that biases / LayerNorm affine terms are non-trivial), a batch of observation windows with realistic padding
patterns, and the reference outputs (logits via evaluate's log-probs, values, entropy); plus the GAE returns /
normalised advantages the reference PPOAgent.update computes on an episodic buffer (ppo.py:77-94)."""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def main():
    _, RefNet = ref_shim.load_agents()
    torch.manual_seed(1234)
    net = RefNet()
    with torch.no_grad():
        for name, p in net.named_parameters():
            if p.dim() == 1:                               # biases, LayerNorm weight/bias: make them non-trivial
                p.add_(0.05 * torch.randn_like(p))
    net.eval()
    g = torch.Generator().manual_seed(7)
    B = 96
    x = torch.rand(B, 5, 14, generator=g)
    x[:, :, 13] = 1.0
    for b in range(B):                                      # episode starts: 0..4 leading zero (padding) rows
        x[b, : (b % 5)] = 0.0
    x[-1] = 0.0                                             # an all-zero window (only the last row is unmasked)
    actions = torch.randint(0, 2, (B,), generator=g)
    with torch.no_grad():
        logp, value, ent = net.evaluate(x, actions)
        xa = net.actor_net(x)[:, -1]
        logits = net.actor_head(xa)
    sd = {k: v.detach().numpy() for k, v in net.state_dict().items()}
    # the encoder layers' uniform draws are redrawn from the seed by tests/helpers.py: only their digests are stored
    drawn = [k for k, v in sd.items() if ".transformer.layers." in k and v.ndim == 2]
    np.savez_compressed(os.path.join(OUT, "policy_net.npz"), obs=x.numpy(), actions=actions.numpy(),
                        logp=logp.numpy(), value=value.numpy(), entropy=ent.numpy(), logits=logits.numpy(),
                        keys=np.array(list(sd.keys())), init_seed=np.int64(1234),
                        **{"p::" + k: v for k, v in sd.items() if k not in drawn},
                        **{"sha256::" + k: np.array(hashlib.sha256(sd[k].tobytes()).hexdigest()) for k in drawn})
    print("policy_net.npz: %d tensors, %d parameters" % (len(sd), sum(v.size for v in sd.values())))
    return sd


def ppo_update_golden(sd):
    """One full-batch PPO update of the UNMODIFIED reference agent (agents/ppo.py:68-181) on a synthetic episodic
    buffer: records the buffer, the losses it returns and the clipped flat gradient of its single minibatch step."""
    PPOAgent, _ = ref_shim.load_agents()
    from configs.config import cfg
    saved = (cfg.BATCH_SIZE, cfg.K_EPOCHS)
    torch.manual_seed(99)
    agent = PPOAgent()
    agent.policy.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})   # initial weights = the network fixture's
    agent.policy_old.load_state_dict(agent.policy.state_dict())
    g = torch.Generator().manual_seed(3)
    T = 192
    obs = torch.rand(T, 5, 14, generator=g); obs[:, :, 13] = 1.0
    done = torch.zeros(T, dtype=torch.bool); done[[60, 130, T - 1]] = True
    start = 0
    for t in range(T):                                   # leading zero rows at episode starts, like the env
        age = t - start
        if age < 4:
            obs[t, : 4 - age] = 0.0
        if done[t]:
            start = t + 1
    rewards = (torch.rand(T, generator=g) * 2 - 0.5).tolist()
    for t in range(T):
        agent.select_action(obs[t].numpy())
        agent.store_transition(rewards[t], bool(done[t]))
    actions = torch.cat(agent.buffer["actions"]).numpy()
    logps = torch.cat(agent.buffer["logprobs"]).numpy()
    values = torch.cat(agent.buffer["values"]).squeeze().numpy()
    captured = {}
    real_clip = torch.nn.utils.clip_grad_norm_

    def spy(params, max_norm):
        params = list(params)
        norm = real_clip(params, max_norm)
        captured["grad"] = torch.cat([p.grad.reshape(-1) for p in params]).numpy().copy()     # after clipping
        captured["norm"] = float(norm)
        return norm

    try:
        cfg.BATCH_SIZE, cfg.K_EPOCHS = T, 1
        torch.nn.utils.clip_grad_norm_ = spy
        out = agent.update()
    finally:
        torch.nn.utils.clip_grad_norm_ = real_clip
        cfg.BATCH_SIZE, cfg.K_EPOCHS = saved
    np.savez_compressed(os.path.join(OUT, "ppo_update.npz"), obs=obs.numpy(), done=done.numpy(),
                        rewards=np.asarray(rewards, np.float32), actions=actions, logps=logps, values=values,
                        grad_clipped_stride5=captured["grad"][::5], grad_norm=np.float64(captured["norm"]),
                        grad_clipped_sumsq=np.float64((captured["grad"].astype(np.float64) ** 2).sum()),
                        loss_actor=np.float64(out["loss_actor"]), loss_critic=np.float64(out["loss_critic"]),
                        entropy=np.float64(out["entropy"]))
    print("ppo_update.npz: T=%d, grad norm %.4f, losses %s" % (T, captured["norm"], out))


if __name__ == "__main__":
    ppo_update_golden(main())
