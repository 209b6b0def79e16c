"""Evaluation path on the GPU: the actor-only forward against get_action and the fp32 network, the episode accumulator
against an independent torch loop, and ub.evaluate end to end (known policy, determinism, shard invariance, scene
pairing across checkpoints, two NCCL ranks).  Weights: tests/golden/policy_net.npz."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from helpers import LOGIT_TOL, assert_logits_close, logit_spread, policy_fixture

import uavenv_b200 as ub

pytestmark = pytest.mark.gpu

KEYS = ("return", "J", "num_assigned", "coverage", "length", "assigns", "valid", "avg_p_dmg", "avg_p_final")


def _net():
    fx, sd = policy_fixture()
    net = ub.TransformerActorCritic().cuda()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return net.eval(), fx


def _windows(B, seed):
    """Random windows with 0..4 leading padding rows (episode starts)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.rand(B, 5, 14, device="cuda", generator=g)
    obs[:, :, 13] = 1.0
    lead = torch.arange(B, device="cuda") % 5
    obs[torch.arange(5, device="cuda")[None, :] < lead[:, None]] = 0.0
    return obs


def _assert_same_records(a, b):
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


# ---- 1-3: the actor-only forward ------------------------------------------------------------------------------------

def test_act_matches_get_action_bit_for_bit():
    """Sizes around the work-item structure switches of the fused kernels, with ragged tails and padded rows.  Before every
    act call a full forward of OTHER windows overwrites the head-hidden rows of every sample, so act can only match if its
    own actor-only launches computed every row; act's logits are also checked against the fp32 network."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    fused = FusedPolicyForward(16500, "cuda", seed=11, env_id_base=5)
    fused.sync(net)
    decoy = _windows(16500, 99)
    for B in (1, 7, 26, 129, 3699, 3700, 7437, 16384, 16500):
        obs = _windows(B, B)
        out = {}
        for greedy in (False, True):
            fused.get_action(decoy, step=8)                              # head-hidden rows of other windows
            decoy_logits = fused.logits[:B].clone()
            a, lp = fused.act(obs, step=3, greedy=greedy)
            out[greedy] = (a.clone(), lp.clone(), fused.logits[:B].clone())
            assert not torch.equal(out[greedy][2], decoy_logits), B
        a_ref, lp_ref, _, _ = (t.clone() for t in fused.get_action(obs, step=3))
        logits_ref = fused.logits[:B].clone()
        a, lp, logits = out[False]                                          # sampled: everything bit-identical
        assert torch.equal(logits, logits_ref), B
        assert torch.equal(a, a_ref) and torch.equal(lp, lp_ref), B
        a, lp, logits = out[True]                                           # greedy: the same logits, their argmax
        assert torch.equal(logits, logits_ref), B
        assert torch.equal(a, (logits[:, 1] > logits[:, 0]).long()), B
        assert torch.allclose(lp, torch.log_softmax(logits, -1).gather(-1, a[:, None]).squeeze(-1), atol=1e-5), B
        with torch.no_grad():
            ref_logits, _ = net.logits_and_value(obs)
        assert_logits_close(logits, ref_logits, net, note=" B=%d" % B)
    fused.close()


def test_greedy_tie_goes_to_action_zero():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    with torch.no_grad():
        net.actor_head[2].weight.zero_()
        net.actor_head[2].bias.fill_(0.25)
    fused = FusedPolicyForward(1000, "cuda")
    fused.sync(net)
    a, _ = fused.act(_windows(1000, 3), greedy=True)
    assert torch.equal(fused.logits[:1000, 0], fused.logits[:1000, 1])
    assert int(a.sum()) == 0
    fused.close()


def test_greedy_matches_argmax_of_the_fp32_network():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, fx = _net()
    obs = torch.from_numpy(fx["obs"]).cuda()
    B = obs.shape[0]
    fused = FusedPolicyForward(B, "cuda")
    fused.sync(net)
    # the gap l1 - l0 of the golden network is mostly its bias b2 (the last layer has std 0.01): centre it on these
    # windows, so that the argmax is decided by what the trunk makes of each window
    with torch.no_grad():
        gap = torch.diff(net.logits_and_value(obs)[0], dim=-1)[:, 0]
        net.actor_head[2].bias[1] -= gap.median()
        ref_logits, _ = net.logits_and_value(obs)
    fused.sync(net)
    a, _ = fused.act(obs, greedy=True)
    gap = ref_logits[:, 1] - ref_logits[:, 0]
    margin = gap.abs() > 2 * LOGIT_TOL * logit_spread(net)     # the largest error of the gap that the logit check allows
    ref_a = ref_logits.argmax(-1)
    assert int(margin.sum()) > B // 5 and set(ref_a[margin].tolist()) == {0, 1}
    assert torch.equal(a[margin], ref_a[margin])
    with torch.no_grad():                                       # an actor with a zero trunk output takes one action
        zero_a = net.actor_head(torch.zeros(B, 128, device="cuda")).argmax(-1)
    assert not torch.equal(zero_a[margin], ref_a[margin])
    fused.close()


def test_act_is_bit_reproducible():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    B = 15013
    fused = FusedPolicyForward(B, "cuda", seed=4)
    fused.sync(net)
    obs = _windows(B, 5)
    for greedy in (True, False):
        a0, lp0 = (t.clone() for t in fused.act(obs, step=1, greedy=greedy))
        l0 = fused.logits[:B].clone()
        for _ in range(10):
            a, lp = fused.act(obs, step=1, greedy=greedy)
            assert torch.equal(a, a0) and torch.equal(lp, lp0) and torch.equal(fused.logits[:B], l0)
    fused.close()


# ---- 4: the accumulator ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,m", [(30, 10), (64, 64)])
def test_accumulator_matches_an_independent_torch_loop(n, m):
    B, quota = 512, 3
    cfg = ub.Config(NUM_UAVS=n, NUM_TARGETS=m, RESET_EPISODES=1)
    env = ub.UAVEnvBatched(B, seed=9, config=cfg)
    rec = ub.EpisodeRecorder(env, quota)
    dev = env.device
    ret = torch.zeros(B, dtype=torch.float64, device=dev)
    length, assigns, valid, episodes = (torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(4))
    ref = {k: torch.zeros(B, quota, dtype=torch.float64, device=dev) for k in
           ("return", "J", "num_assigned", "length", "assigns", "valid", "avg_p_dmg", "avg_p_final")}
    env.reset(full_reset=True)
    step = 0
    while step < quota * n * m:
        a = env.random_actions(step, action_seed=2)
        _, _, done, info = env.step(a)
        rec.record(a)
        step += 1
        ret += info["reward_f64"]                                         # fp64, in step order
        length += 1
        assigns += (a == 1).long()
        valid += (info["is_valid_action"] == 1).long()
        fin = done & (episodes < quota)
        idx = fin.nonzero().squeeze(-1)
        k = episodes[idx]
        for key, val in (("return", ret), ("J", info["J_val"]), ("num_assigned", info["num_assigned"]), ("length", length),
                         ("assigns", assigns), ("valid", valid), ("avg_p_dmg", info["avg_p_dmg"]),
                         ("avg_p_final", info["avg_p_final"])):
            ref[key][idx, k] = val[idx].double()
        episodes += fin.long()
        for t in (ret, length, assigns, valid):
            t.masked_fill_(done, 0)
        if step % 32 == 0 and int(episodes.min()) == quota:
            break
    assert int(episodes.min()) == quota
    got = rec.records()
    assert rec.complete() == B
    assert (got["length"] > 0).all()                                      # exactly `quota` records per env
    for key in ("return", "num_assigned", "length", "assigns", "valid"):
        assert np.array_equal(got[key].astype(np.float64), ref[key].cpu().numpy()), key
    for key in ("J", "avg_p_dmg", "avg_p_final"):                          # float32 copied: equal
        assert np.array_equal(got[key], ref[key].float().cpu().numpy()), key
    env.close()


# ---- 5-6: evaluate end to end -----------------------------------------------------------------------------------------

def test_evaluate_with_an_always_assign_policy_matches_a_direct_run():
    net, _ = _net()
    with torch.no_grad():
        net.actor_head[2].bias.copy_(torch.tensor([-20.0, 20.0]))      # greedy always assigns
    B, quota, seed = 1024, 2, 77
    res = ub.evaluate(net, num_envs=B, episodes_per_env=quota, greedy=True, seed=seed)
    env = ub.UAVEnvBatched(B, seed=seed, config=ub.cfg.copy(RESET_EPISODES=1), env_id_base=0)
    rec = ub.EpisodeRecorder(env, quota)
    ones = torch.ones(B, dtype=torch.int64, device=env.device)
    env.reset(full_reset=True)
    for _ in range(quota * env.N * env.M):
        env.step(ones)
        rec.record(ones)
    assert rec.complete() == B
    direct = rec.records()
    _assert_same_records(res, direct)
    N, M = env.N, env.M
    assert res["length"].shape == (B, quota)
    assert ((res["length"] >= N) & (res["length"] <= N * M)).all()
    assert (res["valid"] <= res["assigns"]).all() and (res["num_assigned"] <= M).all()
    assert (res["valid"] == res["assigns"]).all()                          # omega = 0 (DESIGN section 5)
    s = res["summary"]
    assert s["episodes"] == B * quota and s["valid_assign_rate"] == 1.0
    assert s["J_mean"] == pytest.approx(float(res["J"].astype(np.float64).mean()))
    env.close()


def test_evaluate_leaves_the_callers_module_where_it_is():
    net, _ = _net()
    net = net.cpu()
    before = {k: v.clone() for k, v in net.state_dict().items()}
    res = ub.evaluate(net, num_envs=64, greedy=True, seed=3)
    assert all(p.device.type == "cpu" for p in net.parameters())
    assert all(torch.equal(v, before[k]) for k, v in net.state_dict().items())
    _assert_same_records(res, ub.evaluate({k: v for k, v in before.items()}, num_envs=64, greedy=True, seed=3))


def test_evaluate_is_deterministic_and_shard_invariant():
    net, _ = _net()
    for greedy in (True, False):
        full = ub.evaluate(net, num_envs=2048, episodes_per_env=2, greedy=greedy, seed=5)
        if greedy:
            _assert_same_records(full, ub.evaluate(net, num_envs=2048, episodes_per_env=2, greedy=True, seed=5))
        lo = ub.evaluate(net, num_envs=1024, episodes_per_env=2, greedy=greedy, seed=5, env_id_base=0)
        hi = ub.evaluate(net, num_envs=1024, episodes_per_env=2, greedy=greedy, seed=5, env_id_base=1024)
        _assert_same_records(full, {k: np.concatenate([lo[k], hi[k]]) for k in KEYS})


def test_two_checkpoints_play_the_same_scenes():
    """Scenes are keyed (seed, global env id, scene index): the same first scenes after the reset, and exactly one new
    scene per finished episode, whatever the policy does."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net_a, _ = _net()
    net_b, _ = _net()
    with torch.no_grad():
        net_b.actor_head[2].bias.copy_(torch.tensor([-20.0, 20.0]))
    B, cfg = 64, ub.cfg.copy(RESET_EPISODES=1)
    runs = []
    for net in (net_a, net_b):
        env = ub.UAVEnvBatched(B, seed=123, config=cfg)
        fused = FusedPolicyForward(B, "cuda", seed=123)
        fused.sync(net)
        runs.append((env, fused, env.reset(full_reset=True)))
    sa, sb = runs[0][0].get_scene(), runs[1][0].get_scene()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    dones = []
    for env, fused, obs in runs:
        scene = env.get_state()["scene_index"].copy()
        n_done = 0
        for step in range(200):
            a, _ = fused.act(obs, step, greedy=True)
            obs, _, done, _ = env.step(a)
            d = done.cpu().numpy()
            now = env.get_state()["scene_index"]
            assert np.array_equal(now, scene + d), step
            scene, n_done = now.copy(), n_done + int(d.sum())
        dones.append(n_done)
        fused.close()
        env.close()
    assert min(dones) > 0


# ---- 7: two NCCL ranks ------------------------------------------------------------------------------------------------

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_rank_evaluation_gathers_the_single_gpu_records():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (NCCL refuses two ranks on one device)")
    port = _free_port()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "eval_ddp_worker.py")], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for rank, (p, out) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, out
        assert "rank %d ok" % rank in out
