"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI,
against (1) golden fixtures recorded from the UNMODIFIED reference and (2) the CPU oracle on the
same seeded inputs.

Bars (BASELINE.json north_star): pointers, assigned_target_id, covered flags, done, N0,
is_valid_action - bit-exact; reward, J_val, avg_p_*, observation rows, scores - 1e-5 relative in
fp32 (the fp64 reward side-channel is held to 1e-9).
"""
import numpy as np
import pytest
import torch

from conftest import golden_cases
from helpers import (config_from_fixture, load_fixture, oracle_cfg_from_config, rel_close, scene_from_fixture)

pytestmark = pytest.mark.gpu

RTOL32 = 1e-5     # tolerance named by north_star for fp32 outputs
ATOL32 = 1e-7     # f32 rows near zero (differences of nearly equal probabilities)


def _ub():
    import uavenv_b200 as ub
    return ub


def _check_step(fx, t, env, obs, reward, done, info, copies, window):
    st = env.get_state()
    for c in range(copies):
        assert st["uav_idx"][c] == fx["uav_idx"][t] and st["target_idx"][c] == fx["target_idx"][t], t
        assert np.array_equal(st["assigned_target_id"][c], fx["assigned"][t].astype(np.int32)), t
        assert np.array_equal(st["lock_count"][c] > 0, fx["covered"][t].astype(bool)), t
    done_h = done.cpu().numpy()
    assert (done_h == bool(fx["done"][t])).all(), t
    assert (info["num_assigned"].cpu().numpy() == fx["num_assigned"][t]).all(), t
    assert (info["is_valid_action"].cpu().numpy() == fx["is_valid"][t]).all(), t
    rel_close(reward.cpu().numpy(), np.full(copies, fx["reward"][t]), RTOL32, 1e-6)
    rel_close(info["reward_f64"].cpu().numpy(), np.full(copies, fx["reward"][t]), 1e-9, 1e-11)
    rel_close(info["J_val"].cpu().numpy(), np.full(copies, fx["J_val"][t]), RTOL32, 1e-6)
    rel_close(info["avg_p_dmg"].cpu().numpy(), np.full(copies, fx["avg_p_dmg"][t]), RTOL32, ATOL32)
    rel_close(info["avg_p_final"].cpu().numpy(), np.full(copies, fx["avg_p_final"][t]), RTOL32, ATOL32)


@pytest.mark.parametrize("case", golden_cases())
def test_golden_trajectory_autoreset(case):
    """Replay the reference's recorded trajectories; episodes chain through the in-kernel
    state-only auto-reset (== the reference's reset(full_reset=False) between episodes)."""
    ub = _ub()
    fx = load_fixture(case)
    copies = 3
    cfg = config_from_fixture(fx, RESET_EPISODES=0)       # never regenerate: the injected scene stays
    env = ub.UAVEnvBatched(copies, config=cfg, auto_reset=True)
    obs = env.load_scene(scene_from_fixture(fx, copies)).cpu().numpy()
    assert not obs[:, :4].any()
    rel_close(obs[:, 4], np.tile(fx["reset_row"][0], (copies, 1)), RTOL32, ATOL32)
    pf, pd = env.score_matrix(torch.float64)
    rel_close(pf.cpu().numpy()[0], fx["p_final"], 1e-9, 1e-14)
    rel_close(pd.cpu().numpy()[0], fx["p_damage"], 1e-9, 1e-14)
    pf32, pd32 = env.score_matrix(torch.float32)
    rel_close(pf32.cpu().numpy()[1], fx["p_final"], RTOL32, 1e-12)
    rel_close(pd32.cpu().numpy()[2], fx["p_damage"], RTOL32, 1e-12)
    T = len(fx["action"])
    window = obs[0].copy()
    for t in range(T):
        a = torch.full((copies,), int(fx["action"][t]), dtype=torch.int64, device=env.device)
        obs, reward, done, info = env.step(a)
        # integer state is read BEFORE the auto-reset only through the outputs; the pointer state
        # after an auto-reset is (0,0) of the next episode, so compare pre-reset values on non-final steps
        if not fx["done"][t]:
            _check_step(fx, t, env, obs, reward, done, info, copies, window)
            o = obs.cpu().numpy()
            for c in range(copies):
                rel_close(o[c, 4], fx["obs_row"][t], RTOL32, ATOL32)
                np.testing.assert_array_equal(o[c, :4], window[1:])     # deque(maxlen=5) shift, bit-exact
            window = o[0].copy()
        else:
            assert done.all()
            assert (info["num_assigned"].cpu().numpy() == fx["num_assigned"][t]).all()
            assert (info["is_valid_action"].cpu().numpy() == fx["is_valid"][t]).all()
            rel_close(reward.cpu().numpy(), np.full(copies, fx["reward"][t]), RTOL32, 1e-6)
            rel_close(info["reward_f64"].cpu().numpy(), np.full(copies, fx["reward"][t]), 1e-9, 1e-11)
            rel_close(info["J_val"].cpu().numpy(), np.full(copies, fx["J_val"][t]), RTOL32, 1e-6)
            st = env.get_state()
            assert (st["uav_idx"] == 0).all() and (st["target_idx"] == 0).all()
            assert (st["assigned_target_id"] == -1).all() and (st["lock_count"] == 0).all()
            ep = int(fx["episode"][t]) + 1
            assert (st["episode"] == ep + 1).all()
            o = obs.cpu().numpy()
            assert not o[:, :4].any()
            if ep < len(fx["reset_row"]):
                rel_close(o[:, 4], np.tile(fx["reset_row"][ep], (copies, 1)), RTOL32, ATOL32)
            window = o[0].copy()
    env.close()


@pytest.mark.parametrize("case", ["traj_default_s0", "traj_omega05_s1", "traj_tiny_4x1_omega", "traj_hard_omega05"])
def test_golden_single_env_dropin(case):
    """UAVEnv (B=1, auto_reset off) with the reference's exact signatures and return types."""
    ub = _ub()
    fx = load_fixture(case)
    env = ub.UAVEnv(config=config_from_fixture(fx))
    obs = env.load_scene(scene_from_fixture(fx))
    assert obs.shape == (5, 14) and obs.dtype == np.float32
    ep_prev = 0
    for t in range(len(fx["action"])):
        if fx["episode"][t] != ep_prev:
            ep_prev = int(fx["episode"][t])
            obs = env.reset(full_reset=False)
            rel_close(obs[4], fx["reset_row"][ep_prev], RTOL32, ATOL32)
        obs, reward, done, info = env.step(int(fx["action"][t]))
        assert isinstance(reward, float) and isinstance(done, bool) and isinstance(info, dict)
        assert done == bool(fx["done"][t])
        assert env.uav_idx == fx["uav_idx"][t] and env.target_idx == fx["target_idx"][t]
        rel_close(reward, fx["reward"][t], 1e-9, 1e-11)
        v = info["is_valid_action"]
        assert (-1 if v is None else int(v)) == fx["is_valid"][t]
        assert info["num_assigned"] == fx["num_assigned"][t]
        if done:
            assert obs.shape == (14,) and not obs.any()                  # uav_env.py:188-189
            with pytest.raises(IndexError):
                env.step(1)                                              # uav_env.py:296
        else:
            rel_close(obs[4], fx["obs_row"][t], RTOL32, ATOL32)
    # entity views (env.uavs / env.targets ...) as main.py / test_visualize.py read them
    uavs, targets = env.uavs, env.targets
    assert [u.assigned_target_id for u in uavs] == list(fx["assigned"][-1])
    assert [len(tg.locked_by_uavs) > 0 for tg in targets] == list(fx["covered"][-1].astype(bool))
    assert [tg.id for tg in targets] == list(fx["tgt_id"])
    assert len(env.nfz_list) == len(fx["nfz_x"]) and len(env.interceptors) == len(fx["int_x"])
    env.close()


def _oracle_envs(cfg, B, seed, base=0):
    from oracle import oracle as orc
    ocfg = oracle_cfg_from_config(cfg)
    envs = []
    for b in range(B):
        e = orc.OracleEnv(ocfg)
        e.generate_scene(seed, base + b, 0)
        envs.append(e)
    return envs


@pytest.mark.parametrize("kw", [dict(), dict(COST_WEIGHT_OMEGA=0.5),
                                dict(NUM_UAVS=12, NUM_TARGETS=7, NUM_NFZ=2, NUM_INTERCEPTORS=2, COST_WEIGHT_OMEGA=0.3),
                                dict(NUM_UAVS=5, NUM_TARGETS=1), dict(NUM_UAVS=3, NUM_TARGETS=2, NUM_NFZ=0,
                                                                     NUM_INTERCEPTORS=0)])
def test_generated_scenes_and_rollout_match_oracle(kw):
    """Counter-RNG scene generation + fused step + in-kernel regeneration (every 2nd episode here)
    against the CPU oracle driven with the same Philox streams and the same Bernoulli actions."""
    ub = _ub()
    from oracle import oracle as orc
    cfg = ub.Config(RESET_EPISODES=2, **kw)
    B, seed, base, steps = 40, 1234, 1000, 260
    env = ub.UAVEnvBatched(B, config=cfg, seed=seed, env_id_base=base)
    obs0 = env.reset(full_reset=True).cpu().numpy()
    oenvs = _oracle_envs(cfg, B, seed, base)
    sc = env.get_scene()
    for b, oe in enumerate(oenvs):
        osc = oe.export_scene()
        for k, v in osc.items():
            if v.dtype == np.int32:
                assert np.array_equal(sc[k][b], v), (k, b)
            else:
                rel_close(sc[k][b], v, 1e-13, 1e-15)
    oobs = [oe.reset() for oe in oenvs]
    rel_close(obs0, np.stack(oobs), RTOL32, ATOL32)
    episode = np.ones(B, np.int64)
    scene_idx = np.zeros(B, np.int64)
    for s in range(steps):
        a = env.random_actions(s, action_seed=7)
        a_host = a.cpu().numpy()
        obs, reward, done, info = env.step(a)
        obs_h, rew_h, done_h = obs.cpu().numpy(), info["reward_f64"].cpu().numpy(), done.cpu().numpy()
        nass, valid = info["num_assigned"].cpu().numpy(), info["is_valid_action"].cpu().numpy()
        jval = info["J_val"].cpu().numpy()
        st = env.get_state()
        for b, oe in enumerate(oenvs):
            assert a_host[b] == orc.random_action(7, s, base + b)
            o_obs, o_r, o_done, o_info = oe.step(int(a_host[b]))
            assert bool(done_h[b]) == o_done, (s, b)
            rel_close(rew_h[b], o_r, 1e-9, 1e-11)
            rel_close(jval[b], o_info["J_val"], RTOL32, 1e-6)
            assert nass[b] == o_info["num_assigned"]
            v = o_info["is_valid_action"]
            assert valid[b] == (-1 if v is None else int(v))
            if o_done:
                episode[b] += 1
                if episode[b] % 2 == 0:                       # main_train.py:79 with RESET_EPISODES = 2
                    scene_idx[b] += 1
                    oe.generate_scene(seed, base + b, int(scene_idx[b]))
                o_obs = oe.reset()
            assert st["uav_idx"][b] == oe.uav_idx and st["target_idx"][b] == oe.target_idx, (s, b)
            assert np.array_equal(st["assigned_target_id"][b], oe.assigned()), (s, b)
            assert np.array_equal(st["lock_count"][b] > 0, oe.covered().astype(bool)), (s, b)
            rel_close(obs_h[b], o_obs, RTOL32, ATOL32)
        assert np.array_equal(st["episode"], episode) and np.array_equal(st["scene_index"], scene_idx + 1)
    assert env.recompute_objective() < 1e-9
    env.close()


def test_philox_blocks_and_action_stream_match_oracle():
    ub = _ub()
    from oracle import oracle as orc
    env = ub.UAVEnvBatched(257, env_id_base=5)
    for step in (0, 1, 2 ** 33 + 5):
        a = env.random_actions(step, action_seed=(9 << 32) | 3).cpu().numpy()
        want = [orc.random_action((9 << 32) | 3, step, 5 + b) for b in range(257)]
        assert a.tolist() == want
    env.close()


def test_step_host_equals_device_step_and_non_binary_actions_skip():
    ub = _ub()
    cfg = ub.Config(COST_WEIGHT_OMEGA=0.5)
    B = 300
    e1, e2 = ub.UAVEnvBatched(B, config=cfg, seed=3), ub.UAVEnvBatched(B, config=cfg, seed=3)
    e1.reset(); e2.reset()
    g = torch.Generator().manual_seed(0)
    for s in range(120):
        a = torch.randint(-2, 4, (B,), generator=g, dtype=torch.int64)   # anything but 1 is Skip (uav_env.py:344)
        a_bin = (a == 1).to(torch.int64)
        o1, r1, d1, _ = e1.step(a_bin.cuda())
        if s % 4 == 0:
            r2, d2 = e2.step_host(a.pin_memory())                 # pinned int64: in place over PCIe (a bulk copy per CTA)
        elif s % 4 == 1:
            r2, d2 = e2.step_host(a.to(torch.int8).pin_memory())  # one byte per action (the 44-env tail CTA: plain loads)
        elif s % 4 == 2:
            odd = torch.zeros(B + 1, dtype=torch.int8).pin_memory()   # a pinned buffer that is not 16 B aligned: plain loads
            odd[1:] = a.to(torch.int8)
            r2, d2 = e2.step_host(odd[1:])
        else:
            r2, d2 = e2.step_host(a.clone(), reward_out=torch.zeros(B), done_out=torch.zeros(B, dtype=torch.uint8))
        assert torch.equal(r1.cpu(), r2) and torch.equal(d1.cpu(), d2.bool())   # pageable: staging copies
        assert torch.equal(o1, e2.obs)
    e1.close(); e2.close()


def test_full_size_properties_and_shard_invariance():
    """BASELINE.json config 2 (4096 envs, 30x10): size-independent properties under auto-reset."""
    ub = _ub()
    B, N, M = 4096, 30, 10
    env = ub.UAVEnvBatched(B, seed=42)
    shard = ub.UAVEnvBatched(512, seed=42, env_id_base=1024)       # envs 1024..1535 of the same job
    env.reset(); shard.reset()
    ret = torch.zeros(B, dtype=torch.float64, device="cuda")
    length = torch.zeros(B, dtype=torch.int64, device="cuda")
    n_eps = 0
    for s in range(700):
        a = env.random_actions(s)
        obs, reward, done, info = env.step(a)
        ret += info["reward_f64"]
        length += 1
        # omega = 0: every Assign is accepted (its marginal gain is >= 0).  is_valid_action is None on Skip and
        # (reward != 0) on Assign (uav_env.py:429): False only when p_final is below the rounding of J
        valid = info["is_valid_action"]
        assert bool(((valid == -1) == (a != 1)).all())
        assert int(((valid == 0) & (a == 1)).sum()) <= 1
        if done.any():
            idx = done.nonzero().squeeze(1)
            J, n0 = info["J_val"][idx].double(), info["num_assigned"][idx].double()
            r_final = torch.where(n0 == M, 2.0 * J, J * n0 / M)            # uav_env.py:287-291
            # telescoping: sum of step rewards == 2 * r(X_final)
            assert torch.allclose(ret[idx], 2.0 * r_final, rtol=2e-6, atol=1e-5)
            assert bool(((length[idx] >= N) & (length[idx] <= N * M)).all())
            n_eps += idx.numel()
            ret[idx] = 0
            length[idx] = 0
        sa = shard.random_actions(s)
        so, sr, sd, _ = shard.step(sa)
        assert torch.equal(so, obs[1024:1536]) and torch.equal(sr, reward[1024:1536]) and torch.equal(sd, done[1024:1536])
    assert n_eps > 4 * B
    assert env.recompute_objective() < 1e-9
    env.close(); shard.close()


@pytest.mark.parametrize("nm,B", [((64, 64), 2048), ((256, 256), 512)])
def test_scaled_scenarios_against_oracle_sample(nm, B):
    """BASELINE.json configs 3 / 5 shapes: a large batch steps on the GPU, a sample of envs is
    checked against the oracle step by step, the rest through the objective re-derivation."""
    ub = _ub()
    from oracle import oracle as orc
    cfg = ub.Config(NUM_UAVS=nm[0], NUM_TARGETS=nm[1], COST_WEIGHT_OMEGA=0.25)
    env = ub.UAVEnvBatched(B, config=cfg, seed=11)
    env.reset()
    sample = [0, 1, B // 2, B - 1]
    ocfg = oracle_cfg_from_config(cfg)
    oenvs = {}
    for b in sample:
        oe = orc.OracleEnv(ocfg)
        oe.generate_scene(11, b, 0)
        oe.reset()
        oenvs[b] = oe
    steps = 150 if nm[0] == 64 else 60
    for s in range(steps):
        a = env.random_actions(s, action_seed=5)
        obs, reward, done, info = env.step(a)
        a_h, r_h, d_h, o_h = a.cpu().numpy(), info["reward_f64"].cpu().numpy(), done.cpu().numpy(), obs.cpu().numpy()
        st = env.get_state()
        for b, oe in oenvs.items():
            o_obs, o_r, o_done, _ = oe.step(int(a_h[b]))
            assert not o_done
            assert bool(d_h[b]) == o_done
            rel_close(r_h[b], o_r, 1e-9, 1e-11)
            assert st["uav_idx"][b] == oe.uav_idx and st["target_idx"][b] == oe.target_idx
            assert np.array_equal(st["assigned_target_id"][b], oe.assigned())
            rel_close(o_h[b], o_obs, RTOL32, ATOL32)
    assert env.recompute_objective() < 1e-9
    env.close()


def test_error_paths():
    ub = _ub()
    from target_allocation_ppo_transformer_b200._capi import UavenvError
    env = ub.UAVEnvBatched(8)
    with pytest.raises(UavenvError):
        env.step(torch.zeros(8, dtype=torch.int64, device="cuda"))       # step before reset
    with pytest.raises(UavenvError):
        env.reset(full_reset=False)                                      # no scene yet
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros(7, dtype=torch.int64, device="cuda"))
    with pytest.raises(KeyError):
        env.load_scene({"uav_x": np.zeros(30)})
    # an env range whose end does not fit int32 (1 + INT32_MAX) is refused, not wrapped into [0, B)
    import ctypes as C
    from target_allocation_ppo_transformer_b200._capi import UavenvScene, UavenvState
    L, einval = env._lib, -1                                             # UAVENV_EINVAL (include/uavenv_b200.h)
    assert L.uavenv_get_scene(env._h, C.byref(UavenvScene()), 1, 2**31 - 1) == einval
    assert L.uavenv_get_state(env._h, C.byref(UavenvState()), 1, 2**31 - 1) == einval
    assert L.uavenv_set_episode_counters(env._h, C.byref(C.c_int32(1)), 1, 2**31 - 1) == einval
    assert b"outside" in L.uavenv_last_error(env._h)
    env.close()


def test_scene_generator_matches_reference_distributions():
    """Counter-RNG scene generator vs the reference's _generate_scene (uav_env.py:65-173): moments recorded from
    400 reference scenes (tests/golden/scene_stats.npz, oracle/gen_golden.py) against 4096 generated scenes,
    plus the exact structural constraints (type counts, value multiset, permutations)."""
    ub = _ub()
    import os
    from conftest import GOLDEN
    ref = np.load(os.path.join(GOLDEN, "scene_stats.npz"))
    B = 4096
    env = ub.UAVEnvBatched(B, seed=7)
    env.reset()
    sc = env.get_scene()
    speed = np.hypot(sc["uav_vx"], sc["uav_vy"])
    heading = np.arctan2(sc["uav_vy"], sc["uav_vx"])
    t2 = sc["uav_type"] == 2
    got = {"uav_x": sc["uav_x"], "uav_y": sc["uav_y"], "speed1": speed[~t2], "speed2": speed[t2], "heading": heading,
           "tgt_x": sc["tgt_x"], "tgt_y": sc["tgt_y"], "tgt_vx": sc["tgt_vx"], "nfz_x": sc["nfz_x"], "int_x": sc["int_x"],
           "int_speed": np.hypot(sc["int_vx"], sc["int_vy"]), "n2": (sc["tgt_value"] == 6.0).sum(1),
           "value_sum": sc["tgt_value"].sum(1), "id_at_0": sc["tgt_id"][:, 0], "type_at_0": sc["uav_type"][:, 0]}
    for k, v in got.items():
        mean, std, lo, hi, n = ref[k]
        v = np.asarray(v, np.float64).reshape(-1)
        # means agree within 5 standard errors of the smaller (reference) sample; spreads within 10 %
        se = std / np.sqrt(n) + std / np.sqrt(v.size) + 1e-12
        assert abs(v.mean() - mean) <= 5 * se + 1e-9, (k, v.mean(), mean)
        if std > 0:
            assert abs(v.std() - std) <= 0.1 * std, (k, v.std(), std)
        span = hi - lo
        assert v.min() >= lo - 0.05 * span - 1e-9 and v.max() <= hi + 0.05 * span + 1e-9, k
    # structure: exactly N//4 type-2 UAVs with cost 1.25 / load 1.0 (uav_env.py:81-102)
    assert (t2.sum(1) == 30 // 4).all()
    assert np.array_equal(sc["uav_cost"][t2], np.full(t2.sum(), 1.25)) and (sc["uav_cost"][~t2] == 1.0).all()
    assert (sc["uav_load"][t2] == 1.0).all() and (sc["uav_load"][~t2] == 0.95).all()
    # values: M//2 fours, one sixteen, n2 in [1, M - M//2 - 1] sixes, the rest eights (uav_env.py:121-129)
    vals = sc["tgt_value"]
    assert ((vals == 4.0).sum(1) == 5).all() and ((vals == 16.0).sum(1) == 1).all()
    n2 = (vals == 6.0).sum(1)
    assert n2.min() >= 1 and n2.max() <= 4 and ((vals == 8.0).sum(1) == 4 - n2).all()
    assert set(np.unique(n2)) == {1, 2, 3, 4}
    # target list is a permutation of the ids (uav_env.py:173), uniformly: every id shows up at position 0
    assert (np.sort(sc["tgt_id"], 1) == np.arange(10)).all()
    assert set(np.unique(sc["tgt_id"][:, 0])) == set(range(10))
    counts = np.bincount(sc["tgt_id"][:, 0], minlength=10)
    assert counts.min() > 0.7 * B / 10 and counts.max() < 1.3 * B / 10
    env.close()


def test_pregenerated_scene_flip_equals_inline_generation():
    """The scheduled regeneration takes the scene from the pre-generation service (slot flip) when it is ready
    and generates it in place otherwise; both must give the same scene, and the same one on any shard."""
    ub = _ub()
    cfg = ub.Config(RESET_EPISODES=1, NUM_UAVS=6, NUM_TARGETS=3)      # regenerate at EVERY episode end: the service
    a = ub.UAVEnvBatched(96, config=cfg, seed=5)                       # is often late -> both paths are exercised
    b = ub.UAVEnvBatched(32, config=cfg, seed=5, env_id_base=32)
    a.reset(); b.reset()
    for s in range(120):
        act = a.random_actions(s, action_seed=3)
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act[32:64].clone())
        assert torch.equal(oa[32:64], ob) and torch.equal(ra[32:64], rb) and torch.equal(da[32:64], db)
    sa, sb = a.get_scene(32, 32), b.get_scene()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    st = a.get_state()
    assert (st["scene_index"] >= 5).all()
    a.close(); b.close()


@pytest.mark.parametrize("name,B,N,M,steps", [("configs[2]", 65536, 64, 64, 330), ("configs[4]", 8192, 256, 256, 620)])
def test_baseline_full_size_properties(name, B, N, M, steps):
    """BASELINE.json's full sizes through size-independent properties: telescoping episode return
    (sum of step rewards == 2 r(X_final)), N <= T <= N*M, omega = 0 => every Assign valid, covered count bounds,
    window shift, objective drift, and agreement of a sample of envs with a small shard of the same job."""
    ub = _ub()
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M)
    env = ub.UAVEnvBatched(B, config=cfg, seed=42)
    lo = B // 2
    shard = ub.UAVEnvBatched(64, config=cfg, seed=42, env_id_base=lo)
    prev = env.reset().clone()
    shard.reset()
    ret = torch.zeros(B, dtype=torch.float64, device="cuda")
    length = torch.zeros(B, dtype=torch.int64, device="cuda")
    finished = 0
    for s in range(steps):
        a = env.random_actions(s)
        obs, reward, done, info = env.step(a)
        ret += info["reward_f64"]
        length += 1
        valid = info["is_valid_action"]
        assert bool(((valid == -1) == (a != 1)).all())
        # accepted with reward == 0 only when the marginal gain is below the rounding of J (vanishing p_final, or a
        # target already saturated by many UAVs): a handful per step at most
        assert int(((valid == 0) & (a == 1)).sum()) <= max(2, B // 100)
        assert bool((info["num_assigned"] >= 0).all()) and bool((info["num_assigned"] <= M).all())
        cont = ~done
        assert torch.equal(obs[cont][:, :4], prev[cont][:, 1:])          # deque(maxlen=5) shift, bit-exact
        assert bool((obs[done][:, :4] == 0).all())                        # fresh window after the auto-reset
        if done.any():
            idx = done.nonzero().squeeze(1)
            J, n0 = info["J_val"][idx].double(), info["num_assigned"][idx].double()
            r_final = torch.where(n0 == M, 2.0 * J, J * n0 / M)
            assert torch.allclose(ret[idx], 2.0 * r_final, rtol=2e-6, atol=1e-4)
            assert bool(((length[idx] >= N) & (length[idx] <= N * M)).all())
            finished += idx.numel()
            ret[idx] = 0
            length[idx] = 0
        prev.copy_(obs)
        so, sr, sd, _ = shard.step(shard.random_actions(s))
        assert torch.equal(so, obs[lo:lo + 64]) and torch.equal(sr, reward[lo:lo + 64]) and torch.equal(sd, done[lo:lo + 64])
    assert finished > 0
    assert env.recompute_objective() < 1e-9
    env.close(); shard.close()


@pytest.mark.parametrize("B", [64, 301])
def test_caller_obs_buffer_through_the_raw_c_abi(B):
    """uavenv_step writes the windows into whatever device buffer the caller passes (include/uavenv_b200.h): through the
    TMA bulk store (aligned tiles) or the plain-store tail (301 envs: the last tile is 13 x 280 B, not a multiple of 16)."""
    ub = _ub()
    import ctypes as C
    cfg = ub.Config(COST_WEIGHT_OMEGA=0.5, RESET_EPISODES=3)
    e1, e2 = ub.UAVEnvBatched(B, config=cfg, seed=11), ub.UAVEnvBatched(B, config=cfg, seed=11)
    e1.reset(); e2.reset()
    mine = torch.full((B, 5, 14), -7.0, device="cuda")
    lib = ub.load_library()
    for s in range(150):
        a = e1.random_actions(s)
        o1, r1, d1, _ = e1.step(a)
        rc = lib.uavenv_step(e2._h, C.c_void_p(a.data_ptr()), C.c_void_p(mine.data_ptr()), C.c_void_p(e2.reward.data_ptr()),
                             C.c_void_p(e2._done_u8.data_ptr()), None, None)
        assert rc == 0
        torch.cuda.synchronize()
        assert torch.equal(mine, o1) and torch.equal(e2.reward, r1)
    e1.close(); e2.close()


@pytest.mark.parametrize("case", ["traj_omega05_s0", "traj_omega05_s1", "traj_omega20_s0", "traj_omega20_s2",
                                  "traj_hard_omega05", "traj_tiny_4x1_omega", "traj_n64m64_omega05", "traj_default_s0"])
def test_exact_resummation_path_reproduces_the_reference_decisions(case):
    """tie_band = 1e30 sends EVERY Assign through exact_rewards (the near-tie path of Eq.21: r(X), r(X') re-summed over
    the targets in the reference's list order, uav_env.py:244-293): pointers / validity / N0 bit-exact, f64 reward 1e-9."""
    ub = _ub()
    fx = load_fixture(case)
    cfg = config_from_fixture(fx, RESET_EPISODES=0)
    env = ub.UAVEnvBatched(2, config=cfg, auto_reset=True, tie_band=1e30)
    env.load_scene(scene_from_fixture(fx, 2))
    for t in range(len(fx["action"])):
        a = torch.full((2,), int(fx["action"][t]), dtype=torch.int64, device=env.device)
        obs, reward, done, info = env.step(a)
        assert (done.cpu().numpy() == bool(fx["done"][t])).all(), t
        assert (info["num_assigned"].cpu().numpy() == fx["num_assigned"][t]).all(), t
        assert (info["is_valid_action"].cpu().numpy() == fx["is_valid"][t]).all(), t
        rel_close(info["reward_f64"].cpu().numpy(), np.full(2, fx["reward"][t]), 1e-9, 1e-11)
        if not fx["done"][t]:
            st = env.get_state()
            assert (st["uav_idx"] == fx["uav_idx"][t]).all() and (st["target_idx"] == fx["target_idx"][t]).all(), t
            assert np.array_equal(st["assigned_target_id"][0], fx["assigned"][t].astype(np.int32)), t
    env.close()


@pytest.mark.parametrize("N,M,omega,steps", [(30, 10, 0.5, 420), (30, 10, 2.0, 420), (64, 64, 0.5, 500), (64, 64, 2.0, 500)])
def test_decisions_match_the_oracle_at_scale_with_rollbacks(N, M, omega, steps):
    """Bound on the decision-flip rate at omega > 0 (rollbacks are common, near-ties exist): 4096 envs x `steps` steps
    (several full episodes each, scenes regenerated on schedule) against the OpenMP oracle with the same Philox scenes and
    the same Bernoulli actions - ZERO mismatches in pointers, done, N0, is_valid_action on every step and in
    assigned_target_id (checked every 25 steps and at the end); f64 rewards within 1e-9."""
    ub = _ub()
    from oracle import oracle as orc
    B, seed = 4096, 77
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega, RESET_EPISODES=3)
    env = ub.UAVEnvBatched(B, config=cfg, seed=seed)
    env.reset()
    ob = orc.OracleBatch(oracle_cfg_from_config(cfg), B, seed=seed, reset_episodes=3, threads=orc.max_threads())
    n_done = n_rejected = 0
    for s in range(steps):
        a = env.random_actions(s, action_seed=5)
        obs, reward, done, info = env.step(a)
        a_h = a.cpu().numpy()
        o_r, o_done, o_n0, o_valid, o_k, o_m = ob.step_actions(a_h)
        st = env.get_state()
        assert np.array_equal(done.cpu().numpy(), o_done.astype(bool)), s
        assert np.array_equal(info["num_assigned"].cpu().numpy(), o_n0), s
        assert np.array_equal(info["is_valid_action"].cpu().numpy().astype(np.int32), o_valid), s
        assert np.array_equal(st["uav_idx"], o_k) and np.array_equal(st["target_idx"], o_m), s
        rel_close(info["reward_f64"].cpu().numpy(), o_r, 1e-9, 1e-10)
        n_done += int(o_done.sum()); n_rejected += int((o_valid == 0).sum())
        if s % 25 == 24 or s == steps - 1:
            assert np.array_equal(st["assigned_target_id"], ob.assigned(N)), s
    assert n_rejected > B and n_done >= (B if M == 10 else 0)      # rollbacks really happened; episodes really ended
    ob.close(); env.close()


def test_episode_tags_across_wipe_and_wrap_boundaries():
    """A restart leaves the allocation arrays alone: target records carry an 18-bit episode tag and are wiped every 2^16-th
    episode.  Envs whose counters start just below 65536 and 262144 (set right after the reset) must stay identical to the
    oracle while they cross both boundaries - pointers, assignments, covered flags, rewards, windows."""
    ub = _ub()
    from oracle import oracle as orc
    B, seed = 96, 9
    cfg = ub.Config(NUM_UAVS=5, NUM_TARGETS=3, COST_WEIGHT_OMEGA=0.3, RESET_EPISODES=0)   # the scene stays: no schedule to align
    env = ub.UAVEnvBatched(B, config=cfg, seed=seed)
    obs = env.reset()
    start = np.where(np.arange(B) % 3 == 0, 65530, np.where(np.arange(B) % 3 == 1, 262138, 1)).astype(np.int32)
    env.set_episode_counters(start)
    oenvs = _oracle_envs(cfg, B, seed)
    for oe in oenvs:
        oe.reset()
    n_done = np.zeros(B, np.int64)
    for s in range(400):
        a = env.random_actions(s, action_seed=3)
        a_h = a.cpu().numpy()
        obs, reward, done, info = env.step(a)
        o_h, r_h, d_h = obs.cpu().numpy(), info["reward_f64"].cpu().numpy(), done.cpu().numpy()
        st = env.get_state()
        for b, oe in enumerate(oenvs):
            o_obs, o_r, o_done, o_info = oe.step(int(a_h[b]))
            assert bool(d_h[b]) == o_done, (s, b)
            rel_close(r_h[b], o_r, 1e-9, 1e-11)
            if o_done:
                n_done[b] += 1
                o_obs = oe.reset()
            assert st["uav_idx"][b] == oe.uav_idx and st["target_idx"][b] == oe.target_idx, (s, b)
            assert np.array_equal(st["assigned_target_id"][b], oe.assigned()), (s, b)
            assert np.array_equal(st["lock_count"][b] > 0, oe.covered().astype(bool)), (s, b)
            rel_close(o_h[b], o_obs, RTOL32, ATOL32)
        assert np.array_equal(st["episode"], start + n_done)
    assert n_done.min() >= 20                                   # every env crossed its boundary (6 and 10 episodes away)
    assert env.recompute_objective() < 1e-9
    env.close()
