"""Best-of-K allocation: the replicated device-side scene load (uavenv_load_scene_device) against the host load, the
per-group best member (uavenv_group_best) against get_state, the read-out against the reference's golden trajectories,
and ub.allocate end to end (J recomputed from the allocation in fp64, agreement with evaluate / evaluate_baseline /
record_decisions, best-of-K semantics, chunking invariance).  The CPU tests at the end check the arguments without a
GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden_cases
from helpers import config_from_fixture, load_fixture, scene_from_fixture

import uavenv_b200 as ub


def _error_codes():
    text = open(os.path.join(ROOT, "include", "uavenv_b200.h")).read()
    return {name: int(v) for name, v in re.findall(r"\b(UAVENV_E[A-Z]+)\s*=\s*(-?\d+)", text)}


ERR = _error_codes()
CONFIGS = {"30x10": {}, "64x64": {"NUM_UAVS": 64, "NUM_TARGETS": 64},
           "hard_omega05": dict(ub.HARD_MODE, COST_WEIGHT_OMEGA=0.5)}


def _scenes(S, seed, cfg):
    """S generated scenes (host numpy, get_scene() layout)."""
    gen = ub.UAVEnvBatched(S, seed=seed, config=cfg, auto_reset=False)
    gen.reset(full_reset=True)
    sc = gen.get_scene()
    gen.close()
    return sc


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.int64)


def _net(seed=0):
    torch.manual_seed(seed)
    return ub.TransformerActorCritic()


# ---- 1: replicated device load == host load ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONFIGS))
@pytest.mark.parametrize("K", [1, 3, 33])
def test_replicated_load_equals_host_load(name, K):
    """S scenes x K copies: every replica's scene is the source bit for bit, the state is a fresh episode 1, and the
    first windows, the fp64 score matrix and a whole episode under one action stream equal those of envs loaded from the
    host with load_scene."""
    S, cfg = 5, ub.Config(**CONFIGS[name])
    src = _scenes(S, 41, cfg)
    rep = {k: np.repeat(v, K, axis=0) for k, v in src.items()}
    dev = ub.UAVEnvBatched(S * K, seed=3, config=cfg, auto_reset=False)
    host = ub.UAVEnvBatched(S * K, seed=3, config=cfg, auto_reset=False)
    obs_d = dev.load_scene_device({k: torch.as_tensor(v).cuda() for k, v in src.items()}, copies=K).clone()
    obs_h = host.load_scene(rep).clone()
    got = dev.get_scene()
    for k in src:
        assert got[k].dtype == rep[k].dtype and np.array_equal(got[k].view(np.uint8), rep[k].view(np.uint8)), k
    st = dev.get_state()
    assert (st["episode"] == 1).all() and (st["uav_idx"] == 0).all() and (st["target_idx"] == 0).all()
    assert (st["finished"] == 0).all()
    assert torch.equal(obs_d, obs_h) and torch.equal(dev.obs, host.obs)
    for a, b in zip(dev.score_matrix(torch.float64), host.score_matrix(torch.float64)):
        assert torch.equal(a, b)
    for step in range(dev.N * dev.M):
        a = dev.random_actions(step, action_seed=9).clone()
        od, rd, dd, id_ = dev.step(a)
        oh, rh, dh, ih = host.step(a)
        assert torch.equal(od, oh) and torch.equal(rd, rh) and torch.equal(dd, dh), step
        assert torch.equal(id_["reward_f64"], ih["reward_f64"]), step
        if bool(dd.all()):
            break
    assert bool(dev.done.all())
    dev.close()
    host.close()


@pytest.mark.gpu
def test_load_scene_device_offset_range_and_argument_checks():
    """A load into [first_env, ...) leaves the other envs alone; a range outside [0, B), copies <= 0 and a missing
    required array are refused with UAVENV_EINVAL before anything is launched."""
    cfg = ub.Config()
    a, b = _scenes(2, 5, cfg), _scenes(3, 6, cfg)
    from target_allocation_ppo_transformer_b200 import _capi
    env = ub.UAVEnvBatched(10, seed=1, config=cfg, auto_reset=False)
    env.load_scene({k: np.repeat(v[:1], 10, 0) for k, v in a.items()})
    env.load_scene_device(b, copies=2, first_env=3)          # envs 3..8
    got = env.get_scene()
    for k in a:
        assert np.array_equal(got[k][3:9], np.repeat(b[k], 2, 0)), k
        assert np.array_equal(got[k][[0, 1, 2, 9]], np.repeat(a[k][:1], 4, 0)), k
    for kw in ({"copies": 0}, {"copies": -1}, {"first_env": -1}, {"first_env": 5}, {"copies": 4}):
        with pytest.raises(_capi.UavenvError) as exc:
            env.load_scene_device(b, **{"copies": 2, **kw})
        assert exc.value.code == ERR["UAVENV_EINVAL"], kw
    missing = {k: v for k, v in b.items() if k != "tgt_id"}
    with pytest.raises(KeyError):
        env.load_scene_device(missing)
    L = ub.load_library()
    sc = _capi.UavenvScene()                                  # every pointer NULL
    assert L.uavenv_load_scene_device(env._h, C.byref(sc), 1, 1, 0, None, None) == ERR["UAVENV_EINVAL"]
    assert b"NULL" in L.uavenv_last_error(env._h)
    assert np.array_equal(env.get_scene()["uav_x"], got["uav_x"])
    env.close()


# ---- 2: group_best against get_state ----------------------------------------------------------------------------------

def _play_random(env, action_seed=4):
    for step in range(env.N * env.M):
        _, _, done, _ = env.step(env.random_actions(step, action_seed=action_seed))
        if step % 32 == 31 and bool(done.all()):
            break
    assert bool(env.done.all())


def _expect(st, first_env, G, gs):
    """numpy best-of-group from get_state: (best, J, assigned row, N0, J of every member)."""
    J = st["J_val"][first_env:first_env + G * gs].reshape(G, gs)
    best = np.argmax(J, axis=1)                                  # the first maximum: lowest index
    rows = first_env + np.arange(G) * gs + best
    n0 = (st["lock_count"] > 0).sum(1)
    return best, J[np.arange(G), best], st["assigned_target_id"][rows], n0[rows], J


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(30, 10), (64, 8), (256, 3)])
def test_group_best_matches_get_state(n, m):
    """Every env plays one episode of random actions keyed per env (auto_reset=False); for group sizes 1, 7, 32, 33 and 130
    (from env 0 and from env 3) the best member, its J bits, its allocation row, its N0 and every member's J equal a
    numpy arg-max over get_state()."""
    B = 4 * 130 + 3
    env = ub.UAVEnvBatched(B, seed=17, config=ub.Config(NUM_UAVS=n, NUM_TARGETS=m, COST_WEIGHT_OMEGA=0.5,
                                                         RESET_EPISODES=1), auto_reset=False)
    env.reset(full_reset=True)
    _play_random(env)
    st = env.get_state()
    assert st["finished"].all()
    for gs in (1, 7, 32, 33, 130):
        for first in (0, 3):
            G = (B - first) // gs
            got = {k: v.cpu().numpy() for k, v in env.group_best(gs, first_env=first).items()}
            best, J, row, n0, J_all = _expect(st, first, G, gs)
            assert got["best"].shape == (G,)
            assert np.array_equal(got["best"], best), (gs, first)
            assert np.array_equal(_bits(got["J"]), _bits(J)), (gs, first)
            assert np.array_equal(got["assigned_target_id"], row), (gs, first)
            assert np.array_equal(got["num_covered"], n0), (gs, first)
            assert np.array_equal(_bits(got["J_all"]), _bits(J_all)), (gs, first)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["best_target", "skip"])
@pytest.mark.parametrize("gs", [7, 33, 130])
def test_group_best_ties_go_to_member_zero(policy, gs):
    """Each group holds copies of one scene and every member plays the same deterministic stream, so all members tie:
    the group's best is member 0."""
    S, cfg = 3, ub.Config(COST_WEIGHT_OMEGA=0.5)
    env = ub.UAVEnvBatched(S * gs, seed=2, config=cfg, auto_reset=False)
    env.load_scene_device(_scenes(S, 23, cfg), copies=gs)
    skip = torch.zeros(S * gs, dtype=torch.int64, device=env.device)
    for _ in range(env.N * env.M):
        env.step(env.best_target_actions() if policy == "best_target" else skip)
        if bool(env.done.all()):
            break
    got = env.group_best(gs)
    J_all = got["J_all"].cpu().numpy()
    assert (J_all == J_all[:, :1]).all()
    assert (got["best"].cpu().numpy() == 0).all()
    if policy == "skip":
        assert (got["J"].cpu().numpy() == 0.0).all() and (got["assigned_target_id"].cpu().numpy() == -1).all()
    env.close()


@pytest.mark.gpu
def test_group_best_mid_episode_and_state_errors():
    """Mid-episode, a group with an unfinished member reports -1 (J NaN, N0 -1, a row of -1) and a finished group its
    best; an auto-reset handle is UAVENV_ESTATE; NULL outputs and ranges outside [0, B) are UAVENV_EINVAL."""
    from target_allocation_ppo_transformer_b200 import _capi
    B, gs = 256, 2
    env = ub.UAVEnvBatched(B, seed=9, config=ub.Config(NUM_UAVS=6, NUM_TARGETS=4), auto_reset=False)
    env.reset(full_reset=True)
    for step in range(env.N * env.M):               # until the first group has finished
        env.step(env.random_actions(step, action_seed=5))
        st = env.get_state()
        fin = st["finished"].reshape(-1, gs).all(1)
        if fin.any():
            break
    assert fin.any() and not fin.all()
    got = {k: v.cpu().numpy() for k, v in env.group_best(gs).items()}
    assert np.array_equal(got["best"] >= 0, fin)
    assert np.isnan(got["J"][~fin]).all() and (got["num_covered"][~fin] == -1).all()
    assert (got["assigned_target_id"][~fin] == -1).all()
    best, J, row, n0, _ = _expect(st, 0, B // gs, gs)
    assert np.array_equal(got["best"][fin], best[fin]) and np.array_equal(got["assigned_target_id"][fin], row[fin])
    assert np.array_equal(_bits(got["J"][fin]), _bits(J[fin])) and np.array_equal(got["num_covered"][fin], n0[fin])
    L = ub.load_library()
    out = [torch.zeros(B * 8, dtype=torch.int64, device=env.device) for _ in range(5)]
    p = [C.c_void_p(t.data_ptr()) for t in out]
    for args in ((0, 1, 0), (0, 0, 1), (-1, 1, 1), (0, 65, 4), (255, 1, 2), (0, 1, -3)):
        assert L.uavenv_group_best(env._h, *args, *p, None) == ERR["UAVENV_EINVAL"], args
    for i in range(4):
        q = list(p)
        q[i] = None
        assert L.uavenv_group_best(env._h, 0, 1, 1, *q, None) == ERR["UAVENV_EINVAL"], i
        assert b"non-NULL" in L.uavenv_last_error(env._h)
    assert L.uavenv_group_best(env._h, 0, 1, 1, *p[:4], None, None) == 0    # d_J_all may be NULL
    torch.cuda.synchronize()
    env.close()
    auto = ub.UAVEnvBatched(64, seed=9)
    auto.reset(full_reset=True)
    with pytest.raises(_capi.UavenvError) as exc:
        auto.group_best(4)
    assert exc.value.code == ERR["UAVENV_ESTATE"]
    auto.close()


# ---- 3: the read-out is the reference's allocation --------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", golden_cases())
def test_group_best_reads_out_the_reference_allocation(case):
    """A golden trajectory's scene loaded with load_scene_device, its first episode's actions replayed up to the first
    done: group_best(1) returns the reference's assigned row at that step exactly and its J_val to 1e-9."""
    fx = load_fixture(case)
    env = ub.UAVEnvBatched(1, seed=0, config=config_from_fixture(fx), auto_reset=False)
    env.load_scene_device(scene_from_fixture(fx))
    t_done = int(np.nonzero(fx["done"])[0][0])
    for t in range(t_done + 1):
        env.step(torch.full((1,), int(fx["action"][t]), dtype=torch.int64, device=env.device))
    assert bool(env.done[0])
    got = env.group_best(1)
    assert int(got["best"][0]) == 0
    assert np.array_equal(got["assigned_target_id"][0].cpu().numpy(), fx["assigned"][t_done].astype(np.int32))
    J, want = float(got["J"][0]), float(fx["J_val"][t_done])
    assert abs(J - want) <= 1e-9 * max(abs(want), 1e-12), (J, want)
    env.close()


# ---- 4 - 6: ub.allocate -----------------------------------------------------------------------------------------------

def _J_from_allocation(assigned, scene, pf, omega):
    """J of each scene from its allocation in fp64 numpy: sum_j value_j (1 - prod_{i -> j} (1 - p_final[i, j])) - omega *
    sum of the assigned UAVs' costs.  assigned holds Target.id; p_final is in list order."""
    S, N = assigned.shape
    out = np.zeros(S)
    for s in range(S):
        pos = {int(t): j for j, t in enumerate(scene["tgt_id"][s])}
        nh = np.ones(scene["tgt_id"].shape[1])
        cost = 0.0
        for i in range(N):
            if assigned[s, i] >= 0:
                j = pos[int(assigned[s, i])]
                nh[j] *= 1.0 - pf[s, i, j]
                cost += scene["uav_cost"][s, i]
        out[s] = float(np.sum(scene["tgt_value"][s] * (1.0 - nh))) - omega * cost
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["30x10", "hard_omega05"])
def test_allocate_J_equals_J_recomputed_from_the_allocation(name):
    S, K, cfg = 96, 8, ub.Config(**CONFIGS[name])
    scenes = _scenes(S, 61, cfg)
    env = ub.UAVEnvBatched(S, seed=0, config=cfg, auto_reset=False)
    env.load_scene(scenes)
    pf = env.score_matrix(torch.float64)[0].cpu().numpy()
    env.close()
    res = ub.allocate(_net(), scenes=scenes, samples=K, config=cfg)
    assert res["assigned_target_id"].shape == (S, cfg.NUM_UAVS) and res["assigned_target_id"].dtype == np.int32
    want = _J_from_allocation(res["assigned_target_id"], scenes, pf, float(cfg.COST_WEIGHT_OMEGA))
    np.testing.assert_allclose(res["J"], want, rtol=1e-9, atol=1e-12)
    ids = set(np.unique(scenes["tgt_id"]).tolist()) | {-1}
    assert set(np.unique(res["assigned_target_id"]).tolist()) <= ids
    assert (res["num_covered"] == [len(set(r[r >= 0].tolist())) for r in res["assigned_target_id"]]).all()


@pytest.mark.gpu
def test_allocate_agrees_with_evaluate_evaluate_baseline_and_record_decisions():
    """Same seed, generated scenes: greedy allocate's J is evaluate(greedy)'s as float32, sampled K = 1 is
    evaluate(greedy=False)'s, "best_target" is evaluate_baseline's, and the greedy allocation is the set of accepted
    (UAV, target) pairs record_decisions logs on the same scenes."""
    S, seed, net = 384, 33, _net(1)
    greedy = ub.allocate(net, num_scenes=S, seed=seed)
    ev = ub.evaluate(net, num_envs=S, episodes_per_env=1, greedy=True, seed=seed)
    assert np.array_equal(greedy["J"].astype(np.float32), ev["J"][:, 0])
    assert np.array_equal(greedy["num_covered"], ev["num_assigned"][:, 0])
    sampled = ub.allocate(net, num_scenes=S, samples=1, greedy=False, seed=seed)
    ev_s = ub.evaluate(net, num_envs=S, episodes_per_env=1, greedy=False, seed=seed)
    assert np.array_equal(sampled["J"].astype(np.float32), ev_s["J"][:, 0])
    assert not np.array_equal(sampled["J"], greedy["J"])
    bt = ub.allocate("best_target", num_scenes=S, seed=seed)
    ev_bt = ub.evaluate_baseline("best_target", num_envs=S, seed=seed)
    assert np.array_equal(bt["J"].astype(np.float32), ev_bt["J"][:, 0])
    assert np.array_equal(bt["num_covered"], ev_bt["num_assigned"][:, 0])
    # record_decisions on the same scenes (evaluate's first episode), greedy actions of the same network
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    B = 64
    env = ub.UAVEnvBatched(B, seed=seed, config=ub.cfg.copy(RESET_EPISODES=1), auto_reset=False)
    env.reset(full_reset=True)
    fused = FusedPolicyForward(B, env.device, seed=seed)
    fused.sync(net.to(env.device))
    rec = ub.record_decisions(env, lambda obs: fused.act(obs, greedy=True)[0])
    for b in range(B):
        kept = (rec["action"][:, b] == 1) & (rec["accepted"][:, b] == 1)
        logged = set(zip(rec["uav_id"][kept, b].tolist(), rec["target_id"][kept, b].tolist()))
        row = greedy["assigned_target_id"][b]
        assert logged == {(i, int(row[i])) for i in range(len(row)) if row[i] >= 0}, b
    fused.close()
    env.close()


@pytest.mark.gpu
def test_allocate_best_of_K_chunking_and_reproducibility():
    """J is the row maximum of J_samples and best_sample its first arg-max; samples of a scene differ; the output is
    bit-identical when max_envs splits the scenes into uneven chunks (the last one short, max_envs not a multiple of K)
    and between two calls with the same seed."""
    S, K, net = 40, 8, _net(2)
    full = ub.allocate(net, num_scenes=S, samples=K, seed=7)
    assert full["J_samples"].shape == (S, K) and full["best_sample"].dtype == np.int32
    assert np.array_equal(full["J"], full["J_samples"].max(1))
    assert np.array_equal(full["best_sample"], np.argmax(full["J_samples"], axis=1))
    assert (full["J_samples"].max(1) != full["J_samples"].min(1)).any()
    chunked = ub.allocate(net, num_scenes=S, samples=K, seed=7, max_envs=13 * K + 5)     # 13 + 13 + 13 + 1 scenes
    again = ub.allocate(net, num_scenes=S, samples=K, seed=7)
    for other in (chunked, again):
        for k in ("assigned_target_id", "num_covered", "best_sample"):
            assert np.array_equal(full[k], other[k]), k
        for k in ("J", "J_samples"):
            assert np.array_equal(_bits(full[k]), _bits(other[k])), k
    s = full["summary"]
    assert s["samples"] == K and s["scenes"] == S and s["env_steps"] > 0 and s["scenes_per_s"] > 0
    assert s["J_mean"] == pytest.approx(float(full["J"].mean())) and s["J_samples_mean"] <= s["J_mean"]


# ---- CPU ----------------------------------------------------------------------------------------------------------

def test_new_entry_points_are_declared_exported_and_check_arguments_without_gpu():
    from target_allocation_ppo_transformer_b200 import _capi
    L = ub.load_library()
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "uavenv_b200.h")).read(), flags=re.S)
    for name in ("uavenv_load_scene_device", "uavenv_group_best"):
        assert re.search(r"\b%s\s*\(" % name, text) and hasattr(L, name), name
    assert L.uavenv_abi_version() == 2
    p = C.c_void_p(64)                # never dereferenced: validation fails first
    sc = _capi.UavenvScene(*([64] * len(_capi.SCENE_FIELDS)))
    assert L.uavenv_load_scene_device(None, C.byref(sc), 1, 1, 0, None, None) == ERR["UAVENV_EINVAL"]
    assert L.uavenv_load_scene_device(None, None, 1, 1, 0, None, None) == ERR["UAVENV_EINVAL"]
    assert L.uavenv_group_best(None, 0, 1, 1, p, p, p, p, None, None) == ERR["UAVENV_EINVAL"]


def test_allocate_is_a_lazy_export():
    from target_allocation_ppo_transformer_b200 import allocation
    assert ub.allocate is ub.allocate is allocation.allocate


def test_allocate_rejects_bad_argument_combinations():
    net = ub.TransformerActorCritic()
    scenes = {"uav_x": np.zeros((2, 30))}
    for kw in ({"num_scenes": 4, "samples": 2, "greedy": True}, {"num_scenes": 4, "samples": 0},
               {"num_scenes": 4, "samples": 9, "max_envs": 8}, {"scenes": scenes, "num_scenes": 2}, {},
               {"num_scenes": 0}, {"scenes": {"uav_x": np.zeros(7)}}):
        with pytest.raises(ValueError):
            ub.allocate(net, **kw)
    with pytest.raises(ValueError):
        ub.allocate("best_target", num_scenes=4, samples=2)
    with pytest.raises(RuntimeError):
        ub.allocate(net, num_scenes=4, device="cpu")
