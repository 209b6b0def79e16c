"""Evaluation baselines: the best-target heuristic's kernel (uavenv_best_target_actions) against an fp64 numpy reference
computed before every step from the env's score matrix and state, its per-row cache across auto-resets, reset(),
load_scene() and skipped calls, its episodes replayed on the C oracle, and ub.evaluate_baseline end to end.  The CPU
tests at the end check the arguments without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from helpers import oracle_cfg_from_config

import uavenv_b200 as ub

KEYS = ("return", "J", "num_assigned", "coverage", "length", "assigns", "valid", "avg_p_dmg", "avg_p_final")
NEAR = 1e-12          # relative gap below which two fp64 rewards are a tie the carried and the fresh sums may order apart


def _error_codes():
    """UAVENV_* return codes as include/uavenv_b200.h defines them."""
    text = open(os.path.join(ROOT, "include", "uavenv_b200.h")).read()
    return {name: int(v) for name, v in re.findall(r"\b(UAVENV_E[A-Z]+)\s*=\s*(-?\d+)", text)}


ERR = _error_codes()


def _paper_reward(J, n0, M):
    return np.where(n0 == M, 2.0 * J, J * (n0 / float(M)))


def _fold(x):
    """Sum over the last axis in index order, one running fp64 sum (the reference's _calc_J_X loop)."""
    return np.cumsum(x, axis=-1)[..., -1]


class Reference:
    """The heuristic's action of every env from env.score_matrix(float64) and env.get_state(), in numpy fp64.  Pair scores
    are constant over an episode (nothing moves), so they are re-read only when the scene of a watched env changes, and
    on refresh() (a load_scene keeps the scene index)."""

    def __init__(self, env):
        self.env, self.omega, self.N, self.M = env, float(env.cfg.COST_WEIGHT_OMEGA), env.N, env.M
        self.scene_index = None

    def refresh(self):
        self.pf = self.env.score_matrix(torch.float64)[0].cpu().numpy()
        sc = self.env.get_scene()
        self.value, self.cost = sc["tgt_value"], sc["uav_cost"]
        self.scene_index = self.env.get_state()["scene_index"].copy()

    def __call__(self, watch):
        """(action [B], near-tie flag [B], accept-margin tie flag [B], j* [B], state)."""
        st = self.env.get_state()
        if self.scene_index is None or not np.array_equal(st["scene_index"][watch], self.scene_index[watch]):
            self.refresh()
        B, N, M, w = self.env.num_envs, self.N, self.M, self.omega
        ar = np.arange(B)
        k, m = st["uav_idx"], st["target_idx"]
        active = (k < N) & (st["finished"] == 0)
        kk = np.minimum(k, N - 1)
        nh, cnt = st["not_hit"], st["lock_count"]
        terms = (1.0 - nh) * self.value
        rev = _fold(terms)
        cost_sum = _fold(np.where(st["assigned_target_id"] >= 0, self.cost, 0.0))
        n0 = (cnt > 0).sum(1)
        prev_r = _paper_reward(rev - w * cost_sum, n0, M)
        nh2 = nh * (1.0 - self.pf[ar, kk])                                   # [B, M]
        rows = np.repeat(terms[:, None, :], M, axis=1)                       # row j: target j's term replaced
        rows[:, np.arange(M), np.arange(M)] = (1.0 - nh2) * self.value
        new_r = _paper_reward(_fold(rows) - w * (cost_sum + self.cost[ar, kk])[:, None], n0[:, None] + (cnt == 0), M)
        jstar = np.argmax(new_r, axis=1)                                      # the first maximum: lowest index
        top = np.sort(new_r, axis=1)
        best, second = top[:, -1], top[:, -2]
        near = (best - second) <= NEAR * np.maximum(np.abs(best), np.abs(second))
        # the accept test new_r(j*) >= prev_r on the carried sums can differ from the fresh ones only inside the tie band,
        # and only with a cost term: at omega = 0 both sides grow monotonically and it always holds
        near_accept = (w != 0.0) & (np.abs(best - prev_r) <= NEAR * np.maximum(np.abs(best), np.abs(prev_r)))
        action = (active & (m == jstar) & (best >= prev_r)).astype(np.int64)
        return action, active & near, active & near_accept & ~near, jstar, st


class Checker:
    """Runs the env with the kernel's actions (or random ones on chosen steps) and compares every kernel call with the
    reference on the watched envs (default: all); counts the env-steps excluded as near-ties."""

    def __init__(self, env):
        self.env, self.ref = env, Reference(env)
        self.calls = self.assigns = self.near = self.near_accept = 0

    def kernel_step(self, watch=None):
        watch = np.ones(self.env.num_envs, bool) if watch is None else watch
        want, near, near_accept, jstar, st = self.ref(watch)
        near, near_accept = near & watch, near_accept & watch
        got = self.env.best_target_actions().cpu().numpy()
        ok = watch & ~(near | near_accept)
        bad = np.nonzero(ok & (got != want))[0]
        assert bad.size == 0, ("kernel != reference", bad[:8], got[bad[:8]], want[bad[:8]], st["uav_idx"][bad[:8]],
                               st["target_idx"][bad[:8]], jstar[bad[:8]])
        self.calls += 1
        self.assigns += int(got.sum())
        self.near += int(near.sum())
        self.near_accept += int(near_accept.sum())
        return self.env.step(self.env._actions), got, jstar, near, st

    def random_step(self, step):
        return self.env.step(self.env.random_actions(step, action_seed=3))

    def report(self, note):
        print("\n[best_target %s] %d calls, %d assigns, near-ties excluded: %d (top two), %d (accept margin)" % (
            note, self.calls, self.assigns, self.near, self.near_accept))
        assert self.assigns > 0


# ---- 1: decisions against the fp64 reference ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n,m,omega,episodes", [(30, 10, 0.0, 3), (30, 10, 0.5, 3), (64, 64, 2.0, 1), (4, 3, 0.5, 20)])
def test_best_target_matches_the_fp64_reference_every_step(n, m, omega, episodes):
    """512 envs, RESET_EPISODES = 1 (every episode a new scene): each env is compared until it has finished `episodes`
    episodes."""
    B = 512
    env = ub.UAVEnvBatched(B, seed=31, config=ub.Config(NUM_UAVS=n, NUM_TARGETS=m, COST_WEIGHT_OMEGA=omega, RESET_EPISODES=1))
    env.reset(full_reset=True)
    chk = Checker(env)
    finished = np.zeros(B, np.int64)
    for _ in range(episodes * n * m):
        (_, _, done, _), _, _, _, _ = chk.kernel_step(watch=finished < episodes)
        finished += done.cpu().numpy()
        if finished.min() >= episodes:
            break
    assert finished.min() >= episodes
    chk.report("%dx%d omega=%g" % (n, m, omega))
    env.close()


# ---- 2: the cache across auto-resets, reset(), load_scene() and skipped calls ---------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("reset_episodes", [1, 200])
def test_best_target_cache_across_restarts_resets_scene_loads_and_skipped_calls(reset_episodes):
    """Auto-resets into new scenes (RESET_EPISODES = 1) or state-only restarts (200); a mid-episode reset() of both kinds
    and a mid-episode load_scene(), each followed by random steps before the next kernel call; and blocks of random steps
    throughout, so that rows are entered while the kernel is not called."""
    B, cfg = 512, ub.Config(COST_WEIGHT_OMEGA=0.5, RESET_EPISODES=reset_episodes)
    env = ub.UAVEnvBatched(B, seed=8, config=cfg)
    env.reset(full_reset=True)
    chk = Checker(env)
    other = env.get_scene(0, B)                      # scenes to load later: every env gets its neighbour's first scene
    other = {k: np.roll(v, 1, axis=0) for k, v in other.items()}
    # two full resets 20 steps apart: most envs are in episode 1 at both, so (episode, UAV pointer) keys recur
    events = {250: lambda: env.reset(full_reset=False), 400: lambda: env.reset(full_reset=True),
              420: lambda: env.reset(full_reset=True), 550: lambda: env.load_scene(other)}
    dones = 0
    for s in range(900):
        if s in events:
            events[s]()
            chk.ref.refresh()                        # (a load keeps the scene index)
        if (s // 4) % 3 == 1 or any(e <= s < e + 3 for e in events):
            _, _, done, _ = chk.random_step(s)
        else:
            (_, _, done, _), _, _, _, _ = chk.kernel_step()
        dones += int(done.sum())
    assert dones > 2 * B
    chk.report("cache, RESET_EPISODES=%d" % reset_episodes)
    env.close()


# ---- 3: properties -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_every_uav_assigns_at_omega_zero_and_episode_lengths_follow_j_star():
    """At omega = 0 every Assign is accepted, so each UAV is assigned on its row's j*: assigns == valid == N and an
    episode lasts sum_k (j*_k + 1) steps, with j*_k from the reference when the pointer enters row k (episodes with a
    near-tie at a row entry are left out of the length check)."""
    B, quota = 512, 2
    env = ub.UAVEnvBatched(B, seed=12, config=ub.Config(RESET_EPISODES=1))
    N = env.N
    rec = ub.EpisodeRecorder(env, quota)
    env.reset(full_reset=True)
    chk = Checker(env)
    expect = [[] for _ in range(B)]
    running, tainted = np.zeros(B, np.int64), np.zeros(B, bool)
    for _ in range(quota * N * env.M):
        (_, _, done, _), got, jstar, near, st = chk.kernel_step()
        rec.record(env._actions)
        enter = st["target_idx"] == 0
        running[enter] += jstar[enter] + 1
        tainted |= enter & near
        for b in np.nonzero(done.cpu().numpy())[0]:
            expect[b].append(-1 if tainted[b] else running[b])
            running[b], tainted[b] = 0, False
        if rec.complete() == B:
            break
    assert rec.complete() == B
    r = rec.records()
    assert (r["assigns"] == N).all() and (r["valid"] == N).all()
    want = np.array([e[:quota] for e in expect])
    clean = want >= 0
    assert clean.mean() > 0.9
    assert np.array_equal(r["length"][clean], want[clean])
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("omega", [0.0, 0.5])
def test_kernel_actions_replayed_on_the_oracle(omega):
    """The kernel's actions on 128 envs (one episode, no auto-reset), replayed on the C oracle with the scenes read back by
    get_scene: the same pointers after every step, the same assigned_target_id bit for bit, J within 1e-9."""
    from oracle import oracle as orc
    B = 128
    cfg = ub.Config(COST_WEIGHT_OMEGA=omega)
    env = ub.UAVEnvBatched(B, seed=21, config=cfg, auto_reset=False)
    env.reset(full_reset=True)
    scenes = env.get_scene()
    oenvs = []
    for b in range(B):
        oe = orc.OracleEnv(oracle_cfg_from_config(cfg))
        oe.load_scene({k: v[b] for k, v in scenes.items()})
        oe.reset()
        oenvs.append(oe)
    live = np.ones(B, bool)
    assigns = 0
    for s in range(env.N * env.M):
        a = env.best_target_actions().cpu().numpy()
        assert (a[~live] == 0).all()                 # a finished env is inert
        assigns += int(a.sum())
        _, _, done, _ = env.step(env._actions)
        d = done.cpu().numpy()
        st = env.get_state()
        for b in np.nonzero(live)[0]:
            _, _, o_done, _ = oenvs[b].step(int(a[b]))
            assert bool(d[b]) == o_done, (s, b)
            if not o_done:
                assert st["uav_idx"][b] == oenvs[b].uav_idx and st["target_idx"][b] == oenvs[b].target_idx, (s, b)
            live[b] = not o_done
        if not live.any():
            break
    assert not live.any() and assigns > 0
    st = env.get_state()
    for b, oe in enumerate(oenvs):
        assert np.array_equal(st["assigned_target_id"][b], oe.assigned()), b
        assert abs(st["J_val"][b] - oe.calc_J()) <= 1e-9 * max(1.0, abs(oe.calc_J())), b
    env.close()


@pytest.mark.gpu
def test_best_target_actions_validates_arguments_on_a_live_handle():
    """A real handle: NULL cache or actions is UAVENV_EINVAL, a call before any reset() is UAVENV_ESTATE, and neither
    writes the output."""
    L = ub.load_library()
    env = ub.UAVEnvBatched(64, seed=1)
    cache = torch.zeros(64, dtype=torch.int64, device=env.device)
    out = torch.full((64,), 7, dtype=torch.int64, device=env.device)
    cp, op = C.c_void_p(cache.data_ptr()), C.c_void_p(out.data_ptr())
    assert L.uavenv_best_target_actions(env._h, cp, op, None) == ERR["UAVENV_ESTATE"]
    env.reset(full_reset=True)
    for c, o in ((None, op), (cp, None), (None, None)):
        assert L.uavenv_best_target_actions(env._h, c, o, None) == ERR["UAVENV_EINVAL"]
        assert b"non-NULL" in L.uavenv_last_error(env._h)
    torch.cuda.synchronize()
    assert (out == 7).all() and (cache == 0).all()
    assert L.uavenv_best_target_actions(env._h, cp, op, None) == 0
    torch.cuda.synchronize()
    assert set(out.tolist()) <= {0, 1} and (cache != 0).any()
    env.close()


# ---- 4: evaluate_baseline ---------------------------------------------------------------------------------------------

def _assert_same_records(a, b):
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["best_target", "random"])
def test_evaluate_baseline_is_reproducible_and_shard_invariant(kind):
    full = ub.evaluate_baseline(kind, num_envs=2048, episodes_per_env=2, seed=5)
    _assert_same_records(full, ub.evaluate_baseline(kind, num_envs=2048, episodes_per_env=2, seed=5))
    lo = ub.evaluate_baseline(kind, num_envs=1024, episodes_per_env=2, seed=5, env_id_base=0)
    hi = ub.evaluate_baseline(kind, num_envs=1024, episodes_per_env=2, seed=5, env_id_base=1024)
    _assert_same_records(full, {k: np.concatenate([lo[k], hi[k]]) for k in KEYS})
    assert full["summary"]["episodes"] == 4096


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["best_target", "random"])
def test_evaluate_baseline_equals_a_direct_loop_on_the_scenes_of_evaluate(kind, monkeypatch):
    """The records equal a direct loop of (best_target_actions | random_actions with action seed = seed + 1) -> step ->
    EpisodeRecorder, and the first scenes after the reset are those evaluate(checkpoint) plays with the same seed."""
    from target_allocation_ppo_transformer_b200.envs.uav_env import UAVEnvBatched
    B, quota, seed = 512, 2, 77
    first_scenes = []
    reset = UAVEnvBatched.reset

    def capture(self, full_reset=True, env_mask=None):
        obs = reset(self, full_reset, env_mask)
        first_scenes.append(self.get_scene())
        return obs

    monkeypatch.setattr(UAVEnvBatched, "reset", capture)
    res = ub.evaluate_baseline(kind, num_envs=B, episodes_per_env=quota, seed=seed)
    torch.manual_seed(0)
    ub.evaluate(ub.TransformerActorCritic(), num_envs=B, episodes_per_env=1, seed=seed)
    monkeypatch.undo()
    assert len(first_scenes) == 2
    for k in first_scenes[0]:
        assert np.array_equal(first_scenes[0][k], first_scenes[1][k]), k
    env = ub.UAVEnvBatched(B, seed=seed, config=ub.cfg.copy(RESET_EPISODES=1), env_id_base=0)
    rec = ub.EpisodeRecorder(env, quota)
    env.reset(full_reset=True)
    for step in range(quota * env.N * env.M):
        a = env.best_target_actions() if kind == "best_target" else env.random_actions(step, action_seed=seed + 1)
        env.step(a)
        rec.record(a)
    assert rec.complete() == B
    _assert_same_records(res, rec.records())
    env.close()


@pytest.mark.gpu
def test_best_target_beats_random_and_the_untrained_greedy_network():
    """A sanity bound on the default 30x10 config, not a tuned one."""
    B = 4096
    bt = ub.evaluate_baseline("best_target", num_envs=B)["summary"]
    rnd = ub.evaluate_baseline("random", num_envs=B)["summary"]
    torch.manual_seed(0)
    net = ub.evaluate(ub.TransformerActorCritic(), num_envs=B)["summary"]
    print("\n[J_mean] best_target %.3f +- %.3f, random %.3f +- %.3f, untrained greedy %.3f" % (
        bt["J_mean"], bt["J_sem"], rnd["J_mean"], rnd["J_sem"], net["J_mean"]))
    assert bt["J_mean"] > rnd["J_mean"] and bt["J_mean"] > net["J_mean"]
    assert bt["valid_assign_rate"] == 1.0 and bt["length_mean"] < 30 * 10


# ---- 5: CPU ------------------------------------------------------------------------------------------------------

def test_best_target_actions_is_declared_exported_and_checks_null_arguments_without_gpu():
    L = ub.load_library()
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "uavenv_b200.h")).read(), flags=re.S)
    assert re.search(r"\buavenv_best_target_actions\s*\(", text)
    assert hasattr(L, "uavenv_best_target_actions")
    assert L.uavenv_abi_version() == 2
    assert ERR["UAVENV_EINVAL"] == -1 and ERR["UAVENV_ESTATE"] == -4
    p = C.c_void_p(64)                # never dereferenced: validation fails first
    for h, cache, actions in ((None, p, p), (None, None, p), (None, p, None), (None, None, None)):
        assert L.uavenv_best_target_actions(h, cache, actions, None) == ERR["UAVENV_EINVAL"]


def test_evaluate_baseline_rejects_bad_arguments():
    assert ub.evaluate_baseline is ub.evaluate_baseline
    for kind in ("best", "", None, "greedy"):
        with pytest.raises(ValueError):
            ub.evaluate_baseline(kind, num_envs=8)
    for kw in ({"num_envs": 0}, {"num_envs": -4}, {"episodes_per_env": 0}, {"episodes_per_env": -1}):
        with pytest.raises(ValueError):
            ub.evaluate_baseline("random", device="cuda:0", **kw)
    with pytest.raises(RuntimeError):
        ub.evaluate_baseline("best_target", num_envs=4, device="cpu")
