#!/usr/bin/env python
"""Generate the committed golden fixtures under tests/golden/ by RUNNING THE
UNMODIFIED REFERENCE (imported from /root/reference through oracle/ref_shim.py).

TEST INFRASTRUCTURE ONLY.  Run in the build container (the reference tree is
not present on the GPU box):

    python oracle/gen_golden.py            # writes tests/golden/*.npz

Each trajectory fixture holds, for one reference `UAVEnv` (envs/uav_env.py):
  * the cfg overrides in force (configs/config.py attributes are read at call
    time, so assigning cfg.X before reset() rescales the reference),
  * the scene exported after `reset(full_reset=True)` (list order, fp64),
  * the full score matrices p_final/p_damage[N,M] and p_pen[N]
    (mechanics.calc_advantage / calc_penetration_prob, mechanics.py:118-181),
  * E episodes: episode 0 follows reset(full_reset=True), later ones
    reset(full_reset=False) (the main_train.py:79 schedule inside one scene),
  * per step: the action fed, and everything `step` returned or mutated
    (uav_env.py:295-435): pointers, reward (fp64), done, the five info values,
    the newest observation row (f32[14]), assigned_target_id[N], covered[M].

`kat_mechanics.npz` holds known-answer vectors of the score primitives
(mechanics.py:11-114) at the three check_reward_mechanics.py scenarios plus
random pairs, and the composite KAT quoted in SURVEY.md §4.
"""
import os
import random
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

CFG_KEYS = ["NUM_UAVS", "NUM_TARGETS", "NUM_NFZ", "NUM_INTERCEPTORS", "PARAM_ZETA_D", "PARAM_K",
            "PARAM_C1", "PARAM_C2", "PARAM_C3", "PARAM_C4", "COST_WEIGHT_OMEGA",
            "WEATHER_SPEED_FACTOR", "WEATHER_LOAD_FACTOR", "INTERCEPT_RAD", "MAP_WIDTH", "MAP_HEIGHT",
            "UAV_GEN_X_RANGE", "TARGET_GEN_X_RANGE"]

HARD_MODE = dict(PARAM_K=5.0, UAV_GEN_X_RANGE=(0, 30), NUM_NFZ=2, NUM_INTERCEPTORS=2,
                 INTERCEPT_RAD=3.0, WEATHER_SPEED_FACTOR=0.85, WEATHER_LOAD_FACTOR=0.90)  # configs/config0.py


def run_case(name, seed, episodes, p_assign, overrides, odd_actions=False):
    UAVEnv, mech, cfg = ref_shim.load()
    saved = {k: getattr(cfg, k) for k in CFG_KEYS}
    try:
        for k, v in overrides.items():
            setattr(cfg, k, v)
        random.seed(seed)
        np.random.seed(seed)
        env = UAVEnv()
        arng = np.random.RandomState(10_000 + seed)  # action stream, independent of the scene streams
        rec = {k: [] for k in ("action", "uav_idx", "target_idx", "reward", "done", "J_val", "num_assigned",
                               "is_valid", "avg_p_dmg", "avg_p_final", "obs_row", "assigned", "covered",
                               "episode")}
        reset_rows = []
        scene = None
        t0 = time.time()
        for ep in range(episodes):
            obs = env.reset(full_reset=(ep == 0))
            if ep == 0:
                scene = ref_shim.export_scene(env)
                N, M = len(env.uavs), len(env.targets)
                pf = np.zeros((N, M))
                pd = np.zeros((N, M))
                pp = np.zeros(N)
                for i, u in enumerate(env.uavs):
                    pp[i] = mech.calc_penetration_prob(u, env.targets[0], env.nfz_list, env.interceptors)
                    for j, t in enumerate(env.targets):
                        pf[i, j], pd[i, j] = mech.calc_advantage(u, t, env.nfz_list, env.interceptors)
            assert obs.shape == (5, 14) and not obs[:4].any()
            reset_rows.append(obs[4].copy())
            done = False
            while not done:
                a = int(arng.rand() < p_assign)
                if odd_actions and arng.rand() < 0.15:
                    a = int(arng.choice([2, -1, 7, 255]))  # anything but 1 is Skip (uav_env.py:344)
                obs, reward, done, info = env.step(a)
                rec["action"].append(a)
                rec["uav_idx"].append(env.uav_idx)
                rec["target_idx"].append(env.target_idx)
                rec["reward"].append(float(reward))
                rec["done"].append(bool(done))
                rec["J_val"].append(float(info["J_val"]))
                rec["num_assigned"].append(int(info["num_assigned"]))
                v = info["is_valid_action"]
                rec["is_valid"].append(-1 if v is None else int(bool(v)))
                rec["avg_p_dmg"].append(float(info["avg_p_dmg"]))
                rec["avg_p_final"].append(float(info["avg_p_final"]))
                rec["obs_row"].append(np.zeros(14, np.float32) if done else obs[4].copy())
                rec["assigned"].append([u.assigned_target_id for u in env.uavs])
                rec["covered"].append([len(t.locked_by_uavs) > 0 for t in env.targets])
                rec["episode"].append(ep)
        out = dict(scene)
        out.update(
            cfg_names=np.array(list(CFG_KEYS)),
            cfg_values=np.array([np.atleast_1d(np.asarray(getattr(cfg, k), np.float64))[0] for k in CFG_KEYS]),
            cfg_uav_gen_x=np.asarray(cfg.UAV_GEN_X_RANGE, np.float64),
            cfg_target_gen_x=np.asarray(cfg.TARGET_GEN_X_RANGE, np.float64),
            seed=np.int64(seed), p_final=pf, p_damage=pd, p_pen=pp,
            reset_row=np.asarray(reset_rows, np.float32),
            action=np.asarray(rec["action"], np.int16),
            uav_idx=np.asarray(rec["uav_idx"], np.int32),
            target_idx=np.asarray(rec["target_idx"], np.int32),
            reward=np.asarray(rec["reward"], np.float64),
            done=np.asarray(rec["done"], np.uint8),
            J_val=np.asarray(rec["J_val"], np.float64),
            num_assigned=np.asarray(rec["num_assigned"], np.int32),
            is_valid=np.asarray(rec["is_valid"], np.int8),
            avg_p_dmg=np.asarray(rec["avg_p_dmg"], np.float64),
            avg_p_final=np.asarray(rec["avg_p_final"], np.float64),
            obs_row=np.asarray(rec["obs_row"], np.float32),
            assigned=np.asarray(rec["assigned"], np.int16),
            covered=np.asarray(rec["covered"], np.uint8),
            episode=np.asarray(rec["episode"], np.int32),
        )
        if pf.size > 4096:       # a 256x256 p_final would put the file over 1 MB: tests/helpers.py re-forms the product
            assert np.array_equal(pf, pd * pp[:, None])
            del out["p_final"]
        path = os.path.join(OUT, "traj_%s.npz" % name)
        np.savez_compressed(path, **out)
        T = len(rec["action"])
        nrej = int(((out["is_valid"] == 0)).sum())
        print("%-28s N=%d M=%d steps=%d rejected_or_zero=%d  ref %.1f steps/s  -> %s (%.0f KB)" % (
            name, N, M, T, nrej, T / (time.time() - t0), os.path.basename(path), os.path.getsize(path) / 1024))
    finally:
        for k, v in saved.items():
            setattr(cfg, k, v)


def kat_mechanics():
    _, mech, cfg = ref_shim.load()
    from envs.entities import UAV, Target, NoFlyZone, Interceptor
    rows = []
    # the three check_reward_mechanics.py scenarios (distance km, bearing deg)
    for d, deg in ((140.0, 10.0), (80.0, 5.0), (20.0, 2.0)):
        th = np.deg2rad(deg)
        u = UAV(id=0, pos=np.array([0.0, 0.0]), velocity=np.array([0.4, 0.0]), load=1.0)
        t = Target(id=0, pos=np.array([d * np.cos(th), d * np.sin(th)]), value=8.0)
        t.velocity = np.array([0.01, 0.0])
        rows.append((u, t))
    rs = np.random.RandomState(7)
    for _ in range(61):
        sp = rs.uniform(0.0, 0.9)
        ang = rs.uniform(-np.pi, np.pi)
        u = UAV(id=0, pos=rs.uniform(0, 180, 2), velocity=np.array([np.cos(ang), np.sin(ang)]) * sp,
                load=rs.uniform(0.5, 1.0))
        t = Target(id=0, pos=rs.uniform(0, 180, 2), value=8.0)
        t.velocity = (rs.rand(2) - 0.5) * rs.choice([0.03, 0.6])
        rows.append((u, t))
    # degenerate branches: coincident points (mechanics.py:22), zero UAV speed (:32, :65)
    u = UAV(id=0, pos=np.array([5.0, 5.0]), velocity=np.array([0.3, 0.1]), load=1.0)
    t = Target(id=0, pos=np.array([5.0, 5.0]), value=4.0); t.velocity = np.array([0.01, 0.0])
    rows.append((u, t))
    u = UAV(id=0, pos=np.array([5.0, 5.0]), velocity=np.array([0.0, 0.0]), load=1.0)
    t = Target(id=0, pos=np.array([50.0, 25.0]), value=4.0); t.velocity = np.array([0.01, 0.0])
    rows.append((u, t))
    n = len(rows)
    inp = np.zeros((n, 9))
    out = np.zeros((n, 4))
    for i, (u, t) in enumerate(rows):
        d = mech.get_distance(u.pos, t.pos)
        vt = np.linalg.norm(t.velocity)
        inp[i] = [u.pos[0], u.pos[1], u.velocity[0], u.velocity[1], u.load, t.pos[0], t.pos[1], t.velocity[0],
                  t.velocity[1]]
        out[i] = [mech.calc_dist_score(d), mech.calc_angle_score(u.pos, u.velocity, t.pos),
                  mech.calc_speed_score(np.linalg.norm(u.velocity), vt), mech.calc_damage_prob(u, t)]
    # composite KAT (SURVEY.md §4)
    u = UAV(id=0, pos=np.array([70.0, 80.0]), velocity=0.45 * np.array([np.cos(0.1), np.sin(0.1)]), load=0.95)
    u.cost = 1.0
    t = Target(id=0, pos=np.array([170.0, 60.0]), value=8.0); t.velocity = np.array([0.01, -0.005])
    z = NoFlyZone(id=0, pos=np.array([130.0, 100.0]))
    it = Interceptor(id=0, pos=np.array([150.0, 50.0])); it.velocity = 0.31 * np.array([np.cos(1.0), np.sin(1.0)])
    p_pen = mech.calc_penetration_prob(u, t, [z], [it])
    p_final, p_damage = mech.calc_advantage(u, t, [z], [it])
    sv = mech.get_state_vector(u, t, [z], [it],
                               global_stats={"cost_ratio": 0.1, "value_ratio": 0.2, "target_cost_ratio": 0.05},
                               prev_joint_p=0.3, prev_revenue=2.4, prev_joint_p_damage_only=0.5)
    np.savez_compressed(os.path.join(OUT, "kat_mechanics.npz"), pair_in=inp, pair_out=out,
                        comp_scalars=np.array([p_pen, p_final, p_damage]), comp_state=sv,
                        consts=np.array([cfg.PARAM_ZETA_D, cfg.PARAM_K, cfg.PARAM_C1, cfg.PARAM_C2, cfg.PARAM_C3,
                                         cfg.PARAM_C4]))
    print("kat_mechanics: %d pairs; composite p_pen=%.17g p_final=%.17g p_damage=%.17g" % (
        n, p_pen, p_final, p_damage))


def scene_stats():
    """Moments of the reference scene generator (uav_env.py:65-173), for the statistical test of
    the counter-based generator: 400 default scenes + 200 at (16 UAVs, 9 targets)."""
    UAVEnv, _, cfg = ref_shim.load()
    random.seed(123)
    np.random.seed(123)
    env = UAVEnv()
    acc = {k: [] for k in ("uav_x", "uav_y", "speed1", "speed2", "heading", "tgt_x", "tgt_y", "tgt_vx", "nfz_x",
                           "int_x", "int_speed", "n2", "type2_count", "value_sum", "id_at_0", "type_at_0")}
    for _ in range(400):
        env.reset(full_reset=True)
        for u in env.uavs:
            acc["uav_x"].append(u.pos[0]); acc["uav_y"].append(u.pos[1])
            acc["speed1" if u.uav_type == 1 else "speed2"].append(np.linalg.norm(u.velocity))
            acc["heading"].append(np.arctan2(u.velocity[1], u.velocity[0]))
        for t in env.targets:
            acc["tgt_x"].append(t.pos[0]); acc["tgt_y"].append(t.pos[1]); acc["tgt_vx"].append(t.velocity[0])
        acc["nfz_x"].append(env.nfz_list[0].pos[0])
        acc["int_x"].append(env.interceptors[0].pos[0])
        acc["int_speed"].append(np.linalg.norm(env.interceptors[0].velocity))
        acc["n2"].append(sum(1 for t in env.targets if t.value == 6.0))
        acc["type2_count"].append(sum(1 for u in env.uavs if u.uav_type == 2))
        acc["value_sum"].append(sum(t.value for t in env.targets))
        acc["id_at_0"].append(env.targets[0].id)
        acc["type_at_0"].append(env.uavs[0].uav_type)
    out = {}
    for k, v in acc.items():
        v = np.asarray(v, np.float64)
        out[k] = np.array([v.mean(), v.std(), v.min(), v.max(), len(v)])
    np.savez_compressed(os.path.join(OUT, "scene_stats.npz"), **out)
    print("scene_stats: ", {k: np.round(v[:2], 4).tolist() for k, v in out.items()})


def main():
    os.makedirs(OUT, exist_ok=True)
    kat_mechanics()
    scene_stats()
    # default scene (configs/config.py): omega = 0 (live), plus omega > 0 to exercise the Eq.21 rollback
    for s in range(4):
        run_case("default_s%d" % s, s, 3, 0.5, {})
    run_case("default_odd_actions", 11, 2, 0.5, {}, odd_actions=True)
    run_case("default_p09", 12, 3, 0.9, {})
    run_case("default_p01", 13, 2, 0.1, {})
    for om in (0.5, 2.0):
        for s in range(3):
            run_case("omega%s_s%d" % (str(om).replace(".", ""), s), 20 + s, 3, 0.7, {"COST_WEIGHT_OMEGA": om})
    run_case("hard_s0", 30, 2, 0.5, dict(HARD_MODE))
    run_case("hard_omega05", 31, 2, 0.7, dict(HARD_MODE, COST_WEIGHT_OMEGA=0.5))
    # degenerate sizes: n_remain < 1 branch (uav_env.py:125), no obstacles, single pair
    run_case("tiny_1x1", 40, 3, 0.5, dict(NUM_UAVS=1, NUM_TARGETS=1))
    run_case("tiny_3x2", 41, 3, 0.5, dict(NUM_UAVS=3, NUM_TARGETS=2))
    run_case("tiny_5x3_noobst", 42, 3, 0.5, dict(NUM_UAVS=5, NUM_TARGETS=3, NUM_NFZ=0, NUM_INTERCEPTORS=0))
    run_case("tiny_4x1_omega", 43, 3, 0.8, dict(NUM_UAVS=4, NUM_TARGETS=1, COST_WEIGHT_OMEGA=0.5))
    # scaled scenarios of BASELINE.json configs 3 and 5
    run_case("n64m64_s0", 50, 2, 0.5, dict(NUM_UAVS=64, NUM_TARGETS=64))
    run_case("n64m64_omega05", 51, 1, 0.7, dict(NUM_UAVS=64, NUM_TARGETS=64, COST_WEIGHT_OMEGA=0.5))
    run_case("n256m256_s0", 60, 1, 0.5, dict(NUM_UAVS=256, NUM_TARGETS=256))


if __name__ == "__main__":
    main()
