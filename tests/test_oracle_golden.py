"""Pin the CPU oracle (oracle/uavenv_oracle.c) against fixtures produced by the UNMODIFIED
reference (oracle/gen_golden.py -> tests/golden/*.npz).

Integers / flags / pointers: bit-exact.  fp64 values: 1e-12 relative (glibc libm vs numpy's
transcendental kernels differ in the last ulp).  f32 observation rows: 2 ulp of f32.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from helpers import load_fixture
from oracle import oracle as orc

RTOL64 = 1e-12


def _close(a, b, rtol=RTOL64, atol=1e-15):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def test_kat_mechanics():
    """mechanics.py:11-114 primitives at the check_reward_mechanics.py scenarios + random pairs."""
    fx = np.load(os.path.join(GOLDEN, "kat_mechanics.npz"))
    cfg = orc.make_cfg()
    L = orc.lib()
    import ctypes as C
    for row, want in zip(fx["pair_in"], fx["pair_out"]):
        ux, uy, vx, vy, load, tx, ty, tvx, tvy = [float(v) for v in row]
        d = float(np.hypot(ux - tx, uy - ty))
        got = [L.orc_dist_score(C.byref(cfg), d, 0), L.orc_angle_score(ux, uy, vx, vy, tx, ty),
               L.orc_speed_score(C.byref(cfg), float(np.hypot(vx, vy)), float(np.hypot(tvx, tvy))),
               L.orc_damage_prob(C.byref(cfg), ux, uy, vx, vy, load, tx, ty, tvx, tvy)]
        _close(got, want, rtol=1e-11)
    # the three check_reward_mechanics.py scenarios, literal values quoted in SURVEY.md §4
    lit = np.array([[0.4184863060425645, 0.9613972356240913, 0.97, 0.5348875129707363],
                    [0.7524321560893033, 0.9703088870665727, 0.97, 0.782868611089729],
                    [0.9823793146181776, 0.9257412659243867, 0.97, 0.906564059736086]])
    _close(fx["pair_out"][:3], lit, rtol=1e-12)


def test_kat_composite():
    """SURVEY.md §4 composite KAT: p_pen, p_final, p_damage and the 14-feature row."""
    fx = np.load(os.path.join(GOLDEN, "kat_mechanics.npz"))
    cfg = orc.make_cfg()
    env = orc.OracleEnv(orc.make_cfg(NUM_UAVS=1, NUM_TARGETS=1))
    scene = dict(uav_x=[70.0], uav_y=[80.0], uav_vx=[0.45 * np.cos(0.1)], uav_vy=[0.45 * np.sin(0.1)],
                 uav_load=[0.95], uav_cost=[1.0], uav_type=[1], tgt_x=[170.0], tgt_y=[60.0], tgt_vx=[0.01],
                 tgt_vy=[-0.005], tgt_value=[8.0], tgt_id=[0], nfz_x=[130.0], nfz_y=[100.0], nfz_radius=[1.0],
                 int_x=[150.0], int_y=[50.0], int_vx=[0.31 * np.cos(1.0)], int_vy=[0.31 * np.sin(1.0)])
    env.load_scene(scene)
    pf, pd, pp = env.score_matrix()
    _close([pp[0], pf[0, 0], pd[0, 0]], fx["comp_scalars"])
    _close(fx["comp_scalars"], [0.11001011302846028, 0.06023977429173684, 0.5475839687225159])
    import ctypes as C
    out = np.zeros(14, np.float32)
    orc.lib().orc_state_vector_raw(1.0, 8.0, 0.1, 0.2, 0.05, float(pf[0, 0]), float(pd[0, 0]), 0.3, 2.4, 0.5, 1,
                                   out.ctypes.data_as(C.POINTER(C.c_float)))
    np.testing.assert_allclose(out, fx["comp_state"], rtol=3e-7, atol=1e-9)
    del cfg


@pytest.mark.parametrize("case", golden_cases())
def test_trajectory_matches_reference(case):
    fx = load_fixture(case)
    env = orc.OracleEnv(orc.cfg_from_fixture(fx))
    env.load_scene(fx)
    pf, pd, pp = env.score_matrix()
    _close(pf, fx["p_final"]); _close(pd, fx["p_damage"]); _close(pp, fx["p_pen"])
    T = len(fx["action"])
    ep_prev = -1
    window = None
    for t in range(T):
        if fx["episode"][t] != ep_prev:
            ep_prev = int(fx["episode"][t])
            obs = env.reset()
            assert not obs[:4].any()
            np.testing.assert_allclose(obs[4], fx["reset_row"][ep_prev], rtol=3e-7, atol=1e-9)
            window = obs
        obs, reward, done, info = env.step(int(fx["action"][t]))
        assert env.uav_idx == fx["uav_idx"][t] and env.target_idx == fx["target_idx"][t], (case, t)
        assert done == bool(fx["done"][t])
        assert np.array_equal(env.assigned(), fx["assigned"][t].astype(np.int32)), (case, t)
        assert np.array_equal(env.covered(), fx["covered"][t]), (case, t)
        _close(reward, fx["reward"][t], atol=1e-12)
        _close(info["J_val"], fx["J_val"][t], atol=1e-12)
        assert info["num_assigned"] == fx["num_assigned"][t]
        v = info["is_valid_action"]
        assert (-1 if v is None else int(v)) == fx["is_valid"][t]
        _close(info["avg_p_dmg"], fx["avg_p_dmg"][t]); _close(info["avg_p_final"], fx["avg_p_final"][t])
        if done:
            assert obs.shape == (14,) and not obs.any()          # uav_env.py:188-189
        else:
            np.testing.assert_allclose(obs[4], fx["obs_row"][t], rtol=3e-7, atol=1e-9)
            np.testing.assert_array_equal(obs[:4], window[1:])   # deque(maxlen=5) shift
            window = obs
