"""Certified upper bound on the best J of a scene (uavenv_upper_bound, ub.upper_bound, ub.allocate(bound=True)): the
kernel against an fp64 numpy re-implementation of the rule in include/uavenv_b200.h at the configs, at every shape class
of the matrix's home and of the per-thread loops, and on a CTA's later scenes; validity against brute force on tiny
scenes (one with p = 1 exactly) and against every allocator of the project at scale; the exact cases M = 1 and
all-negative gradients; monotonicity in iters; launch independence; argument checks.  The CPU tests at the end need no
GPU."""
import ctypes as C
import itertools
import math
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_gpu_improve import CONFIGS, _bits, _loaded, _np, _random_rows, _scenes

import uavenv_b200 as ub

ERR = {name: int(v) for name, v in re.findall(r"\b(UAVENV_E[A-Z]+)\s*=\s*(-?\d+)",
                                              open(os.path.join(ROOT, "include", "uavenv_b200.h")).read())}
AMAX = 40.0
THREADS = 256         # bound_kernel's CTA: the fixed order of its line-search sums
NEWTON = 10
NEAR = 1e-12          # relative gap of a UAV's two best gradients below which a scene is left out of the comparison
ITERS = (1, 2, 5, 256)


# ---- the fp64 reference of the bound rule --------------------------------------------------------------------------

def _seq(x):
    """Sum in index order (np.add.accumulate adds one element at a time)."""
    x = np.asarray(x, np.float64)
    return float(np.add.accumulate(x)[-1]) if x.size else 0.0


def _block_sum(x):
    """block_sum2's order: thread i adds x[i], x[i + 256], ... from 0; xor-butterfly within each warp of 32; warps 0..7
    added in order."""
    x = np.asarray(x, np.float64)
    acc = np.zeros(THREADS)
    for r in range(0, x.size, THREADS):
        row = np.zeros(THREADS)
        row[:min(THREADS, x.size - r)] = x[r:r + THREADS]
        acc = acc + row
    v = acc.reshape(-1, 32)
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[:, lanes ^ o]
    tot = v[0, 0]
    for w in range(1, v.shape[0]):
        tot = tot + v[w, 0]
    return float(tot)


def ref_bound(p, val, cost, omega, iters):
    """History of the iteration on one scene, in the kernel's operation order: per iteration t (1-based) the entry
    (bound after t iterations, F at iterate t, stopped at t), so the outputs of a call with any cap c are those of entry
    min(c, stop) - 1.  near: some UAV's two best gradients (or its best and the pick threshold 0) lie within NEAR."""
    N, M = p.shape
    with np.errstate(divide="ignore"):
        a = np.minimum(-np.log1p(-p), AMAX)
    tv, tc = _seq(val), _seq(cost)
    margin = tv * math.exp(-AMAX) + 1e-12 * (tv + omega * tc)
    s, C, best, near, hist = np.zeros(M), 0.0, math.inf, False, []
    oc = omega * cost
    ks = np.arange(N)
    for t in range(1, iters + 1):
        nh = np.exp(-s)
        w = val * nh
        F = _seq(val * (1.0 - nh)) - omega * C
        lin = _seq(w * s)
        g = w[None, :] * a - oc[:, None]
        jb = np.argmax(g, axis=1)
        gb = g[ks, jb]
        if M > 1:
            second = np.partition(g, M - 2, axis=1)[:, M - 2]
            close = (gb - second <= NEAR * np.maximum(np.abs(gb), np.abs(second))) & (gb > 0)
            near |= bool(close.any())
        near |= bool(((gb != 0) & (np.abs(gb) <= NEAR * np.maximum(oc, np.abs(w[jb] * a[ks, jb])))).any())
        pick = gb > 0.0
        G = _seq(np.where(pick, gb, 0.0))
        Cs = _seq(np.where(pick, cost, 0.0))
        U = (F + G) - (lin - omega * C)
        best = min(best, U)
        stop = U - F <= 1e-9 * max(1.0, abs(U))
        hist.append((best + margin, F, stop))
        if stop:
            break
        sig = np.zeros(M)
        np.add.at(sig, jb[pick], a[ks[pick], jb[pick]])                   # ascending k per target, from 0
        d, dC = sig - s, Cs - C

        def ev(gam):
            q = (val * np.exp(-(s + gam * d))) * d
            return _block_sum(q) - omega * dC, _block_sum(q * d)

        gam = 1.0
        p1, p2 = ev(1.0)
        if p1 < 0.0:
            lo, hi = 0.0, 1.0
            for _ in range(NEWTON):
                c = gam + p1 / p2
                if c == gam:
                    break
                if not (lo < c < hi):
                    c = 0.5 * (lo + hi)
                gam = c
                p1, p2 = ev(gam)
                if p1 > 0.0:
                    lo = gam
                else:
                    hi = gam
        s = s + gam * d
        C = C + gam * dC
    return hist, near


def ref_outputs(hist, cap):
    """(bound, relaxed, iters) of a call with iteration cap `cap` from ref_bound's history."""
    i = min(cap, len(hist)) - 1
    return hist[i][0], hist[i][1], i + 1


def test_block_sum_order_and_reference_on_a_hand_made_scene():
    """_block_sum adds a 300-element vector in block_sum2's order (equal to the plain sum to rounding), and the reference
    on a 3 x 2 scene: iteration 1's U is the linear bound sum_k max(0, max_j v_j a_kj - omega c_k), and the bound at 256
    iterations lies between the brute-force optimum and that."""
    x = np.random.default_rng(0).standard_normal(300)
    assert _block_sum(x) == pytest.approx(float(np.sum(x)), rel=1e-12, abs=1e-12)
    p = np.array([[0.9, 0.1], [0.2, 0.8], [0.5, 0.5]])
    val, cost, omega = np.array([1.0, 2.0]), np.array([0.1, 0.1, 5.0]), 0.1
    a = -np.log1p(-p)
    lin = sum(max(0.0, float(np.max(val * a[k] - omega * cost[k]))) for k in range(3))
    hist, _ = ref_bound(p, val, cost, omega, 256)
    assert hist[0][0] == pytest.approx(lin, rel=1e-12) and hist[0][1] == 0.0
    Jstar = _brute_force(p, val, cost, omega)
    assert Jstar <= hist[-1][0] <= lin


# ---- helpers ---------------------------------------------------------------------------------------------------------

def _brute_force(p, val, cost, omega):
    """The best J over all (M+1)^N allocations (products in ascending UAV order, J as the env sums it)."""
    N, M = p.shape
    best = -math.inf
    for t in itertools.product(range(-1, M), repeat=N):
        nh = np.ones(M)
        for k, j in enumerate(t):
            if j >= 0:
                nh[j] *= 1.0 - p[k, j]
        rev = 0.0
        for j in range(M):
            rev += (1.0 - nh[j]) * val[j]
        c = 0.0
        for k, j in enumerate(t):
            if j >= 0:
                c += cost[k]
        best = max(best, rev - omega * c)
    return best


def _compare(got, scenes, pf, omega, caps, idx=None, label=""):
    """got[cap] (entry i: scene idx[i]) against the reference at every cap: bound and relaxed to 1e-9 relative, iters
    exactly.  Returns (scenes compared, scenes left out for a near tie)."""
    idx = list(range(pf.shape[0])) if idx is None else list(idx)
    kept = left = 0
    for i, s in enumerate(idx):
        hist, near = ref_bound(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega, max(caps))
        if near:
            left += 1
            continue
        for cap in caps:
            b, r, it = ref_outputs(hist, cap)
            assert got[cap]["iters"][i] == it, (label, s, cap, got[cap]["iters"][i], it)
            assert got[cap]["bound"][i] == pytest.approx(b, rel=1e-9, abs=1e-12), (label, s, cap)
            assert got[cap]["relaxed"][i] == pytest.approx(r, rel=1e-9, abs=1e-12), (label, s, cap)
        kept += 1
    return kept, left


# ---- 1: against the reference --------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_bound_equals_fp64_reference(name):
    """bound, relaxed and iters at iters = 1, 2, 5 and 256 equal the reference's (relaxed after t iterations pins the
    path: every pick of the first t - 1 iterations matched)."""
    cfg = ub.Config(**CONFIGS[name])
    S, omega = 24, float(cfg.COST_WEIGHT_OMEGA)
    scenes = _scenes(S, 73, cfg)
    env, pf = _loaded(scenes, cfg)
    got = {cap: _np(env.upper_bound(iters=cap)) for cap in ITERS}
    kept, left = _compare(got, scenes, pf, omega, ITERS, label=name)
    print("\n[bound %s] %d of %d scenes equal the reference, %d left out for a near tie; iters at 256: mean %.1f" % (
        name, kept, S, left, got[256]["iters"].mean()))
    assert left <= max(2, S // 4)
    env.close()


# (N, M, scenes, where a lives): N > 256 (two passes of the per-UAV loops), M > 256 (two passes of the per-target
# loops), both sides of improve_p_in_smem's 64 KB line, and 256 x 256
SHAPES = [(300, 4, 6, "shared"), (8, 300, 8, "shared"), (64, 64, 8, "shared"), (128, 64, 6, "shared"),
          (129, 64, 6, "workspace"), (64, 129, 6, "workspace"), (256, 256, 3, "workspace")]


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,S,where", [pytest.param(*c, id="%dx%d-%s" % (c[0], c[1], c[3])) for c in SHAPES])
def test_shape_classes_equal_fp64_reference(N, M, S, where):
    omega = 0.25
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 67, cfg)
    env, pf = _loaded(scenes, cfg)
    assert (env._lib.uavenv_improve_workspace_bytes(env._h) == 0) == (where == "shared")
    got = {cap: _np(env.upper_bound(iters=cap)) for cap in ITERS}
    kept, left = _compare(got, scenes, pf, omega, ITERS, label="%dx%d" % (N, M))
    print("\n[bound %dx%d %s] %d of %d scenes equal, %d left out for a near tie" % (N, M, where, kept, S, left))
    assert kept >= 1 and left <= max(1, S // 3)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,waves,extra", [((256, 256), 2, 7), ((64, 64), 8, 50)], ids=["256x256", "64x64"])
def test_later_scenes_of_a_cta_equal_fp64_reference(shape, waves, extra):
    """waves * SMs + extra scenes in one call: 256x256 runs one CTA per SM (workspace), 64x64 at most 8 per SM (shared),
    so the last scenes are a CTA's second and third or later.  The scenes around each multiple of the SM count and the
    last equal the reference, and each alone in a call gives the same bits."""
    N, M = shape
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    S, omega, cap = waves * sms + extra, 0.25, 64
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 39, cfg)
    env, pf = _loaded(scenes, cfg)
    got = _np(env.upper_bound(iters=cap))
    sub = sorted({0, S - 1} | {c * sms + d for c in range(1, waves + 1) for d in (-1, 0)})
    kept, left = _compare({cap: {k: v[sub] for k, v in got.items()}}, scenes, pf, omega, (cap,), idx=sub, label="later")
    print("\n[bound %dx%d, %d scenes, %d SMs] %d of %d checked scenes equal, %d left out" % (N, M, S, sms, kept, len(sub),
                                                                                          left))
    assert left <= max(1, len(sub) // 4)
    for s in sub:
        one = _np(env.upper_bound(first_env=s, count=1, iters=cap))
        for k in got:
            a, b = got[k][s:s + 1], one[k]
            assert np.array_equal(_bits(a) if a.dtype == np.float64 else a, _bits(b) if b.dtype == np.float64 else b), (k, s)
    env.close()


# ---- 2: validity -----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(3, 2), (4, 3), (5, 4), (6, 3), (6, 4)])
def test_bound_is_at_least_the_brute_force_optimum(N, M):
    worst = []
    for omega in (0.0, 0.5, 2.0):
        cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
        S = 12 if N * M < 24 else 6
        for seed in (3, 4):
            scenes = _scenes(S, seed, cfg)
            env, pf = _loaded(scenes, cfg)
            for cap in (1, 5, 256):
                got = _np(env.upper_bound(iters=cap))
                assert np.isfinite(got["bound"]).all() and (got["bound"] >= got["relaxed"]).all()
                for s in range(S):
                    J = _brute_force(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega)
                    assert got["bound"][s] >= J, (omega, seed, cap, s, got["bound"][s], J)
                    if cap == 256:
                        worst.append((got["bound"][s] - J) / max(abs(J), 1.0))
            env.close()
    print("\n[bound %dx%d brute force] %d scenes, relative gap at 256 iterations: mean %.4f, max %.4f" % (
        N, M, len(worst), float(np.mean(worst)), float(np.max(worst))))


@pytest.mark.gpu
def test_bound_is_finite_and_valid_where_p_is_one():
    """No obstacles (p_pen = 1) and UAV 0 on a still target 0 with a high load: damage_prob clips to 1, so p = 1 and
    -log1p(-p) is infinite; the capped a keeps the bound finite and above the brute-force optimum."""
    for omega in (0.0, 0.5):
        cfg = ub.Config(NUM_UAVS=5, NUM_TARGETS=3, NUM_NFZ=0, NUM_INTERCEPTORS=0, COST_WEIGHT_OMEGA=omega)
        scenes = _scenes(4, 5, cfg)
        for f in ("x", "y"):
            scenes["uav_" + f][:, 0] = scenes["tgt_" + f][:, 0]
        scenes["tgt_vx"][:, 0] = 0.0
        scenes["tgt_vy"][:, 0] = 0.0
        scenes["uav_load"][:, 0] = 10.0
        env, pf = _loaded(scenes, cfg)
        assert (pf[:, 0, 0] == 1.0).all()
        got = _np(env.upper_bound())
        assert np.isfinite(got["bound"]).all() and np.isfinite(got["relaxed"]).all()
        for s in range(4):
            J = _brute_force(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega)
            assert got["bound"][s] >= J, (omega, s)
            hist, _ = ref_bound(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega, 256)
            b, r, it = ref_outputs(hist, 256)
            assert got["iters"][s] == it and got["bound"][s] == pytest.approx(b, rel=1e-9)
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,S", [(30, 10, 256), (64, 64, 128), (256, 256, 32)], ids=["30x10", "64x64", "256x256"])
def test_bound_is_at_least_every_allocation_the_project_makes(N, M, S):
    """On the same scenes: allocate with K = 16 sampled episodes, with and without improve=True, the best-target
    heuristic with and without the local search, and the local search from random rows all stay at or below the bound.
    allocate(bound=True) returns the same bits as upper_bound."""
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=0.5)
    scenes = _scenes(S, 47, cfg)
    torch.manual_seed(1)
    net = ub.TransformerActorCritic()
    ubd = ub.upper_bound(scenes, config=cfg)
    bound = ubd["bound"]
    res = {"sampled_16": ub.allocate(net, scenes=scenes, samples=16, seed=2, config=cfg, bound=True),
           "sampled_16_improve": ub.allocate(net, scenes=scenes, samples=16, seed=2, config=cfg, improve=True, bound=True),
           "best_target": ub.allocate("best_target", scenes=scenes, config=cfg),
           "best_target_improve": ub.allocate("best_target", scenes=scenes, config=cfg, improve=True),
           "random_improve": ub.improve_allocation(scenes, _random_rows(scenes, np.random.default_rng(4)), config=cfg)}
    for label, r in res.items():
        assert (r["J"] <= bound).all(), (label, int(np.argmax(r["J"] - bound)))
    for label in ("sampled_16", "sampled_16_improve"):
        assert np.array_equal(_bits(res[label]["J_bound"]), _bits(bound)), label
    assert set(res["sampled_16"]) == set(res["best_target"]) | {"J_bound"}
    assert set(res["sampled_16_improve"]) == set(res["best_target_improve"]) | {"J_bound"}
    s = res["sampled_16"]["summary"]
    assert s["J_bound_mean"] == pytest.approx(float(bound.mean())) and s["gap_mean"] == pytest.approx(
        float((bound - res["sampled_16"]["J"]).mean()))
    gaps = {k: float(((bound - r["J"]) / np.maximum(np.abs(r["J"]), 1e-9)).mean()) for k, r in res.items()}
    print("\n[bound %dx%d] bound %.4f, relaxed %.4f, iters %.1f; mean relative gap %s" % (
        N, M, bound.mean(), ubd["relaxed"].mean(), ubd["iters"].mean(),
        ", ".join("%s %.4f" % kv for kv in gaps.items())))


# ---- 3: exact cases ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_single_target_at_omega_zero_is_exact():
    """M = 1, omega = 0: every UAV picks the target, gamma = 1, and iteration 2 is the allocation "everyone assigned",
    where U = F: the bound is J(all assigned) plus the margin, after 2 iterations."""
    cfg = ub.Config(NUM_UAVS=6, NUM_TARGETS=1, COST_WEIGHT_OMEGA=0.0)
    S = 32
    scenes = _scenes(S, 9, cfg)
    env, pf = _loaded(scenes, cfg)
    got = _np(env.upper_bound())
    val, cost = scenes["tgt_value"][:, 0], scenes["uav_cost"]
    any_p = (pf[:, :, 0] > 0).any(axis=1)
    assert any_p.sum() >= S // 2
    for s in range(S):
        J_all = val[s] * (1.0 - math.prod((1.0 - pf[s, :, 0]).tolist()))
        margin = val[s] * math.exp(-AMAX) + 1e-12 * val[s]
        assert got["bound"][s] == pytest.approx(J_all + margin, rel=1e-12, abs=1e-12), s
        assert got["relaxed"][s] == pytest.approx(J_all, rel=1e-12, abs=1e-12), s
        assert got["iters"][s] == (2 if any_p[s] else 1), s
    env.close()


@pytest.mark.gpu
def test_all_gradients_negative_gives_the_margin():
    """omega so large that every g < 0 at the empty allocation: no UAV picks, U_1 = F = 0, one iteration, and the bound is
    the margin alone; the optimum is the empty allocation, J* = 0."""
    omega = 1e6
    cfg = ub.Config(NUM_UAVS=4, NUM_TARGETS=3, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(8, 13, cfg)
    env, pf = _loaded(scenes, cfg)
    got = _np(env.upper_bound())
    for s in range(8):
        tv, tc = _seq(scenes["tgt_value"][s]), _seq(scenes["uav_cost"][s])
        margin = tv * math.exp(-AMAX) + 1e-12 * (tv + omega * tc)
        assert got["bound"][s] == pytest.approx(margin, rel=1e-15) and got["relaxed"][s] == 0.0 and got["iters"][s] == 1
        assert _brute_force(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega) == 0.0
    env.close()


# ---- 4: monotone in iters, launch independence -------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(30, 10), (256, 256)])
def test_bound_is_monotone_in_iters(shape):
    """A run with cap b repeats the first a iterations of a run with cap a < b bit for bit, so its bound (a minimum over
    more iterations) is no larger; where the run with cap a stopped early, both runs stop there with equal bits."""
    N, M = shape
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=0.5)
    scenes = _scenes(48, 19, cfg)
    env, _ = _loaded(scenes, cfg)
    caps = (1, 2, 3, 8, 64, 256, 1024)
    got = {c: _np(env.upper_bound(iters=c)) for c in caps}
    for a, b in zip(caps, caps[1:]):
        assert (got[b]["bound"] <= got[a]["bound"]).all(), (a, b)
        early = got[a]["iters"] < a
        for k in got[a]:
            x, y = got[a][k][early], got[b][k][early]
            assert np.array_equal(_bits(x) if x.dtype == np.float64 else x, _bits(y) if y.dtype == np.float64 else y), (a, b)
    assert (got[1024]["bound"] < got[1]["bound"]).any()
    print("\n[bound %dx%d] bound by cap: %s" % (N, M, ", ".join("%d: %.4f" % (c, got[c]["bound"].mean()) for c in caps)))
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(30, 10), (256, 256)])
def test_bits_do_not_depend_on_count_stride_or_chunking(shape):
    N, M = shape
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=0.5)
    S, K = 40, 3
    scenes = _scenes(S, 17, cfg)
    one, _ = _loaded(scenes, cfg)
    rep = ub.UAVEnvBatched(S * K, seed=0, config=cfg, auto_reset=False)
    rep.load_scene_device({k: torch.as_tensor(v).cuda() for k, v in scenes.items()}, copies=K)
    a, b = _np(one.upper_bound(iters=64)), _np(one.upper_bound(iters=64))
    c = _np(rep.upper_bound(first_env=K - 1, count=S, env_stride=K, iters=64))
    parts = [_np(one.upper_bound(first_env=lo, count=hi - lo, iters=64)) for lo, hi in ((0, 7), (7, 8), (8, 40))]
    d = {k: np.concatenate([p[k] for p in parts]) for k in a}
    e = ub.upper_bound(scenes, iters=64, config=cfg, max_envs=9)
    for other in (b, c, d, e):
        for k in a:
            x, y = a[k], other[k]
            assert np.array_equal(_bits(x) if x.dtype == np.float64 else x, _bits(y) if y.dtype == np.float64 else y), k
    one.close()
    rep.close()


# ---- 5: argument checks on a live handle -------------------------------------------------------------------------------

@pytest.mark.gpu
def test_argument_checks_on_a_live_handle():
    big = ub.Config(NUM_UAVS=256, NUM_TARGETS=256)
    env = ub.UAVEnvBatched(4, seed=0, config=big, auto_reset=False)
    L, h, d = env._lib, env._h, env.device
    f64 = torch.empty(4, dtype=torch.float64, device=d)
    i32 = torch.empty(4, dtype=torch.int32, device=d)
    ws = torch.empty(L.uavenv_improve_workspace_bytes(h), dtype=torch.uint8, device=d)
    P = lambda t: C.c_void_p(t.data_ptr())       # noqa: E731

    def call(first=0, count=4, stride=1, iters=8, bo=P(f64), r=P(f64), it=P(i32), w=P(ws)):
        return L.uavenv_upper_bound(h, first, count, stride, iters, bo, r, it, w, None)

    assert call() == ERR["UAVENV_ESTATE"]                     # no reset / scene load yet
    env.reset(full_reset=True)
    torch.cuda.synchronize()
    assert call() == 0
    torch.cuda.synchronize()
    for kw in ({"bo": None}, {"r": None}, {"it": None}, {"w": None}, {"count": 0}, {"stride": 0}, {"iters": 0},
               {"first": -1}, {"first": 1}, {"count": 3, "stride": 2}, {"first": 4, "count": 1}):
        assert call(**kw) == ERR["UAVENV_EINVAL"], kw
    assert b"uavenv_upper_bound" in L.uavenv_last_error(h)
    assert call(count=2, stride=3) == 0
    torch.cuda.synchronize()
    env.close()


# ---- 6: no GPU needed ------------------------------------------------------------------------------------------------

def test_symbol_declared_and_exported():
    text = open(os.path.join(ROOT, "include", "uavenv_b200.h")).read()
    assert re.search(r"\buavenv_upper_bound\s*\(", text)
    assert hasattr(ub.load_library(), "uavenv_upper_bound")


def test_null_handle_call():
    L = ub.load_library()
    assert L.uavenv_upper_bound(None, 0, 1, 1, 1, None, None, None, None, None) == ERR["UAVENV_EINVAL"]


def test_lazy_export():
    first, second = ub.upper_bound, ub.upper_bound
    assert callable(first) and first is second
    from target_allocation_ppo_transformer_b200 import allocation
    assert first is allocation.upper_bound


def test_upper_bound_rejects_bad_arguments():
    scenes = {"uav_x": np.zeros((2, 30))}
    for kw in ({"scenes": {}}, {"scenes": {"uav_x": np.zeros(7)}}, {"scenes": scenes, "iters": 0},
               {"scenes": scenes, "max_envs": 0}):
        with pytest.raises(ValueError):
            ub.upper_bound(**kw)
    with pytest.raises(RuntimeError):
        ub.upper_bound(scenes, device="cpu")
