"""Local search on allocations (uavenv_improve_allocation, ub.improve_allocation, ub.allocate(improve=True)): every applied
move against an fp64 numpy re-implementation of the rule in include/uavenv_b200.h (at the configs, at every shape class
of the candidate walk and of p's home, on a CTA's later scenes, on exact ties and under a cap that stops mid-search),
local optimality at 64x64 (p in shared memory) and 256x256 (p in the workspace), max_moves = 0, determinism and layout
independence, flagged rows, argument checks, and allocate's improve path.  The CPU tests at the end need no GPU."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT

import uavenv_b200 as ub


def _error_codes():
    text = open(os.path.join(ROOT, "include", "uavenv_b200.h")).read()
    return {name: int(v) for name, v in re.findall(r"\b(UAVENV_E[A-Z]+)\s*=\s*(-?\d+)", text)}


ERR = _error_codes()
NEAR = 1e-9          # relative gap of a round's two best gains below which a scene is left out of the exact comparison
CONFIGS = {"30x10": {}, "30x10_omega05": {"COST_WEIGHT_OMEGA": 0.5}, "hard_omega05": dict(ub.HARD_MODE, COST_WEIGHT_OMEGA=0.5),
           "hard_omega2": dict(ub.HARD_MODE, COST_WEIGHT_OMEGA=2.0), "64x8": {"NUM_UAVS": 64, "NUM_TARGETS": 8},
           "tiny_3x2": {"NUM_UAVS": 3, "NUM_TARGETS": 2}, "tiny_4x1": {"NUM_UAVS": 4, "NUM_TARGETS": 1}}


# ---- the fp64 reference of the search rule ---------------------------------------------------------------------------

def _prod(p, t, j, skip=-1):
    """Product over UAVs i != skip on target j of (1 - p[i, j]) in ascending i (math.prod multiplies in order)."""
    return math.prod((1.0 - p[[i for i in range(len(t)) if t[i] == j and i != skip], j]).tolist(), start=1.0)


def _J(nh, val, cost, t, omega):
    rev = 0.0
    for j in range(len(nh)):
        rev += (1.0 - nh[j]) * val[j]
    c = 0.0
    for k in range(len(t)):
        if t[k] >= 0:
            c += cost[k]
    return rev - omega * c


def _gains(p, t, nh, nhx, val, cost, omega):
    """Gains of every candidate in candidate order (moves [N, M+1] row-major, then swaps (k1 < k2) lexicographic);
    -inf where the candidate does not exist.  Elementwise in the kernel's operation order."""
    N, M = p.shape
    a = np.asarray(t)
    ac = np.maximum(a, 0)
    on = (a >= 0).astype(np.float64)
    ga = np.where(a >= 0, val[ac] * (nh[ac] - nhx), 0.0)
    gb = np.concatenate([np.zeros((N, 1)), (val * nh)[None, :] * p], axis=1)
    ind = on[:, None] - np.concatenate([[0.0], np.ones(M)])[None, :]
    mv = (ga[:, None] + gb) + (omega * cost)[:, None] * ind
    mv[np.arange(N), a + 1] = -np.inf
    ks = np.arange(N)
    g1 = np.where((a >= 0)[:, None], val[ac][:, None] * (nh[ac][:, None] - nhx[:, None] * (1.0 - p[ks[None, :], ac[:, None]])),
                  0.0)
    g2 = np.where((a >= 0)[None, :], val[ac][None, :] * (nh[ac][None, :] - nhx[None, :] * (1.0 - p[ks[:, None], ac[None, :]])),
                  0.0)
    sw = (g1 + g2) + (omega * (cost[:, None] - cost[None, :])) * (on[:, None] - on[None, :])
    sw = np.where(a[:, None] != a[None, :], sw, -np.inf)
    iu = np.triu_indices(N, 1)
    return np.concatenate([mv.reshape(-1), sw[iu]]), iu


def ref_search(p, val, cost, omega, t0, max_moves, last_wins_tie=False):
    """(t, moves, converged, J_in, J_out, near, kinds) of the search from t0 (target positions, -1 = none).  kinds counts
    moves to -1, swaps with an unassigned side and applied rounds whose best gain two or more candidates reach exactly
    ("ties", their candidate indices in "tied").  last_wins_tie gives an exact tie to the highest candidate index: a
    mutant of the rule, for showing that a test meets ties."""
    N, M = p.shape
    t = list(int(x) for x in t0)
    nh = np.array([_prod(p, t, j) for j in range(M)])
    nhx = np.array([_prod(p, t, t[k], k) if t[k] >= 0 else 1.0 for k in range(N)])
    J_in = _J(nh, val, cost, t, omega)
    J, moves, near = J_in, 0, False
    kinds = {"to_none": 0, "swap_none": 0, "moves": 0, "swaps": 0, "ties": 0, "tied": []}
    while True:
        g, iu = _gains(p, t, nh, nhx, val, cost, omega)
        c = g.size - 1 - int(np.argmax(g[::-1])) if last_wins_tie else int(np.argmax(g))
        best = g[c]
        if not best > 1e-12 * max(1.0, abs(J)):
            conv = True
            break
        if moves >= max_moves:
            conv = False
            break
        second = np.max(np.delete(g, c)) if g.size > 1 else -np.inf
        # (an exact tie is no exclusion: both sides compute the same bits, and the candidate order decides)
        near |= bool(0.0 < best - second <= NEAR * max(abs(best), abs(second)))
        if second == best:
            kinds["ties"] += 1
            kinds["tied"].append(np.flatnonzero(g == best))
        moves += 1
        J += best
        if c < N * (M + 1):
            k1, b = divmod(c, M + 1)
            touched = (t[k1], b - 1)
            t[k1] = b - 1
            kinds["moves"] += 1
            kinds["to_none"] += b == 0
        else:
            k1, k2 = int(iu[0][c - N * (M + 1)]), int(iu[1][c - N * (M + 1)])
            touched = (t[k1], t[k2])
            t[k1], t[k2] = t[k2], t[k1]
            kinds["swaps"] += 1
            kinds["swap_none"] += min(touched) < 0
        for j in touched:
            if j >= 0:
                nh[j] = _prod(p, t, j)
        for k in range(N):
            if t[k] < 0:
                nhx[k] = 1.0
            elif t[k] in touched:
                nhx[k] = _prod(p, t, t[k], k)
    return np.array(t), moves, conv, J_in, _J(nh, val, cost, t, omega), near, kinds


def test_reference_search_on_a_hand_made_scene():
    """The reference itself (no GPU): a swap, a move to none and a covering move on a 3 x 2 scene whose optimum is known."""
    p = np.array([[0.9, 0.1], [0.2, 0.8], [0.5, 0.5]])
    val, cost = np.array([1.0, 1.0]), np.array([0.1, 0.1, 5.0])
    t, moves, conv, J_in, J_out, _, kinds = ref_search(p, val, cost, 0.1, [1, 0, 0], 100)
    assert conv and list(t) == [0, 1, -1] and moves >= 2 and J_out > J_in
    assert J_out == pytest.approx(0.9 + 0.8 - 0.1 * 0.2)
    g, _ = _gains(p, list(t), np.array([0.1, 0.2]), np.ones(3), val, cost, 0.1)
    assert g.max() <= 1e-12
    t, moves, conv, *_ = ref_search(p, val, cost, 0.1, [1, 0, 0], 0)
    assert list(t) == [1, 0, 0] and moves == 0 and not conv


# ---- fixtures -------------------------------------------------------------------------------------------------------

def _scenes(S, seed, cfg):
    gen = ub.UAVEnvBatched(S, seed=seed, config=cfg, auto_reset=False)
    gen.reset(full_reset=True)
    sc = gen.get_scene()
    gen.close()
    return sc


def _loaded(scenes, cfg):
    """An env holding the scenes, and their fp64 p_final [S, N, M] (list order)."""
    S = scenes["uav_x"].shape[0]
    env = ub.UAVEnvBatched(S, seed=0, config=cfg, auto_reset=False)
    env.load_scene(scenes)
    return env, env.score_matrix(torch.float64)[0].cpu().numpy()


def _random_rows(scenes, rng, p_none=None):
    ids = scenes["tgt_id"]
    S, M = ids.shape
    N = scenes["uav_x"].shape[1]
    pos = rng.integers(-1, M, size=(S, N))
    if p_none is not None:
        pos = np.where(rng.random((S, N)) < p_none, -1, np.maximum(pos, 0))
    return np.where(pos >= 0, np.take_along_axis(ids, np.maximum(pos, 0), axis=1), -1).astype(np.int32)


def _positions(rows, ids):
    lut = [{int(v): j for j, v in enumerate(r)} for r in ids]
    return np.array([[lut[s][int(x)] if x >= 0 else -1 for x in row] for s, row in enumerate(rows)])


def _net(seed=0):
    torch.manual_seed(seed)
    return ub.TransformerActorCritic()


def _np(res):
    return {k: v.cpu().numpy() for k, v in res.items()}


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.int64)


# ---- 1: move by move against the reference -----------------------------------------------------------------------------

def _check(got, scenes, pf, rows, omega, max_moves, label, kinds=None, idx=None):
    """Checks the kernel's results got (entry i: scene idx[i], default every scene) of a search from rows [S, N] against
    ref_search: J_before to 1e-12 for every scene; the rows, moves, converged, N0 exactly and J to 1e-12.  A scene in
    which some round's two best gains lie within NEAR without being equal may differ (a last-bit difference could pick
    either) and is then left out.  Returns (the scenes that matched, the scenes with such a near tie), and adds the
    reference's counts of the matched scenes to kinds."""
    idx = list(range(len(rows))) if idx is None else list(idx)
    pos = _positions(np.asarray(rows)[idx], scenes["tgt_id"][idx])
    kept, nears = [], []
    for i, s in enumerate(idx):
        t, moves, conv, J_in, J_out, near, kd = ref_search(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega,
                                                           pos[i], max_moves)
        assert got["J_before"][i] == pytest.approx(J_in, rel=1e-12, abs=1e-12), (label, s)
        want = np.where(t >= 0, scenes["tgt_id"][s][np.maximum(t, 0)], -1)
        ok = {"rows": np.array_equal(got["assigned_target_id"][i], want),
              "moves": got["moves"][i] == moves and bool(got["converged"][i]) == conv,
              "J": got["J"][i] == pytest.approx(J_out, rel=1e-12, abs=1e-12),
              "N0": got["num_covered"][i] == len(set(t[t >= 0].tolist()))}
        if near:
            nears.append(s)
            if not all(ok.values()):
                continue
        assert all(ok.values()), (label, s, ok, got["moves"][i], moves)
        kept.append(s)
        for k in kinds or ():
            kinds[k] += kd[k]
    return kept, nears


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_search_equals_fp64_reference(name):
    """Final rows, move counts and converged flags equal the reference's exactly and J to 1e-12, from empty, random and
    allocate() allocations; scenes whose two best gains of some round lie within NEAR (but are not equal) are counted and
    left out when they differ.  With omega > 0 moves to none occur; swaps with an unassigned side need a UAV whose cost
    outweighs a positive contribution, which the default scenes have at omega = 0.5 (HARD_MODE's p_final is almost
    everywhere 0 at 30 x 10, so there every gain is a cost and single moves to none always win)."""
    cfg = ub.Config(**CONFIGS[name])
    S, omega = 48, float(cfg.COST_WEIGHT_OMEGA)
    scenes = _scenes(S, 71, cfg)
    env, pf = _loaded(scenes, cfg)
    N = env.N
    rng = np.random.default_rng(5)
    inputs = {"empty": np.full((S, N), -1, np.int32), "random": _random_rows(scenes, rng),
              "allocate": ub.allocate(_net(2), scenes=scenes, samples=2, seed=4, config=cfg)["assigned_target_id"]}
    kinds = {"to_none": 0, "swap_none": 0, "moves": 0, "swaps": 0}
    excluded = near = 0
    for label, rows in inputs.items():
        kept, nears = _check(_np(env.improve_allocation(rows)), scenes, pf, rows, omega, 16 * N, label, kinds)
        excluded, near = excluded + S - len(kept), near + len(nears)
    print("\n[improve %s] moves %d (to none %d), swaps %d (an unassigned side %d), near-tie scenes %d, excluded %d of %d" % (
        name, kinds["moves"], kinds["to_none"], kinds["swaps"], kinds["swap_none"], near, excluded, 3 * S))
    # HARD_MODE's p_final is almost everywhere ~0, so its gains are costs apart by terms of ~1e-10: most near-ties are there
    assert excluded <= max(2, 3 * S // 8)
    assert kinds["moves"] > 0
    if float(cfg.COST_WEIGHT_OMEGA) > 0:
        assert kinds["to_none"] > 0
    if name == "30x10_omega05":
        assert kinds["swap_none"] > 0
    env.close()


# Shapes at which the kernel's candidate walk or p's home changes.  Each of the 256 threads steps through the moves by
# dq UAV rows and dr targets, divmod(256, M + 1), and through the swaps by 256, skipping whole short rows; p is in shared
# memory while N * M * 8 <= 64 KB, else in the workspace.  (N, M, omega, scenes per input, p in, dq, dr)
SHAPES = [(1, 7, 0.25, 48, "shared", 32, 0),            # no swaps at all
          (8, 300, 0.25, 32, "shared", 0, 256),         # M + 1 > 256; fewer swaps (28) than threads
          (16, 255, 0.25, 32, "shared", 1, 0),          # M + 1 = 256
          (40, 63, 0.25, 32, "shared", 4, 0),           # M + 1 = 64 divides 256
          (64, 64, 0.25, 24, "shared", 3, 61),          # the largest square on the shared path
          (64, 64, 2.0, 24, "shared", 3, 61),           # moves to none and swaps with an unassigned side are common
          (128, 64, 0.25, 12, "shared", 3, 61),         # N * M * 8 = 64 KB: the last shape on the shared path
          (129, 64, 0.25, 12, "workspace", 3, 61),      # the first shapes on the workspace path
          (64, 129, 0.25, 12, "workspace", 1, 126),
          (300, 4, 0.25, 10, "shared", 51, 1),          # N > 256: the per-UAV loops take two passes; 44 850 swaps
          (256, 256, 0.25, 10, "workspace", 0, 256)]    # BASELINE config 5


def _shape_id(N, M, omega, S, path, dq, dr):
    return "%dx%d%s-%s-dq%d-dr%d" % (N, M, "" if omega == 0.25 else "_omega%g" % omega, path, dq, dr)


def _perturbed(rows, ids, rng, frac=0.05):
    """rows with max(1, round(frac * N)) UAVs of each scene put on a random target or none."""
    rows = rows.copy()
    S, N = rows.shape
    n = max(1, round(frac * N))
    for s in range(S):
        pos = rng.integers(-1, ids.shape[1], n)
        rows[s, rng.choice(N, n, replace=False)] = np.where(pos >= 0, ids[s][np.maximum(pos, 0)], -1)
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,omega,S,path,dq,dr", [pytest.param(*c, id=_shape_id(*c)) for c in SHAPES])
def test_shape_classes_equal_fp64_reference(N, M, omega, S, path, dq, dr):
    """test_search_equals_fp64_reference's exact comparison where the candidate walk and p's home change form, from
    empty rows, random rows, a pile-up (every UAV on the first target: the longest products) and a perturbed optimum
    (the kernel's result for the random rows with ~5 % of the UAVs moved: gains near the threshold)."""
    assert divmod(256, M + 1) == (dq, dr)
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 61, cfg)
    env, pf = _loaded(scenes, cfg)
    assert (env._lib.uavenv_improve_workspace_bytes(env._h) == 0) == (path == "shared")
    ids, rng = scenes["tgt_id"], np.random.default_rng(1000 * N + M)
    rows = {"empty": np.full((S, N), -1, np.int32), "random": _random_rows(scenes, rng, p_none=0.5),
            "pileup": np.ascontiguousarray(np.repeat(ids[:, :1], N, axis=1))}
    kinds = {"to_none": 0, "swap_none": 0, "moves": 0, "swaps": 0}
    got, excluded = {}, 0
    for label in ("empty", "random", "pileup", "perturbed"):
        if label == "perturbed":
            rows[label] = _perturbed(got["random"]["assigned_target_id"], ids, rng)
        got[label] = _np(env.improve_allocation(rows[label]))
        kept, nears = _check(got[label], scenes, pf, rows[label], omega, 16 * N, label, kinds)
        excluded += S - len(kept)
        print("\n[improve %s] %s: %d of %d scenes equal (%d with a near tie), %d excluded, moves/scene %.1f" % (
            _shape_id(N, M, omega, S, path, dq, dr), label, len(kept), S, len(nears), S - len(kept),
            got[label]["moves"].mean()), end="")
    print("\n  moves %d (to none %d), swaps %d (an unassigned side %d)" % (
        kinds["moves"], kinds["to_none"], kinds["swaps"], kinds["swap_none"]))
    assert excluded <= max(2, 4 * S // 8)
    assert kinds["moves"] > 0 and (kinds["swaps"] > 0) == (N > 1)
    if omega == 2.0:
        assert kinds["to_none"] > 0 and kinds["swap_none"] > 0
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,waves,extra", [((256, 256), 2, 7), ((64, 64), 8, 50)], ids=["256x256", "64x64"])
def test_later_scenes_of_a_cta_equal_fp64_reference(shape, waves, extra):
    """A persistent CTA reuses its workspace slice (256x256: the grid is one CTA per SM) or its shared memory (64x64: at
    most 8 CTAs per SM) for its next scene.  waves * SMs + extra scenes in one call, so the last ones are some CTA's
    second or later scene; the scenes around each multiple of the SM count, the last and a few random ones equal the
    reference, and each alone in a call (the first scene of CTA 0) gives the same bits."""
    N, M = shape
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    S, omega = waves * sms + extra, 0.25
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 37, cfg)
    env, pf = _loaded(scenes, cfg)
    rng = np.random.default_rng(N)
    rows = _random_rows(scenes, rng, p_none=0.5)
    got = _np(env.improve_allocation(rows))
    sub = sorted({0, S - 1} | {c * sms + d for c in range(1, waves + 1) for d in (-1, 0, 1)} |
                 set(rng.choice(S, 4, replace=False).tolist()))
    kept, nears = _check({k: v[sub] for k, v in got.items()}, scenes, pf, rows, omega, 16 * N, "later scenes", idx=sub)
    print("\n[improve %dx%d, %d scenes, %d SMs] %d of %d checked scenes equal (%d with a near tie)" % (
        N, M, S, sms, len(kept), len(sub), len(nears)))
    assert len(sub) - len(kept) <= max(2, len(sub) // 8)
    for s in sub:
        one = _np(env.improve_allocation(rows[s:s + 1], first_env=s))
        for k in got:
            if got[k].dtype == np.float64:
                assert np.array_equal(_bits(got[k][s:s + 1]), _bits(one[k])), (k, s)
            else:
                assert np.array_equal(got[k][s:s + 1], one[k]), (k, s)
    env.close()


@pytest.mark.gpu
def test_exact_ties_go_to_the_lowest_candidate_index():
    """Generated 64x63 scenes (M + 1 = 64) in which UAVs 1 and 4 copy UAV 0 and target 40 copies target 3's position,
    velocity and value (keeping its id).  Equal candidates of UAVs 0, 1 and 4 are 64 (other warps) and 256 (the same
    thread) apart, so the in-thread first maximum, the warp arg-max and the cross-warp reduction each meet exact ties;
    the rounds where each does are counted from the reference's tied candidates.  The kernel equals the reference, and a
    reference that gives a tie to the highest index does not."""
    N, M, S, omega = 64, 63, 64, 0.25
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 43, cfg)
    for f in scenes:
        if f.startswith("uav_"):
            scenes[f][:, [1, 4]] = scenes[f][:, :1]
        elif f.startswith("tgt_") and f != "tgt_id":
            scenes[f][:, 40] = scenes[f][:, 3]
    env, pf = _loaded(scenes, cfg)
    for a, b in ((pf[:, 0], pf[:, 1]), (pf[:, 0], pf[:, 4]), (pf[:, :, 3], pf[:, :, 40])):
        assert np.array_equal(_bits(a), _bits(b))
    rows = {"empty": np.full((S, N), -1, np.int32), "random": _random_rows(scenes, np.random.default_rng(9), p_none=0.5)}
    kinds = {"ties": 0, "tied": []}
    compared = rejected = 0
    for label in rows:
        got = _np(env.improve_allocation(rows[label]))
        kept, _ = _check(got, scenes, pf, rows[label], omega, 16 * N, label, kinds)
        pos = _positions(rows[label], scenes["tgt_id"])
        for s in kept:
            t, moves, *_ = ref_search(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega, pos[s], 16 * N,
                                      last_wins_tie=True)
            want = np.where(t >= 0, scenes["tgt_id"][s][np.maximum(t, 0)], -1)
            rejected += not (np.array_equal(got["assigned_target_id"][s], want) and got["moves"][s] == moves)
        compared += len(kept)
    n_moves, stage = N * (M + 1), {"thread": 0, "warp": 0, "block": 0}
    for c in kinds["tied"]:
        th = np.where(c < n_moves, c, c - n_moves) % 256                   # the thread that scores candidate c
        w = th // 32
        stage["thread"] += len(np.unique(th)) < len(th)
        stage["warp"] += any(len(np.unique(th[w == x])) > 1 for x in np.unique(w))
        stage["block"] += len(np.unique(w)) > 1
    print("\n[improve ties 64x63] %d of %d scenes equal; %d rounds with an exact tie (in a thread %d, in a warp "
          "%d, across warps %d); the highest-index-wins reference disagrees on %d scenes" % (
              compared, 2 * S, kinds["ties"], stage["thread"], stage["warp"], stage["block"], rejected))
    assert 2 * S - compared <= max(2, 2 * S // 8)
    assert kinds["ties"] >= 8 and min(stage.values()) > 0
    assert rejected > 0
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(64, 64), (256, 256)], ids=["64x64", "256x256"])
def test_cap_stops_at_the_reference_state_mid_search(shape):
    """max_moves = half the reference's moves from random rows: the rows, J, N0 and moves after exactly that many moves,
    converged = False."""
    N, M = shape
    S, omega = 16 if N == 64 else 8, 0.25
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=omega)
    scenes = _scenes(S, 53, cfg)
    env, pf = _loaded(scenes, cfg)
    rows = _random_rows(scenes, np.random.default_rng(3), p_none=0.5)
    pos = _positions(rows, scenes["tgt_id"])
    compared = 0
    for s in range(S):
        cap = ref_search(pf[s], scenes["tgt_value"][s], scenes["uav_cost"][s], omega, pos[s], 16 * N)[1] // 2
        assert cap > 0
        got = _np(env.improve_allocation(rows[s:s + 1], first_env=s, max_moves=cap))
        assert got["moves"][0] == cap and not got["converged"][0]
        compared += len(_check(got, scenes, pf, rows, omega, cap, "cap %d" % cap, idx=[s])[0])
    print("\n[improve %dx%d cap] %d of %d scenes equal" % (N, M, compared, S))
    assert S - compared <= max(2, S // 8)
    env.close()


# ---- 2: local optimality at scale -----------------------------------------------------------------------------------

def _max_gain(p, t, val, cost, omega):
    N, M = p.shape
    nh = np.ones(M)
    for i in range(N):
        if t[i] >= 0:
            nh[t[i]] *= 1.0 - p[i, t[i]]
    nhx = np.array([_prod(p, t, t[k], k) if t[k] >= 0 else 1.0 for k in range(N)])
    return _gains(p, t, nh, nhx, val, cost, omega)[0].max()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(64, 64), (256, 256)])
def test_local_optimum_at_scale(shape):
    """64x64 keeps p in shared memory, 256x256 in the workspace.  Converged rows admit no qualifying move or swap
    (recomputed in numpy), J never falls, J equals J recomputed from the rows, ids are scene ids or -1, N0 counts them."""
    N, M = shape
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=0.25)
    S = 256
    scenes = _scenes(S, 81, cfg)
    env, pf = _loaded(scenes, cfg)
    rows = _random_rows(scenes, np.random.default_rng(8), p_none=0.5)
    ws = env._lib.uavenv_improve_workspace_bytes(env._h)
    assert (ws == 0) == (N * M * 8 <= 64 * 1024)
    res = ub.improve_allocation(scenes, rows, config=cfg)
    assert np.array_equal(res["J_before"], _np(env.improve_allocation(rows, max_moves=0))["J"])
    assert (res["J"] >= res["J_before"]).all() and (res["moves"] > 0).all()
    assert res["converged"].mean() > 0.9
    omega = float(cfg.COST_WEIGHT_OMEGA)
    pos = _positions(res["assigned_target_id"], scenes["tgt_id"])
    for s in range(S):
        val, cost = scenes["tgt_value"][s], scenes["uav_cost"][s]
        nh = np.ones(M)
        for i in range(N):
            if pos[s, i] >= 0:
                nh[pos[s, i]] *= 1.0 - pf[s, i, pos[s, i]]
        J = float(np.sum(val * (1.0 - nh))) - omega * float(np.sum(cost[pos[s] >= 0]))
        assert res["J"][s] == pytest.approx(J, rel=1e-9), s
        assert res["num_covered"][s] == len(set(pos[s][pos[s] >= 0].tolist()))
        if res["converged"][s] and s % 8 == 0:
            assert _max_gain(pf[s], list(pos[s]), val, cost, omega) <= 1e-12 * max(1.0, abs(res["J"][s])) * (1 + 1e-6)
    ids = set(np.unique(scenes["tgt_id"]).tolist()) | {-1}
    assert set(np.unique(res["assigned_target_id"]).tolist()) <= ids
    print("\n[improve %dx%d] J %.4f -> %.4f, moves %.1f, converged %.3f, %.0f scenes/s" % (
        N, M, res["summary"]["J_before_mean"], res["summary"]["J_mean"], res["summary"]["moves_mean"],
        res["summary"]["converged_frac"], res["summary"]["scenes_per_s"]))
    env.close()


# ---- 3: max_moves = 0 ----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["30x10", "hard_omega05"])
def test_max_moves_zero_returns_the_input_and_group_best_J(name):
    cfg = ub.Config(**CONFIGS[name])
    S, K = 64, 4
    scenes = _scenes(S, 91, cfg)
    env = ub.UAVEnvBatched(S * K, seed=2, config=cfg, auto_reset=False)
    env.load_scene_device({k: torch.as_tensor(v).cuda() for k, v in scenes.items()}, copies=K)
    for step in range(env.N * env.M):
        _, _, done, _ = env.step(env.random_actions(step, action_seed=3))
        if bool(done.all()):
            break
    gb = env.group_best(K, 0, S)
    res = _np(env.improve_allocation(gb["assigned_target_id"], env_stride=K, max_moves=0))
    gb = _np(gb)
    assert np.array_equal(res["assigned_target_id"], gb["assigned_target_id"])
    assert (res["moves"] == 0).all() and np.array_equal(_bits(res["J"]), _bits(res["J_before"]))
    np.testing.assert_allclose(res["J_before"], gb["J"], rtol=1e-9, atol=1e-12)
    assert np.array_equal(res["num_covered"], gb["num_covered"])
    env.close()


# ---- 4: determinism and layout independence ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(30, 10), (256, 256)])
def test_bits_do_not_depend_on_call_stride_or_chunking(shape):
    N, M = shape
    cfg = ub.Config(NUM_UAVS=N, NUM_TARGETS=M, COST_WEIGHT_OMEGA=0.5)
    S, K = 40, 3
    scenes = _scenes(S, 17, cfg)
    rows = torch.as_tensor(_random_rows(scenes, np.random.default_rng(1))).cuda()
    one = ub.UAVEnvBatched(S, seed=0, config=cfg, auto_reset=False)
    one.load_scene(scenes)
    rep = ub.UAVEnvBatched(S * K, seed=0, config=cfg, auto_reset=False)
    rep.load_scene_device({k: torch.as_tensor(v).cuda() for k, v in scenes.items()}, copies=K)
    a, b = _np(one.improve_allocation(rows)), _np(one.improve_allocation(rows))
    c = _np(rep.improve_allocation(rows, first_env=K - 1, env_stride=K))
    parts = [_np(one.improve_allocation(rows[lo:hi], first_env=lo)) for lo, hi in ((0, 7), (7, 8), (8, 40))]
    d = {k: np.concatenate([p[k] for p in parts]) for k in a}
    for other in (b, c, d):
        for k in a:
            if a[k].dtype == np.float64:
                assert np.array_equal(_bits(a[k]), _bits(other[k])), k
            else:
                assert np.array_equal(a[k], other[k]), k
    assert (a["moves"] > 0).any()
    one.close()
    rep.close()


# ---- 5: flagged rows and argument checks on a live handle ---------------------------------------------------------------

@pytest.mark.gpu
def test_invalid_rows_are_flagged_and_neighbours_unchanged():
    cfg = ub.Config()
    S = 8
    scenes = _scenes(S, 23, cfg)
    env, _ = _loaded(scenes, cfg)
    rows = _random_rows(scenes, np.random.default_rng(2))
    clean = _np(env.improve_allocation(rows))
    bad = rows.copy()
    bad[2, 5] = 10_000
    bad[5, 0] = -2
    got = _np(env.improve_allocation(bad))
    for s in (2, 5):
        assert (got["assigned_target_id"][s] == -1).all() and got["moves"][s] == -1 and got["num_covered"][s] == -1
        assert np.isnan(got["J"][s]) and np.isnan(got["J_before"][s]) and not got["converged"][s]
    keep = [s for s in range(S) if s not in (2, 5)]
    for k in clean:
        assert np.array_equal(_bits(clean[k][keep]) if clean[k].dtype == np.float64 else clean[k][keep],
                              _bits(got[k][keep]) if got[k].dtype == np.float64 else got[k][keep]), k
    res = ub.improve_allocation(scenes, bad)
    assert res["summary"]["invalid_rows"] == 2 and np.isfinite(res["summary"]["J_mean"])
    env.close()


@pytest.mark.gpu
def test_argument_checks_on_a_live_handle():
    big = ub.Config(NUM_UAVS=256, NUM_TARGETS=256)
    env = ub.UAVEnvBatched(4, seed=0, config=big, auto_reset=False)
    L, h, d = env._lib, env._h, env.device
    rows = torch.full((4, 256), -1, dtype=torch.int32, device=d)
    i32 = torch.empty(4, dtype=torch.int32, device=d)
    f64 = torch.empty(4, dtype=torch.float64, device=d)
    u8 = torch.empty(4, dtype=torch.uint8, device=d)
    out = torch.empty_like(rows)
    ws_bytes = L.uavenv_improve_workspace_bytes(h)
    assert ws_bytes >= 256 * 256 * 8
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=d)
    P = lambda t: C.c_void_p(t.data_ptr())       # noqa: E731

    def call(first=0, count=4, stride=1, max_moves=10, a=P(rows), o=P(out), jo=P(f64), w=P(ws)):
        return L.uavenv_improve_allocation(h, first, count, stride, a, max_moves, o, P(f64), jo, P(i32), P(i32), P(u8), w,
                                           None)

    assert call() == ERR["UAVENV_ESTATE"]                     # no reset / scene load yet
    env.reset(full_reset=True)
    torch.cuda.synchronize()
    assert call() == 0
    torch.cuda.synchronize()
    for kw in ({"a": None}, {"o": None}, {"jo": None}, {"w": None}, {"count": 0}, {"stride": 0}, {"max_moves": -1},
               {"first": -1}, {"first": 1}, {"count": 3, "stride": 2}, {"first": 4, "count": 1}):
        assert call(**kw) == ERR["UAVENV_EINVAL"], kw
    assert call(count=2, stride=3) == 0
    torch.cuda.synchronize()
    env.close()


# ---- 6: allocate(improve=True) ----------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["30x10", "30x10_omega05"])
def test_allocate_improve(name):
    cfg = ub.Config(**CONFIGS[name])
    S, K, net = 200, 4, _net(3)
    scenes = _scenes(S, 29, cfg)
    plain = ub.allocate(net, scenes=scenes, samples=K, seed=6, config=cfg, max_envs=256)
    imp = ub.allocate(net, scenes=scenes, samples=K, seed=6, config=cfg, max_envs=256, improve=True)
    assert np.array_equal(plain["best_sample"], imp["best_sample"])
    assert np.array_equal(_bits(plain["J_samples"]), _bits(imp["J_samples"]))
    assert np.array_equal(_bits(plain["J"]), _bits(imp["J_before_improve"]))
    assert (imp["J"] >= plain["J"]).all() and (imp["J"] > plain["J"]).any()
    pol = ub.improve_allocation(scenes, plain["assigned_target_id"], config=cfg)
    assert np.array_equal(imp["assigned_target_id"], pol["assigned_target_id"])
    assert np.array_equal(_bits(imp["J"]), _bits(pol["J"]))
    assert np.array_equal(imp["moves"], pol["moves"]) and np.array_equal(imp["num_covered"], pol["num_covered"])
    assert set(plain) | {"J_before_improve", "moves", "converged"} == set(imp)


# ---- 7: no GPU needed ------------------------------------------------------------------------------------------------

def test_symbols_declared_and_exported():
    text = open(os.path.join(ROOT, "include", "uavenv_b200.h")).read()
    L = ub.load_library()
    for name in ("uavenv_improve_allocation", "uavenv_improve_workspace_bytes"):
        assert re.search(r"\b%s\s*\(" % name, text), name
        assert hasattr(L, name), name


def test_null_handle_calls():
    L = ub.load_library()
    assert L.uavenv_improve_allocation(None, 0, 1, 1, None, 0, None, None, None, None, None, None, None, None) == \
        ERR["UAVENV_EINVAL"]
    assert L.uavenv_improve_workspace_bytes(None) == 0


def test_lazy_export():
    first, second = ub.improve_allocation, ub.improve_allocation
    assert callable(first) and first is second
    from target_allocation_ppo_transformer_b200 import allocation
    assert first is allocation.improve_allocation


def test_improve_allocation_rejects_bad_arguments():
    scenes = {"uav_x": np.zeros((2, 30))}
    rows = np.full((2, 30), -1, np.int32)
    for kw in ({"scenes": {}, "assigned_target_id": rows}, {"scenes": {"uav_x": np.zeros(7)}, "assigned_target_id": rows},
               {"scenes": scenes, "assigned_target_id": rows[:1]}, {"scenes": scenes, "assigned_target_id": rows * 1.0},
               {"scenes": scenes, "assigned_target_id": rows, "max_moves": -1},
               {"scenes": scenes, "assigned_target_id": rows, "max_envs": 0}):
        with pytest.raises(ValueError):
            ub.improve_allocation(**kw)
    with pytest.raises(RuntimeError):
        ub.improve_allocation(scenes, rows, device="cpu")
