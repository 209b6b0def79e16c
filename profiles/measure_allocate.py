#!/usr/bin/env python
"""Timing of best-of-K allocation (one JSON object per line, also written to --out):
  - ub.allocate: scenes/s and env-steps/s on the 30x10 and 64x64 configs with K in {1, 16, 128} samples per scene at
    S*K = 65536 envs, seeded untrained weights (sampled; greedy at K = 1), the scenes given as device tensors, the
    median of 5 calls after one warm-up call of the same shape;
  - uavenv_load_scene_device (65536 scenes, and 4096 scenes x 16 copies) against the host uavenv_load_scene of 65536
    scenes: CUDA events around the device load (median of 20), a host clock around the synchronous host load (median of 5);
  - group_best_kernel over 65536 finished envs in groups of K: CUDA events around the C call, median of 200 calls;
  - the share of forward rows spent on already-finished envs in allocate's loop (a separate, untimed pass that reads
    `done` after every step), the data for compacting finished envs out of the forward batch.
The first line records the card and its power limit.
    python profiles/measure_allocate.py [--out profiles/r3_allocate.jsonl]"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from measure_eval import ROOT, card  # noqa: E402
import uavenv_b200 as ub  # noqa: E402

CONFIGS = (("30x10", 30, 10), ("64x64", 64, 64))
TOTAL = 65536
SAMPLES = (1, 16, 128)
REPEATS = 5


def scenes_of(cfg, S, seed=11):
    env = ub.UAVEnvBatched(S, seed=seed, config=cfg, auto_reset=False, with_info=False)
    env.reset(full_reset=True)
    sc = env.get_scene()
    env.close()
    return sc


def net_of():
    torch.manual_seed(0)
    return ub.TransformerActorCritic()


def allocate_row(name, cfg, K, dev_scenes, net):
    S = TOTAL // K
    sc = {k: v[:S] for k, v in dev_scenes.items()}
    ub.allocate(net, scenes=sc, samples=K, config=cfg)                    # warm-up of this shape
    runs = [ub.allocate(net, scenes=sc, samples=K, config=cfg)["summary"] for _ in range(REPEATS)]
    s = sorted(runs, key=lambda r: r["wall_s"])[REPEATS // 2]            # the median call
    return {"what": "allocate", "config": name, "samples": K, "scenes": S, "envs": S * K, "greedy": K == 1,
            "calls": REPEATS, "scenes_per_s": s["scenes_per_s"], "env_steps_per_s": s["env_steps_per_s"],
            "wall_s_median": s["wall_s"], "wall_s_all": [r["wall_s"] for r in runs], "env_steps": s["env_steps"],
            "J_mean": s["J_mean"], "J_samples_mean": s["J_samples_mean"]}


def finished_share_row(name, cfg, K, dev_scenes, net):
    """allocate's loop once more, untimed, counting the finished rows the forward processes at every step."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    S = TOTAL // K
    env = ub.UAVEnvBatched(S * K, seed=1, config=cfg, auto_reset=False)
    fused = FusedPolicyForward(S * K, env.device, seed=1)
    fused.sync(net.cuda())
    env.load_scene_device({k: v[:S] for k, v in dev_scenes.items()}, copies=K)
    finished_rows, steps = 0, 0
    while steps < env.N * env.M:
        finished_rows += int(env.done.sum()) if steps else 0             # rows already done when this step's forward ran
        env.step(fused.act(env.obs, steps, greedy=K == 1)[0])
        steps += 1
        if bool(env.done.all()):
            break
    fused.close()
    env.close()
    return {"what": "allocate_finished_rows", "config": name, "samples": K, "envs": S * K, "steps": steps,
            "finished_row_share": finished_rows / float(steps * S * K)}


def load_rows(name, cfg, host_scenes, dev_scenes):
    env = ub.UAVEnvBatched(TOTAL, seed=1, config=cfg, auto_reset=False, with_info=False)
    rows = []
    host = []
    for i in range(6):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        env.load_scene(host_scenes)                                       # synchronous
        host.append((time.perf_counter() - t0) * 1e3)
    rows.append({"what": "load_scene_host", "config": name, "scenes": TOTAL, "copies": 1,
                 "ms_median": statistics.median(host[1:])})
    for S, K in ((TOTAL, 1), (TOTAL // 16, 16)):
        sc = {k: v[:S] for k, v in dev_scenes.items()}
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(21)]
        for e0, e1 in ev:
            e0.record()
            env.load_scene_device(sc, copies=K)
            e1.record()
        torch.cuda.synchronize()
        ms = [e0.elapsed_time(e1) for e0, e1 in ev[1:]]
        rows.append({"what": "load_scene_device", "config": name, "scenes": S, "copies": K,
                     "ms_median": statistics.median(ms)})
    # a finished episode in every env, then group_best over all of them
    for step in range(env.N * env.M):
        env.step(env.random_actions(step))
        if step % 32 == 31 and bool(env.done.all()):
            break
    L = ub.load_library()
    for K in SAMPLES:
        out = env.group_best(K)                                           # outputs allocated once, then the C call
        ptrs = [C.c_void_p(out[k].data_ptr()) for k in ("best", "J", "assigned_target_id", "num_covered", "J_all")]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(200)]
        for e0, e1 in ev:
            e0.record()
            assert L.uavenv_group_best(env._h, 0, TOTAL // K, K, *ptrs, None) == 0
            e1.record()
        torch.cuda.synchronize()
        us = [e0.elapsed_time(e1) * 1e3 for e0, e1 in ev]
        rows.append({"what": "group_best_kernel", "config": name, "envs": TOTAL, "group_size": K,
                     "us_median": statistics.median(us), "us_mean": statistics.mean(us)})
    env.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_allocate.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("measure_allocate.py times the GPU path and needs a CUDA device")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        def emit(row):
            line = json.dumps(row)
            print(line, flush=True)
            f.write(line + "\n")

        emit(card())
        net = net_of()
        for name, n, m in CONFIGS:
            cfg = ub.Config(NUM_UAVS=n, NUM_TARGETS=m)
            host_scenes = scenes_of(cfg, TOTAL)
            dev_scenes = {k: torch.as_tensor(v).cuda() for k, v in host_scenes.items()}
            for row in load_rows(name, cfg, host_scenes, dev_scenes):
                emit(row)
            for K in SAMPLES:
                emit(allocate_row(name, cfg, K, dev_scenes, net))
            for K in SAMPLES:
                emit(finished_share_row(name, cfg, K, dev_scenes, net))


if __name__ == "__main__":
    main()
