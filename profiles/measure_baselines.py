#!/usr/bin/env python
"""Timing of the evaluation baselines (one JSON object per line, also written to --out):
  - uavenv_best_target_actions per call inside an evaluation loop (best-target actions -> env step -> episode
    accumulate), CUDA events around each launch, median over the steps after a warm-up - the method measure_eval.py uses
    for the accumulate kernel;
  - ub.evaluate_baseline ("best_target" and "random"): episodes/s and env-steps/s, one episode per env;
at B in {4096, 16384, 65536} on the 30x10, 64x64 and 256x256 configs.  The first line records the card and its power limit.
    python profiles/measure_baselines.py [--out profiles/r3_baselines.jsonl]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from measure_eval import ROOT, card  # noqa: E402
import uavenv_b200 as ub  # noqa: E402

CONFIGS = (("30x10", 30, 10), ("64x64", 64, 64), ("256x256", 256, 256))


def kernel_row(name, cfg, B, steps=300, warm=20):
    env = ub.UAVEnvBatched(B, seed=5, config=cfg)
    rec = ub.EpisodeRecorder(env, 4)
    env.reset(full_reset=True)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for s in range(steps):
        ev[s][0].record()
        a = env.best_target_actions()
        ev[s][1].record()
        env.step(a)
        ev[s][2].record()
        rec.record(a)
    torch.cuda.synchronize()
    kern = [e0.elapsed_time(e1) * 1e3 for e0, e1, _ in ev[warm:]]
    step = [e1.elapsed_time(e2) * 1e3 for _, e1, e2 in ev[warm:]]
    env.close()
    return {"what": "best_target_kernel", "config": name, "B": B, "steps_timed": steps - warm,
            "best_target_us_median": statistics.median(kern), "best_target_us_mean": statistics.mean(kern),
            "best_target_us_first_call": ev[0][0].elapsed_time(ev[0][1]) * 1e3, "env_step_us_median": statistics.median(step)}


def evaluate_row(name, cfg, B, kind):
    res = ub.evaluate_baseline(kind, num_envs=B, episodes_per_env=1, config=cfg)
    s = res["summary"]
    return {"what": "evaluate_baseline", "kind": kind, "config": name, "num_envs": B, "episodes_per_env": 1,
            "episodes_per_s": s["episodes_per_s"], "env_steps_per_s": s["env_steps_per_s"], "wall_s": s["wall_s"],
            "env_steps": s["env_steps"], "length_mean": s["length_mean"], "J_mean": s["J_mean"], "J_sem": s["J_sem"],
            "coverage_mean": s["coverage_mean"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_baselines.jsonl"))
    ap.add_argument("--sizes", type=int, nargs="*", default=[4096, 16384, 65536])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("measure_baselines.py times the GPU path and needs a CUDA device")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        def emit(row):
            line = json.dumps(row)
            print(line, flush=True)
            f.write(line + "\n")

        emit(card())
        for kind in ("best_target", "random"):       # warm-up: module loads, first allocations
            ub.evaluate_baseline(kind, num_envs=4096)
        for name, n, m in CONFIGS:
            cfg = ub.Config(NUM_UAVS=n, NUM_TARGETS=m, RESET_EPISODES=1)
            for B in args.sizes:
                emit(kernel_row(name, cfg, B))
                for kind in ("best_target", "random"):
                    emit(evaluate_row(name, cfg, B, kind))


if __name__ == "__main__":
    main()
