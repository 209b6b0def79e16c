#!/usr/bin/env python
"""Timing of the evaluation path (one JSON object per line, also written to --out):
  - the actor-only greedy forward `act` against `get_action`, CUDA-graph replay, the two alternated within the run;
  - uavenv_episode_accumulate per step at 65536 envs (CUDA events around each launch of a real evaluation loop);
  - ub.evaluate at 16384 envs on the default 30x10 config and on 64x64: episodes/s and env-steps/s.
The first line records the card and its power limit.
    python profiles/measure_eval.py [--out profiles/r3_eval.jsonl]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import uavenv_b200 as ub  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"what": "card", "torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def graph_of(fn):
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    return g


def time_graph(g, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters          # us per call


def forward_rows(net, sizes, rounds=15, iters=50):
    rows = []
    for B in sizes:
        obs = torch.rand(B, 5, 14, device="cuda")
        obs[::4, :2] = 0.0
        fused = ub.FusedPolicyForward(B, "cuda")
        fused.sync(net)
        g_full = graph_of(lambda: fused.get_action(obs, 7))
        g_act = graph_of(lambda: fused.act(obs, 7, greedy=True))
        for g in (g_full, g_act):
            time_graph(g, 20)
        full, act = [], []
        for _ in range(rounds):                         # alternated: drifts in clock or load hit both alike
            full.append(time_graph(g_full, iters))
            act.append(time_graph(g_act, iters))
        f, a = statistics.median(full), statistics.median(act)
        rows.append({"what": "forward_graph_replay", "B": B, "get_action_us": f, "act_greedy_us": a, "act_over_get_action": a / f,
                     "get_action_us_minmax": [min(full), max(full)], "act_greedy_us_minmax": [min(act), max(act)],
                     "rounds": rounds, "calls_per_round": iters})
        fused.close()
    return rows


def accumulate_row(net, B=65536, steps=300):
    cfg = ub.cfg.copy(RESET_EPISODES=1)
    env = ub.UAVEnvBatched(B, seed=5, config=cfg)
    rec = ub.EpisodeRecorder(env, 32)
    fused = ub.FusedPolicyForward(B, "cuda", seed=5)
    fused.sync(net)
    obs = env.reset(full_reset=True)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True),
           torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):
        a, _ = fused.act(obs, s, greedy=False)
        ev[s][0].record()
        obs, _, _, _ = env.step(a)
        ev[s][1].record()
        rec.record(a)
        ev[s][2].record()
    torch.cuda.synchronize()
    warm = 20
    step_us = [e0.elapsed_time(e1) * 1e3 for e0, e1, _ in ev[warm:]]
    acc_us = [e1.elapsed_time(e2) * 1e3 for _, e1, e2 in ev[warm:]]
    episodes = int((rec.records()["length"] > 0).sum())
    fused.close(); env.close()
    return {"what": "episode_accumulate", "B": B, "steps_timed": steps - warm, "accumulate_us_median": statistics.median(acc_us),
            "accumulate_us_mean": statistics.mean(acc_us), "env_step_us_median": statistics.median(step_us),
            "episodes_recorded": episodes, "config": "30x10"}


def evaluate_rows(net, B=16384):
    rows = []
    for name, cfg, quota in (("30x10", ub.cfg.copy(), 4), ("64x64", ub.Config(NUM_UAVS=64, NUM_TARGETS=64), 1)):
        ub.evaluate(net, num_envs=B, episodes_per_env=1, config=cfg)          # warm-up: module loads, first allocations
        for greedy in (True, False):
            s = ub.evaluate(net, num_envs=B, episodes_per_env=quota, greedy=greedy, config=cfg)["summary"]
            rows.append({"what": "evaluate", "config": name, "num_envs": B, "episodes_per_env": quota, "greedy": greedy,
                         "episodes_per_s": s["episodes_per_s"], "env_steps_per_s": s["env_steps_per_s"], "wall_s": s["wall_s"],
                         "env_steps": s["env_steps"], "length_mean": s["length_mean"], "J_mean": s["J_mean"]})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_eval.jsonl"))
    ap.add_argument("--sizes", type=int, nargs="*", default=[4096, 16384, 65536])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("measure_eval.py times the GPU path and needs a CUDA device")
    torch.manual_seed(0)
    net = ub.TransformerActorCritic().cuda().eval()     # untrained weights, seeded: the timings do not depend on them
    rows = [card()] + forward_rows(net, args.sizes) + [accumulate_row(net)] + evaluate_rows(net)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
