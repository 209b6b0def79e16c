#!/usr/bin/env python
"""Timing and effect of the allocation local search (one JSON object per line, also written to --out):
  - improve_kernel on 4096 scenes at 30x10, 64x64 (p in shared memory) and 256x256 (p in the workspace): CUDA events
    around the C call uavenv_improve_allocation, median of repeated calls on the same input (the kernel reads its input
    rows and writes separate outputs, so every call does the same work), for three inputs per config: the best of 16
    sampled episodes of seeded untrained weights (ub.allocate), the best-target heuristic's allocation (ub.allocate
    "best_target") and uniformly random allocations; with the moves per scene, the converged share and J before / after;
  - ub.allocate(improve=True) against ub.allocate(improve=False) end to end (K = 16, 4096 scenes, median of 3 calls).
The first line records the card and its power limit.
    python profiles/measure_improve.py [--out profiles/r3_improve.jsonl] [--configs 30x10,64x64,256x256]"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from measure_eval import ROOT, card  # noqa: E402
import uavenv_b200 as ub  # noqa: E402

CONFIGS = {"30x10": (30, 10), "64x64": (64, 64), "256x256": (256, 256)}
S = 4096
K = 16


def scenes_of(cfg, seed=11):
    env = ub.UAVEnvBatched(S, seed=seed, config=cfg, auto_reset=False, with_info=False)
    env.reset(full_reset=True)
    sc = env.get_scene()
    env.close()
    return sc


def net_of():
    torch.manual_seed(0)
    return ub.TransformerActorCritic()


def random_rows(scenes, seed=3):
    rng = np.random.default_rng(seed)
    ids = scenes["tgt_id"]
    pos = rng.integers(-1, ids.shape[1], size=scenes["uav_x"].shape)
    return np.where(pos >= 0, np.take_along_axis(ids, np.maximum(pos, 0), axis=1), -1).astype(np.int32)


def kernel_row(name, cfg, env, label, rows, repeats):
    """CUDA events around the C call on the same input; the result of the last call summarised."""
    a = torch.as_tensor(rows).cuda().to(torch.int32).contiguous()
    out = env.improve_allocation(a)                                       # warm-up; allocates outputs and workspace
    torch.cuda.synchronize()
    L, N = env._lib, env.N
    ptrs = [C.c_void_p(out[k].data_ptr()) for k in ("assigned_target_id", "J_before", "J", "num_covered", "moves",
                                                     "converged")]
    ws = env._improve_workspace
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeats)]
    for e0, e1 in ev:
        e0.record()
        assert L.uavenv_improve_allocation(env._h, 0, S, 1, C.c_void_p(a.data_ptr()), 16 * N, *ptrs,
                                           C.c_void_p(ws.data_ptr() if ws is not None else None), None) == 0
        e1.record()
    torch.cuda.synchronize()
    ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    r = {k: v.cpu().numpy() for k, v in out.items()}
    return {"what": "improve_kernel", "config": name, "input": label, "scenes": S,
            "p_in": "workspace" if env._lib.uavenv_improve_workspace_bytes(env._h) else "shared",
            "calls": repeats, "ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms),
            "scenes_per_s": S / (statistics.median(ms) * 1e-3),
            "moves_mean": float(r["moves"].mean()), "moves_max": int(r["moves"].max()),
            "converged_share": float(r["converged"].mean()),
            "J_before_mean": float(r["J_before"].mean()), "J_after_mean": float(r["J"].mean()),
            "J_gain_mean": float((r["J"] - r["J_before"]).mean()),
            "J_gain_rel_mean": float(((r["J"] - r["J_before"]) / np.maximum(np.abs(r["J_before"]), 1e-12)).mean())}


def allocate_rows(name, cfg, dev_scenes, net):
    rows = []
    for improve in (False, True):
        ub.allocate(net, scenes=dev_scenes, samples=K, config=cfg, improve=improve)      # warm-up of this shape
        runs = [ub.allocate(net, scenes=dev_scenes, samples=K, config=cfg, improve=improve) for _ in range(3)]
        res = sorted(runs, key=lambda r: r["summary"]["wall_s"])[1]
        s = res["summary"]
        row = {"what": "allocate", "config": name, "samples": K, "scenes": S, "improve": improve,
               "wall_s_median": s["wall_s"], "wall_s_all": [r["summary"]["wall_s"] for r in runs],
               "scenes_per_s": s["scenes_per_s"], "J_mean": s["J_mean"]}
        if improve:
            row["J_before_improve_mean"] = s["J_before_improve_mean"]
            row["moves_mean"] = s["moves_mean"]
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_improve.jsonl"))
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("measure_improve.py times the GPU path and needs a CUDA device")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        def emit(row):
            line = json.dumps(row)
            print(line, flush=True)
            f.write(line + "\n")

        emit(card())
        net = net_of()
        for name in args.configs.split(","):
            n, m = CONFIGS[name]
            cfg = ub.Config(NUM_UAVS=n, NUM_TARGETS=m)
            host = scenes_of(cfg)
            dev_scenes = {k: torch.as_tensor(v).cuda() for k, v in host.items()}
            inputs = {"sampled_best_of_16": ub.allocate(net, scenes=dev_scenes, samples=K, config=cfg)["assigned_target_id"],
                      "best_target": ub.allocate("best_target", scenes=dev_scenes, config=cfg)["assigned_target_id"],
                      "random": random_rows(host)}
            env = ub.UAVEnvBatched(S, seed=0, config=cfg, auto_reset=False, with_info=False)
            env.load_scene_device(dev_scenes)
            for label, rows in inputs.items():
                emit(kernel_row(name, cfg, env, label, rows, 5 if n >= 256 else 20))
            env.close()
            if n < 256:
                for row in allocate_rows(name, cfg, dev_scenes, net):
                    emit(row)


if __name__ == "__main__":
    main()
