#!/usr/bin/env python
"""Cost and tightness of the certified upper bound (one JSON object per line, also written to --out):
  - bound_kernel on 4096 scenes at 30x10, 64x64 (a in shared memory) and 256x256 (a in the workspace) for iters = 64,
    256 and 1024: CUDA events around the C call uavenv_upper_bound, median of repeated calls (every call does the same
    work: the kernel reads only the scenes), with the iterations actually run and the mean bound / relaxed value;
  - improve_kernel on the same scenes from the best of 16 sampled episodes, timed the same way, for comparison;
  - the gap bound - J of the project's allocations on the same scenes (the first --gap-scenes of them): the best of 16
    sampled episodes of seeded untrained weights, and the best-target heuristic, each polished by the local search.
The first line records the card and its power limit.
    python profiles/measure_bound.py [--out profiles/r3_bound.jsonl] [--configs 30x10,64x64,256x256]"""
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
from measure_improve import CONFIGS, K, S, net_of, scenes_of  # noqa: E402
import uavenv_b200 as ub  # noqa: E402

ITERS = (64, 256, 1024)
GAP_SCENES = {"30x10": 4096, "64x64": 4096, "256x256": 512}


def events(fn, repeats):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeats)]
    for e0, e1 in ev:
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    return {"calls": repeats, "ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms),
            "scenes_per_s": S / (statistics.median(ms) * 1e-3)}


def bound_row(name, env, iters, repeats):
    out = env.upper_bound(iters=iters)                                   # warm-up; allocates outputs and workspace
    torch.cuda.synchronize()
    L, ws = env._lib, env._improve_workspace
    ptrs = [C.c_void_p(out[k].data_ptr()) for k in ("bound", "relaxed", "iters")]
    wsp = C.c_void_p(ws.data_ptr() if ws is not None else None)
    t = events(lambda: L.uavenv_upper_bound(env._h, 0, S, 1, iters, *ptrs, wsp, None) == 0 or sys.exit("call failed"),
               repeats)
    r = {k: v.cpu().numpy() for k, v in out.items()}
    row = {"what": "bound_kernel", "config": name, "scenes": S, "iters": iters,
           "a_in": "workspace" if L.uavenv_improve_workspace_bytes(env._h) else "shared"}
    row.update(t)
    row.update({"iters_run_mean": float(r["iters"].mean()), "iters_run_max": int(r["iters"].max()),
                "stopped_early_share": float((r["iters"] < iters).mean()), "bound_mean": float(r["bound"].mean()),
                "relaxed_mean": float(r["relaxed"].mean()),
                "bound_minus_relaxed_rel_mean": float(((r["bound"] - r["relaxed"]) / np.abs(r["bound"])).mean())})
    return row, r["bound"]


def improve_row(name, env, rows, repeats):
    a = torch.as_tensor(rows).cuda().to(torch.int32).contiguous()
    out = env.improve_allocation(a)
    torch.cuda.synchronize()
    L, N, ws = env._lib, env.N, env._improve_workspace
    ptrs = [C.c_void_p(out[k].data_ptr()) for k in ("assigned_target_id", "J_before", "J", "num_covered", "moves",
                                                     "converged")]
    wsp = C.c_void_p(ws.data_ptr() if ws is not None else None)
    t = events(lambda: L.uavenv_improve_allocation(env._h, 0, S, 1, C.c_void_p(a.data_ptr()), 16 * N, *ptrs, wsp,
                                                   None) == 0 or sys.exit("call failed"), repeats)
    row = {"what": "improve_kernel", "config": name, "scenes": S, "input": "sampled_best_of_16"}
    row.update(t)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bound.jsonl"))
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("measure_bound.py times the GPU path and needs a CUDA device")
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
            env = ub.UAVEnvBatched(S, seed=0, config=cfg, auto_reset=False, with_info=False)
            env.load_scene_device(dev_scenes)
            bounds = {}
            for iters in ITERS:
                row, bounds[iters] = bound_row(name, env, iters, 20)
                emit(row)
            rows = ub.allocate(net, scenes=dev_scenes, samples=K, config=cfg)["assigned_target_id"]
            emit(improve_row(name, env, rows, 20))
            env.close()
            G = GAP_SCENES[name]
            sub = {k: v[:G] for k, v in dev_scenes.items()}
            allocs = {"sampled_best_of_16_improve": ub.allocate(net, scenes=sub, samples=K, config=cfg, improve=True),
                      "best_target_improve": ub.allocate("best_target", scenes=sub, config=cfg, improve=True)}
            for label, res in allocs.items():
                J = res["J"]
                for iters in ITERS:
                    b = bounds[iters][:G]
                    rel = (b - J) / np.abs(J)
                    emit({"what": "gap", "config": name, "allocation": label, "scenes": G, "iters": iters,
                          "J_mean": float(J.mean()), "bound_mean": float(b.mean()), "gap_mean": float((b - J).mean()),
                          "gap_rel_mean": float(rel.mean()), "gap_rel_median": float(np.median(rel)),
                          "gap_rel_max": float(rel.max()), "bound_below_J": int((b < J).sum())})


if __name__ == "__main__":
    main()
