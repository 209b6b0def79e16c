#!/usr/bin/env python
"""Timing of the rollout forward of the policy: tcgen05 path (csrc/policy_forward.cu) vs the fp32 PyTorch mirror
(library kernels: cuBLAS / ATen) on the same weights and observations.  One JSON object per line.
    python profiles/measure_policy.py [B ...]"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import uavenv_b200 as ub  # noqa: E402

FLOP_FULL = 4.04e6       # SURVEY.md 3.6: all five tokens through every layer
FLOP_LAST = 2.0 * (2 * 5 * 14 * 128 + 3 * (5 * 128 * 256 + 128 * 128 * 2 + 2 * 128 * 256) + 5 * (128 * 384 + 128 * 128 + 2 * 128 * 256)
                   - 5 * 128 * 256 + 2 * 128 * 64 + 3 * 64)   # last-token formulation actually executed


def timeit(fn, warm=3, iters=20):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    sizes = [int(x) for x in sys.argv[1:]] or [4096, 16384, 65536]
    net = ub.TransformerActorCritic().cuda().eval()
    for B in sizes:
        obs = torch.rand(B, 5, 14, device="cuda")
        fused = ub.FusedPolicyForward(B, "cuda")
        fused.sync(net)
        step = [0]

        def run_fused():
            step[0] += 1
            fused.get_action(obs, step[0])

        def run_torch():
            with torch.no_grad():
                net.get_action(obs)

        ms_f = timeit(run_fused)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run_fused()
            with torch.cuda.graph(g, stream=side):
                fused.get_action(obs, 7)
        torch.cuda.current_stream().wait_stream(side)
        ms_g = timeit(g.replay)
        torch.backends.cuda.matmul.allow_tf32 = False
        ms_t = timeit(run_torch, 2, 5)
        torch.backends.cuda.matmul.allow_tf32 = True
        ms_t32 = timeit(run_torch, 2, 5)
        print(json.dumps({"B": B, "fused_ms": ms_f, "fused_graph_ms": ms_g, "torch_fp32_ms": ms_t, "torch_tf32_ms": ms_t32,
                          "fused_samples_per_sec": B / (ms_g * 1e-3), "torch_samples_per_sec": B / (ms_t32 * 1e-3),
                          "fused_TFLOPs_executed": B * FLOP_LAST / (ms_g * 1e-3) / 1e12,
                          "speedup_vs_torch_tf32": ms_t32 / ms_g}))
        fused.close()


if __name__ == "__main__":
    main()
