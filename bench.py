#!/usr/bin/env python
"""Benchmark of the rollout hot path: env-steps/s of the fused step kernel (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c5] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one uavenv_step launch over the whole env batch of this GPU with synthetic Bernoulli(1/2)
actions (SURVEY.md §8d).  Prints ONE JSON line (rank 0).  N > 1: launched by torchrun, one rank per GPU,
env batch sharded by global env id, no data-path collective (weak scaling: the per-GPU batch is fixed).

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32 / float64,
rank 0's envs): the step's (obs, reward, done, info), or with --workload c4 the last update's losses and the
parameters it left.  Scenes and actions are seeded, so two builds run with the same arguments can be compared
output for output.

Timing: W (>= 3) warm-up steps, then exactly K timed steps; every timed step is bracketed by CUDA events on
the launching stream and preceded by an L2 flush (a 256 MiB write) outside the bracket; per-rank time = sum
of the K brackets; job time = max over ranks.  `value` has the actions resident in HBM; `e2e` drives the same
step through the host-buffer entry point (uavenv_step_host): actions host->device and reward/done
device->host inside each bracket.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only and is left as the build left it: no __pycache__ either

# BASELINE.json configs.  c3 is the configuration the 1/2/4/8-GPU env-steps/s metric is quoted on and the
# default; c2 (4096 default-size envs, the bit-exact parity config) and c5 (large swarm) are selectable.
WORKLOADS = {
    "c2": dict(name="configs[1]: 4096 envs x (30 UAVs x 10 targets), env step only", envs_per_gpu=4096, N=30, M=10),
    "c3": dict(name="configs[2]: 65536 envs x (64 UAVs x 64 targets), env step only", envs_per_gpu=65536, N=64, M=64),
    "c5": dict(name="configs[4]: 8192 envs/GPU x (256 UAVs x 256 targets), auto-reset", envs_per_gpu=8192, N=256,
               M=256),
}
PPO = dict(name="configs[3]: PPO rollout + update, transformer policy, 16384 envs x (30 UAVs x 10 targets)",
           envs_per_gpu=16384, N=30, M=10, horizon=32)
ACTION_SEED = 1
SCENE_SEED = 42          # configs/config.py:85 SEED
BURN_IN_STEPS = 300      # untimed: de-synchronises the envs' decision pointers (episodes are ~2N steps long)
POOL = 64                # pre-generated action vectors cycled through the timed steps
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 64_000_000  # --dump-outputs: above this, a fixed seeded sample of the envs is written


def step_outputs(step_out, env_id_base):
    """The (obs, reward, done, info) a step returned, on the host as float32 / float64 numpy arrays, one row per env;
    a seeded sample of the envs (sorted, the same on every run) when all of them would exceed DUMP_BYTES."""
    import numpy as np
    obs, reward, done, info = step_out
    host = {"obs": obs, "reward": reward, "done": done}
    host.update(info)
    host = {k: v.cpu().numpy() for k, v in host.items()}
    host = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float32) for k, v in host.items()}
    B = len(host["obs"])
    host["env_id"] = np.arange(env_id_base, env_id_base + B, dtype=np.float64)
    per_env = sum(v.nbytes for v in host.values()) // B
    if B * per_env > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_env, replace=False))
        host = {k: v[keep] for k, v in host.items()}
    return host


def write_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# Algorithmic bytes per env-step of THIS design (DESIGN.md section 4.1 derives each term): io 38 (int64 action 8,
# reward 4, done 1, info 25), header read 144 / write 124, window ring read 224 / write 56, window out 280,
# records of the new pointer pair 128, accept path (p = 1/2 under Bernoulli actions) 0.5 * (32 + 4).
ALGO_BYTES_PER_ENV_STEP = 38 + 144 + 124 + 224 + 56 + 280 + 128 + 0.5 * (32 + 4)


def survey_bytes(M):     # SURVEY.md §8d traffic model (re-sums J over all M targets every step)
    return 665 + 20 * M


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t_begin, self.t_end = None, None

    def mark_begin(self):
        """The timed region starts now: only samples taken from here on (until mark_end) are reported."""
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        lo = (self.t_begin or 0.0) - 0.05
        hi = (self.t_end or time.time()) + 0.15
        inside = [ln for ts, ln in self.lines if lo <= ts <= hi]
        if not inside:                      # a region shorter than the sampling period: the sample nearest to it
            inside = [min(self.lines, key=lambda x: abs(x[0] - lo))[1]] if self.lines else []
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_config(ub, w, reset_episodes=200):
    return ub.Config(NUM_UAVS=w["N"], NUM_TARGETS=w["M"], RESET_EPISODES=reset_episodes)


# The reference's own Python loop (envs/uav_env.py:295 under main_train.py:79's reset schedule, random actions), measured in
# the BUILD container (8 vCPU Xeon, py3.12, numpy 2.3) by oracle/gen_golden.py while it recorded the golden trajectories.
# The Python tree does not exist on the GPU box, so this is a recorded constant, not a live measurement.
PY_REFERENCE_STEPS_PER_SEC_PER_CORE = {"c2": 86.0, "c3": 43.0, "c5": 9.8, "c4": 86.0}
PY_REFERENCE_PROVENANCE = ("unmodified reference UAVEnv.step (envs/uav_env.py:295), 1 core, build container; recorded by "
                           "oracle/gen_golden.py; SURVEY.md section 6 probe: 88-98 / 45 / 13.5")
CPU_BURN_IN_STEPS = 300   # same burn-in as the GPU arm: the envs' decision pointers and episode phases are de-synchronised


def timed_oracle(w, sample, min_seconds, min_steps=0):
    """Steady-state throughput of the reference ALGORITHM (oracle/uavenv_oracle.c, the C port pinned to the Python
    reference) on all host threads: CPU_BURN_IN_STEPS untimed steps, then whole steps until min_seconds AND min_steps
    are reached.  Used by BOTH CPU arms (cpu_baseline and --impl reference) so that their numbers are comparable."""
    from oracle import oracle as orc
    ocfg = orc.make_cfg(NUM_UAVS=w["N"], NUM_TARGETS=w["M"])
    threads = orc.max_threads()
    sample = max(threads * 8, sample)
    batch = orc.OracleBatch(ocfg, sample, seed=SCENE_SEED, reset_episodes=200, threads=threads)
    for s in range(CPU_BURN_IN_STEPS):
        batch.step_random(s, ACTION_SEED)
    t0, s = time.perf_counter(), CPU_BURN_IN_STEPS
    while True:
        batch.step_random(s, ACTION_SEED)
        s += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds and s - CPU_BURN_IN_STEPS >= min_steps:
            break
    n = s - CPU_BURN_IN_STEPS
    batch.close()
    return {"value": sample * n / dt, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "sample": "%d envs x %d steps of the same workload after %d burn-in steps, reference algorithm (C port of "
                      "envs/uav_env.py pinned to the Python reference, OpenMP over envs), %.1f s" % (
                          sample, n, CPU_BURN_IN_STEPS, dt),
            "timed_steps": n, "seconds": dt, "sample_envs": sample}


def cpu_sample_envs(w):
    return 1024 if w["N"] <= 64 else 128


def run_reference(args, w, rank, world):
    """The reference's CPU algorithm (oracle port: the reference itself is Python and cannot travel to the GPU
    box) on all host threads, in the SAME steady-state protocol as cpu_baseline (burn-in, then >= 3 s of whole steps of
    a bounded sample of the workload's envs, however small --steps is)."""
    if rank != 0:
        return
    r = timed_oracle(w, cpu_sample_envs(w), min_seconds=3.0, min_steps=args.steps)
    value = r["value"]
    print(json.dumps({
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / r["timed_steps"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["name"], "num_uavs": w["N"], "num_targets": w["M"], "sample_envs": r["sample_envs"],
                   "timed_steps_actual": r["timed_steps"], "burn_in_steps": CPU_BURN_IN_STEPS,
                   "actions": "Bernoulli(0.5) counter RNG", "reset_schedule": "full reset every 200 episodes",
                   "python_reference_steps_per_sec_per_core": PY_REFERENCE_STEPS_PER_SEC_PER_CORE.get(args.workload),
                   "python_reference_provenance": PY_REFERENCE_PROVENANCE},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def cpu_baseline(w, seconds=12.0):
    r = timed_oracle(w, cpu_sample_envs(w), min_seconds=seconds)
    return {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}


def measure_ppo(rank, local_rank, world, dev, B, T, K, W, with_clocks=True, dump=None):
    """BASELINE.json configs[3]: end-to-end PPO samples/s = transitions collected AND trained on (K_EPOCHS = 5) per
    second.  One iteration = `T` rollout steps (tcgen05 policy forward + fused env step) followed by the PPO update (GAE
    kernel; per minibatch the hand-written bf16 forward + loss + backward, one flat NCCL gradient all-reduce at N > 1,
    fused clip + Adam - replayed as one CUDA graph).  K iterations are timed with ONE CUDA-event bracket, max over ranks.
    The gradient all-reduce (the only collective) is also timed alone, eagerly, with events around 50 calls on the
    same 1.68 MB flat buffer.  Returns the record (rank 0) or None; `dump` (a dict) receives the last iteration's
    losses and the flat parameters its update left."""
    import numpy as np
    import torch
    import uavenv_b200 as ub
    from target_allocation_ppo_transformer_b200 import parallel
    env = ub.UAVEnvBatched(B, device=dev, seed=SCENE_SEED, env_id_base=rank * B)
    agent = ub.PPOAgent(B, T, dev, fused_rollout=True, env_id_base=rank * B, seed=SCENE_SEED,
                        update_precision=os.environ.get("UAVENV_UPDATE_PRECISION", "fused"),
                        graph_update=os.environ.get("UAVENV_GRAPH_UPDATE", "1") != "0")
    obs = env.reset()
    split = [torch.cuda.Event(enable_timing=True) for _ in range(3)]   # rollout | update boundaries of the last iteration

    def iteration():
        nonlocal obs
        split[0].record()
        while not agent.full():
            a = agent.select_action(obs)
            obs, reward, done, _ = env.step(a)
            agent.store_transition(reward, done)
        split[1].record()
        out = agent.update(obs)
        split[2].record()
        return out

    sampler = ClockSampler(local_rank)
    if rank == 0 and with_clocks:
        sampler.start()                 # nvidia-smi takes a moment to come up: started before the warm-up
    for _ in range(W):
        iteration()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    parallel.barrier(); torch.cuda.synchronize(dev)
    sampler.mark_begin()
    e0.record()
    for _ in range(K):
        stats = iteration()
    e1.record()
    torch.cuda.synchronize(dev); parallel.barrier()
    sampler.mark_end()
    if dump is not None:
        dump.update({k: np.float64(v) for k, v in stats.items()})
        dump["policy_params"] = agent._flat_params.cpu().numpy()
    ms = parallel.reduce_scalar(e0.elapsed_time(e1), "max", dev)
    clocks = sampler.stop() if (rank == 0 and with_clocks) else None
    roll_ms = parallel.reduce_scalar(split[0].elapsed_time(split[1]), "max", dev)
    upd_ms = parallel.reduce_scalar(split[1].elapsed_time(split[2]), "max", dev)
    ar_us = parallel.reduce_scalar(agent.time_gradient_allreduce(50), "max", dev)
    n_mb = 5 * (B * T // agent.minibatch_size)
    launches_mb = agent.launches_per_minibatch()
    rec = None
    if rank == 0:
        samples = B * T * world * K
        rec = {
            "metric": "ppo_samples_per_sec", "value": samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 rollout forward (tcgen05) / %s update%s / f64 env" % (
                "bf16 tcgen05 (fp32 accumulation, fp32 gradients)" if agent.update_precision == "fused" else agent.update_precision,
                ", CUDA-graph replay" if agent.graph_update else ""), "data": "synthetic",
            "config": {"workload": PPO["name"], "envs_per_gpu": B, "horizon": T, "k_epochs": 5,
                       "minibatch": agent.minibatch_size, "minibatch_steps_per_iteration": n_mb, "last_stats": stats,
                       "last_iteration_ms": {"rollout": roll_ms, "update": upd_ms},
                       "parallelism": "env-sharded x%d, flat fp32 gradient all-reduce (NCCL) per minibatch" % world},
            "comm": {"collective": "ncclAllReduce(sum) of the flat fp32 gradient, %d B, once per minibatch step" % (
                         4 * agent.num_params),
                     "nranks": world, "allreduce_us_per_minibatch": ar_us if world > 1 else 0.0,
                     "allreduce_share_of_iteration": (ar_us * 1e-3 * n_mb) / (ms / K) if world > 1 else 0.0,
                     "how": "CUDA events around 50 back-to-back all_reduce calls on the same buffer, max over ranks"},
            "e2e": {"value": samples / (ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 24,
                    "note": "the whole loop is device-resident; only the three mean losses leave the GPU per update"},
            # own kernels per iteration: T x (fused policy blocks + heads + env step) + 2 GAE + the minibatch steps
            "gpu_launches": K * (T * 4 + 2 + launches_mb * n_mb),   # per rollout step: env step, two fused forward kernels, heads / sampling
            "clocks": clocks}
    agent.close()       # drop the captured graph before the communicator it references goes away
    env.close()
    return rec


def run_ppo(args):
    """--workload c4: the PPO record as the main JSON line."""
    import torch
    import uavenv_b200  # noqa: F401  (registers the package under its importable name)
    from target_allocation_ppo_transformer_b200 import parallel
    if args.impl == "reference":
        if int(os.environ.get("RANK", 0)) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "the reference's PPO loop is Python/PyTorch code that "
                              "does not exist on the GPU box; in the build container it runs at ~59 samples/s (SURVEY.md 6)"}))
        return
    rank, local_rank, world = parallel.init("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, T = args.envs_per_gpu or PPO["envs_per_gpu"], PPO["horizon"]
    K, W = args.steps, min(args.warmup, 3)
    dump = {} if args.dump_outputs and rank == 0 else None
    rec = measure_ppo(rank, local_rank, world, dev, B, T, K, W, dump=dump)
    if rank == 0:
        print(json.dumps(rec))
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 200); with --workload c4, timed PPO iterations (default 5)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS) + ["c4"],
                    help="c3 (default) / c2 / c5: env-steps/s of the fused step; c4: end-to-end PPO samples/s")
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ppo", action="store_true", help="skip the configs[3] PPO sub-record of the default line")
    ap.add_argument("--ppo-iterations", type=int, default=3, help="timed PPO iterations of the `ppo` sub-record")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic only: keep L2 warm between steps")
    ap.add_argument("--reset-episodes", type=int, default=200, help="diagnostic only: cfg.RESET_EPISODES (200)")
    ap.add_argument("--flush-mode", default="write+read", choices=["write+read", "write", "read", "sleep"],
                    help="diagnostic only: what runs between timed steps (default: the documented L2 flush)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (not with --impl reference)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.workload == "c4" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm runs on the host")
    args.warmup = max(args.warmup, 3)
    if args.workload == "c4":
        return run_ppo(args)
    w = dict(WORKLOADS[args.workload])
    if args.envs_per_gpu:
        w["envs_per_gpu"] = args.envs_per_gpu

    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return

    import numpy as np
    import torch
    import uavenv_b200 as ub
    from target_allocation_ppo_transformer_b200 import parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the env has no CPU fallback")
    rank, local_rank, world = parallel.init("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = w["envs_per_gpu"]
    K, W = args.steps, args.warmup
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                 # nvidia-smi takes a moment to come up: started before the burn-in
    env = ub.UAVEnvBatched(B, device=dev, seed=SCENE_SEED, env_id_base=rank * B, config=make_config(ub, w, args.reset_episodes))
    env.reset(full_reset=True)
    # steady state of the main_train.py:79 schedule: after long training the envs sit at different phases of
    # the 200-episode regeneration cycle; start them staggered so regenerations are amortised into the timing
    gid = np.arange(rank * B, (rank + 1) * B, dtype=np.uint64)
    env.set_episode_counters((1 + (gid * np.uint64(2654435761) >> np.uint64(7)) % np.uint64(200)).astype(np.int32))
    for s in range(BURN_IN_STEPS):
        env.step(env.random_actions(s, ACTION_SEED))
    pool = torch.empty(POOL, B, dtype=torch.int64, device=dev)
    for i in range(POOL):
        env.random_actions(BURN_IN_STEPS + i, ACTION_SEED, out=pool[i])
    pool_host = pool.cpu().pin_memory()                        # int64, the dtype Categorical.sample() yields
    pool_host_i8 = pool.cpu().to(torch.int8).pin_memory()      # one byte per binary action
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    sweep = torch.zeros(L2_FLUSH_BYTES // 8, dtype=torch.int64, device=dev)
    sink = torch.zeros(1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev)

    def flush_l2(i):
        if args.no_flush:
            return
        if args.flush_mode in ("write+read", "write"):
            flush.fill_(i & 0xff)      # L2 flush (256 MiB write), outside the bracket ...
        if args.flush_mode in ("write+read", "read"):
            sink.add_(sweep.sum())     # ... then a 256 MiB read sweep, so the timed kernel starts on a
                                       # cold but CLEAN L2 and does not pay write-backs of the flush data
        if args.flush_mode == "sleep":
            torch.cuda._sleep(60000)   # diagnostic: GPU-side delay only (L2 stays warm, host runs ahead)

    def timed(step_fn, n_warm, n_timed):
        for i in range(n_warm):        # warm-up = the timed loop's exact sequence (flush, then step), untimed: the first
            flush_l2(i)                # call of the flush ops allocates, which would otherwise stall the host inside the
            step_fn(i)                 # first timed bracket and show up there as a ~100 us launch gap
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_timed)]
        parallel.barrier()
        torch.cuda.synchronize(dev)
        # lead-in: ~0.25 ms of untimed flush work queued ahead of the first bracket, so that the host (which comes out of
        # the barrier late under torchrun) is enqueueing ahead of the GPU when bracket 0 opens - a bracket only measures
        # the kernel if its launch is already waiting in the stream (without this, bracket 0 read 40-120 us at N > 1)
        # (two untimed steps ride along: at N > 1 the first step after the barrier's NCCL kernel read ~30 us against 18.5 for
        # every later one - one cold bracket in 20 is 0.6 us on the mean)
        for j in range(2):
            flush_l2(j)
            step_fn(n_warm + j)
        for i in range(n_timed):
            flush_l2(i)
            ev[i][0].record(stream)
            out = step_fn(n_warm + i)
            ev[i][1].record(stream)
        timed.last_out = out
        torch.cuda.synchronize(dev)
        parallel.barrier()
        raw = [a.elapsed_time(b) for a, b in ev]
        if os.environ.get("UAVENV_BENCH_DUMP") and rank == 0:       # diagnostic: every bracket of this rank, in order
            print("brackets_us " + " ".join("%.1f" % (1e3 * x) for x in raw), file=sys.stderr)
        per = sorted(raw)
        timed.last_us = {"min": 1e3 * per[0], "median": 1e3 * per[len(per) // 2], "p90": 1e3 * per[(9 * len(per)) // 10],
                         "max": 1e3 * per[-1], "max_at_step": raw.index(per[-1])}   # this rank's brackets (diagnostic)
        return parallel.reduce_scalar(sum(per), "max", dev)

    graph_us = None
    if os.environ.get("UAVENV_BENCH_GRAPH"):
        # diagnostic: POOL steps captured in one CUDA graph and replayed back to back (no host gaps, warm L2)
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for i in range(3):
                env.step(pool[i])
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for i in range(POOL):
                    env.step(pool[i])
            for _ in range(3):
                g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(5):
                g.replay()
            e1.record(side)
        torch.cuda.synchronize(dev)
        graph_us = 1e3 * e0.elapsed_time(e1) / (5 * POOL)
        print("graph replay: %.2f us/step" % graph_us, file=sys.stderr)

    # --- device-resident inputs: the fused kernel alone --------------------------------------------------
    sampler.mark_begin()
    ms_dev = timed(lambda i: env.step(pool[i % POOL]), W, K)
    step_us = dict(timed.last_us)
    # the env's output buffers still hold the last timed step: copied before anything steps the env again
    dump = step_outputs(timed.last_out, rank * B) if args.dump_outputs and rank == 0 else None
    # the same bracket around a ~2 us kernel (the action generator): what the protocol itself costs per step
    ms_floor = timed(lambda i: env.random_actions(i, ACTION_SEED), 3, min(K, 50)) / min(K, 50)
    # --- end to end through the host-buffer entry point ----------------------------------------------------
    ms_e2e = timed(lambda i: env.step_host(pool_host_i8[i % POOL]), W, K)
    ms_e2e_i64 = timed(lambda i: env.step_host(pool_host[i % POOL]), W, K)
    # ... and with step()'s full 4-tuple crossing the boundary: the [B,5,14] window is copied to pinned host memory too
    obs_host = torch.empty(B, 5, 14, dtype=torch.float32).pin_memory()
    ms_e2e_obs = timed(lambda i: env.step_host(pool_host_i8[i % POOL], obs_out=obs_host), W, K)
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    drift = env.recompute_objective()
    drift = parallel.reduce_scalar(drift, "max", dev)

    if rank == 0:
        total_envs = B * world
        value = total_envs * K / (ms_dev * 1e-3)
        e2e_value = total_envs * K / (ms_e2e * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        per_launch_s = ms_dev * 1e-3 / K
        achieved = ALGO_BYTES_PER_ENV_STEP * B / per_launch_s / 1e9
        surv = survey_bytes(w["M"]) * B / per_launch_s / 1e9
        traffic = traffic_src = None     # DRAM bytes per launch from the committed ncu capture of this command (ncu cannot run
        try:                              # inside a timed run); null for workloads without a capture
            rec = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")))[args.workload]
            traffic, traffic_src = rec["per_launch_total"], rec["source"]
        except Exception:
            pass
        out = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["name"], "envs_per_gpu": B, "num_uavs": w["N"], "num_targets": w["M"],
                       "actions": "Bernoulli(0.5), counter RNG keyed (seed=1, step, global env id), resident in HBM",
                       "auto_reset": True, "reset_schedule": "full reset every %d episodes, staggered steady state" % args.reset_episodes,
                       "burn_in_steps": BURN_IN_STEPS, "l2": "flushed between timed steps (256 MiB write, then a 256 MiB read sweep leaving clean lines)"
                       if not args.no_flush else "NOT flushed (diagnostic)",
                       "timing": "CUDA events per step on the launching stream, summed; max over ranks",
                       "pair_evals_per_sec": value, "objective_drift_max_abs": drift,
                       "bracket_floor_us": 1e3 * ms_floor, "step_bracket_us_rank0": step_us,
                       "parallelism": "env-sharded x%d, no rollout collective" % world},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "uavk::step_kernel",
                         "bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650",
                         "survey_model": {"bytes_per_env_step": survey_bytes(w["M"]), "achieved": surv,
                                          "frac": surv / peak,
                                          "note": "SURVEY §8d counts a 20*M B re-read of all target products per "
                                                  "step; this kernel carries the objective incrementally and does "
                                                  "not move those bytes"}},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": B * 1, "d2h_bytes_per_step": B * 5,
                    "api": "UAVEnvBatched.step_host -> uavenv_step_host_i8 (pinned host int8 actions in; f32 reward + u8 "
                           "done out, in place over PCIe; observation window stays in HBM for the policy)",
                    "int64_actions": {"value": total_envs * K / (ms_e2e_i64 * 1e-3), "ms_per_step": ms_e2e_i64 / K,
                                      "h2d_bytes_per_step": B * 8},
                    # the reference's step() returns (obs, reward, done, info) (envs/uav_env.py:435): the same call with
                    # the observation window ALSO copied to pinned host memory inside the bracket
                    "with_obs": {"value": total_envs * K / (ms_e2e_obs * 1e-3), "ms_per_step": ms_e2e_obs / K,
                                 "h2d_bytes_per_step": B * 1, "d2h_bytes_per_step": B * (5 + 280),
                                 "pcie_d2h_gbs": B * 285 / (ms_e2e_obs / K * 1e-3) / 1e9,
                                 "api": "UAVEnvBatched.step_host(actions, obs_out=pinned [B,5,14])"}},
            "gpu_launches": K, "clocks": clocks,
        }
        out["config"]["python_reference_steps_per_sec_per_core"] = PY_REFERENCE_STEPS_PER_SEC_PER_CORE.get(args.workload)
        out["config"]["python_reference_provenance"] = PY_REFERENCE_PROVENANCE
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(w)
    env.close()
    del env, pool, flush, sweep
    torch.cuda.empty_cache()
    if not args.no_ppo:
        # second half of the BASELINE metric ("end-to-end PPO samples/sec", configs[3]) on the same N GPUs: rollout +
        # update with the NCCL gradient all-reduce, so the driver's 1/2/4/8 runs carry its scaling curve too
        ppo = measure_ppo(rank, local_rank, world, dev, PPO["envs_per_gpu"], PPO["horizon"], max(1, args.ppo_iterations), 2,
                          with_clocks=False)
        if rank == 0:
            out["ppo"] = {k: ppo[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "dtype",
                                              "config", "comm", "gpu_launches")}
    if rank == 0:
        print(json.dumps(out))
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
