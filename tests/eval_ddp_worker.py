"""Worker of tests/test_gpu_evaluate.py (one process per GPU, NCCL): ub.evaluate under a two-rank process group must
return, on every rank, the records of a single-GPU evaluation over both ranks' envs.

    RANK=r LOCAL_RANK=r WORLD_SIZE=2 MASTER_ADDR=127.0.0.1 MASTER_PORT=... python tests/eval_ddp_worker.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import uavenv_b200 as ub
from helpers import policy_fixture
from target_allocation_ppo_transformer_b200 import parallel

KEYS = ("return", "J", "num_assigned", "length", "assigns", "valid", "avg_p_dmg", "avg_p_final")


def main():
    rank, local_rank, world = parallel.init("nccl")
    torch.cuda.set_device(local_rank)
    _, sd = policy_fixture()
    net = ub.TransformerActorCritic()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    B, quota, modes = 512, 2, (True, False)
    gathered = {g: ub.evaluate(net, num_envs=B, episodes_per_env=quota, greedy=g, seed=31) for g in modes}
    dist.destroy_process_group()
    ok = True
    for g in modes:
        # the same global envs [0, world * B) on this GPU alone, outside the process group
        ref = ub.evaluate(net, num_envs=B * world, episodes_per_env=quota, greedy=g, seed=31, env_id_base=0)
        same = gathered[g]["return"].shape == (B * world, quota) and all(np.array_equal(gathered[g][k], ref[k]) for k in KEYS)
        print("rank %d greedy=%s identical to one GPU: %s" % (rank, g, same), flush=True)
        ok = ok and same
    print("rank %d %s" % (rank, "ok" if ok else "FAILED"), flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
