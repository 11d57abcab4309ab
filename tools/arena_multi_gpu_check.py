"""arena.play_arena under torchrun (each rank its own GPU and its own block of game ids), called without an engine, against one
engine playing every game alone on the same GPU:
     torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 tools/arena_multi_gpu_check.py
Every rank checks its per-game arrays against its slice of the single-engine run and the summed statistics against that run's.
Prints one JSON line on rank 0."""
import json
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from citadels_self_play_b200 import Engine, arena

N, SEED, GID0 = 50, 20261020, 70_000
seats = [arena.pure(30), arena.random_seat(), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.random_seat()]
res = arena.play_arena(N, seats=seats, seed=SEED, first_gid=GID0)
first, count = arena.rank_block(N, rank, world)
eng = Engine(capacity=64, device=local)
solo = eng.arena(N, seats, seed=SEED, first_gid=GID0)
eng.close()
assert res["first_gid"] == GID0 + first and len(res["winner"]) == count
for k in ("winner", "points", "steps", "searches"):
    assert np.array_equal(res[k], solo[k][first:first + count]), (rank, k)
for k in ("games", "steps", "steps_sq", "errors", "wins", "points_sum", "points_sq", "max_steps"):
    assert res["stats"][k] == solo["stats"][k], (rank, k, res["stats"][k], solo["stats"][k])
devs = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
dist.all_gather(devs, torch.tensor([torch.cuda.current_device()], dtype=torch.int64, device="cuda"))
if rank == 0:
    print(json.dumps(dict(world=world, games=N, devices=[int(d.item()) for d in devs], wins=res["winners"],
                          equals_single_engine=True)), flush=True)
dist.barrier()
dist.destroy_process_group()
