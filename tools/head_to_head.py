"""Is checkpoint A better than checkpoint B?  Both value models play deep MCCFR against each other on the device arena
(arena.head_to_head): every deal is played twice, with --pattern and with A and B swapped, so that the luck of the deal and of
the seats cancels.

    python tools/head_to_head.py --a pretrain/best_model.pt --b init:1 --games 2000 --out result.json
    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29513 tools/head_to_head.py --a ... --b ... --out result.json

A checkpoint is a state_dict as train.py writes it (.pt, loaded with value_model.load_checkpoint), a .npz holding the state_dict's
tensors under sd_* keys (tests/golden/value_best_model.npz), or init:SEED, a freshly initialised ValueOnlyNN(418, 512) after
torch.manual_seed(SEED).  Writes one JSON file (rank 0): the head_to_head result (wins, shares with Wilson 99 % intervals, wins
per seat of each pass, pair counts, the sign test of A-won-both against B-won-both), wall seconds, the CUDA-event time of the
advance / search / apply phases of each pass (max over ranks) and the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from arena_experiment import gpu_info


def load_model(spec):
    """A ValueOnlyNN(418, 512) in eval mode from a .pt state_dict, a .npz of sd_* tensors or init:SEED."""
    from citadels_self_play_b200.value_model import ValueOnlyNN, load_checkpoint
    if spec.startswith("init:"):
        torch.manual_seed(int(spec[5:]))
        return ValueOnlyNN(418, 512).eval()
    if spec.endswith(".npz"):
        with np.load(spec) as f:
            sd = {k[3:]: torch.from_numpy(f[k]) for k in f.files if k.startswith("sd_")}
        m = ValueOnlyNN(418, 512)
        m.load_state_dict(sd)
        return m.eval()
    return load_checkpoint(spec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="checkpoint A: FILE.pt, FILE.npz or init:SEED")
    ap.add_argument("--b", required=True, help="checkpoint B")
    ap.add_argument("--games", type=int, default=2000, help="deals; each is played twice")
    ap.add_argument("--iterations", type=int, default=200)
    ap.add_argument("--depth", type=int, default=10)
    ap.add_argument("--weight", type=float, default=5.0, help="model_reward_weights")
    ap.add_argument("--pattern", default="ABABAB", help="seat 0..5: A, B or R (random)")
    ap.add_argument("--seed", type=int, default=20261020)
    ap.add_argument("--first-gid", type=int, default=0)
    ap.add_argument("--capacity", type=int, default=4096, help="roots per search launch")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if distributed:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = (dist.get_rank(), dist.get_world_size()) if distributed else (0, 1)
    from citadels_self_play_b200 import Engine, arena, sharding
    model_a, model_b = load_model(args.a), load_model(args.b)
    player = arena.deep(args.iterations, args.depth, args.weight)
    dev = "cuda:%d" % local if distributed else "cpu"
    eng = Engine(capacity=args.capacity, device=local)
    try:
        # loads the modules and the kernels' first-launch state outside the timed call, on games the timed call does not play
        arena.head_to_head(2 * world, model_a, model_b, player=player, pattern=args.pattern, engine=eng, seed=args.seed,
                           first_gid=args.first_gid + args.games + 1_000_000)
        if distributed:
            dist.barrier()
        t0 = time.perf_counter()
        r = arena.head_to_head(args.games, model_a, model_b, player=player, pattern=args.pattern, engine=eng, seed=args.seed,
                               first_gid=args.first_gid)
        wall = sharding.reduce_max([time.perf_counter() - t0], dev)[0]
    finally:
        eng.close()
    phases = [sharding.reduce_max([p["phase_ms"][k] for k in ("advance", "search", "apply")], dev) for p in r["passes"]]
    passes = [dict(stats=p["stats"], phase_ms_max_over_ranks=dict(zip(("advance", "search", "apply"), ph)))
              for p, ph in zip(r["passes"], phases)]
    result = {k: v for k, v in r.items() if k != "passes"}
    out = dict(gpu=gpu_info(local), world=world, a=args.a, b=args.b, seed=args.seed, first_gid=args.first_gid,
               iterations=args.iterations, depth=args.depth, weight=args.weight, result=result, passes=passes, wall_s=wall,
               game_pairs_per_s=result["games"] / wall)
    if rank == 0:
        print(json.dumps(dict(result, wall_s=wall)), flush=True)
        d = os.path.dirname(os.path.abspath(args.out))
        os.makedirs(d, exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
