"""The self-play loop on one GPU: play with model N, record, train model N+1 on the records, play N+1 against N.

    python tools/self_play.py --init init:1 --rounds 2 --games 256 --h2h-games 256 --out selfplay.json

Each round records an arena of the current model (default: six deep seats on value-model slot 0, root mode, winner labels; see
citadels_self_play_b200/selfplay.py for why deep seats are recorded that way), splits the records by game, trains from the
dataset on the device starting from the current model, saves <--dir>/round_<k>.pt and plays arena.head_to_head(new, previous).
--init is a state_dict (.pt), a .npz of sd_* tensors or init:SEED (tools/head_to_head.load_model).  Writes one JSON file: per
round the record and drop counts, records per game, the arena's per-phase CUDA-event times (record included), the loss curves,
the head-to-head result; wall time; the GPU's name and power limit read in the same run.

Under torchrun, one rank per GPU:
    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29514 tools/self_play.py --init init:1 --out sp.json
every rank records its own block of the round's games on its own GPU (LOCAL_RANK), selfplay.gather_dataset brings all records to
rank 0's engine, rank 0 splits and trains, the new model is broadcast, and every rank plays its block of the head-to-head deals.
The JSON then also holds world, the records each rank contributed and the gather's wall time.
--save-datasets DIR writes each round's dataset (all ranks' records) to DIR/round_<k>.npz; --window K trains round k on its own
records plus the saved datasets of rounds k-K+1 .. k-1."""
import argparse
import copy
import datetime
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from arena_experiment import gpu_info
from head_to_head import load_model


def _file_sizes(path):
    """(records, option slots) of a selfplay.save_dataset file"""
    with np.load(path, allow_pickle=False) as z:
        return len(z["meta"]), len(z["options"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--init", required=True, help="starting model: FILE.pt, FILE.npz or init:SEED")
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--games", type=int, default=256, help="recorded games per round")
    ap.add_argument("--h2h-games", type=int, default=256, help="head-to-head deals per round (each played twice)")
    ap.add_argument("--label", choices=("winner", "node_value"), default="winner")
    ap.add_argument("--mode", choices=("root", "tree"), default="root")
    ap.add_argument("--threshold", type=float, default=15.0, help="tree mode: node_value.sum() >= threshold")
    ap.add_argument("--iterations", type=int, default=200)
    ap.add_argument("--depth", type=int, default=10)
    ap.add_argument("--weight", type=float, default=5.0, help="model_reward_weights")
    ap.add_argument("--epochs", type=int, default=20)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--gamma", type=float, default=1.0)
    ap.add_argument("--batch-size", type=int, default=64)
    ap.add_argument("--val-fraction", type=float, default=0.1)
    ap.add_argument("--max-records", type=int, default=0, help="dataset rows (0: 256 per game in root mode, 2048 in tree mode)")
    ap.add_argument("--seed", type=int, default=20261020)
    ap.add_argument("--capacity", type=int, default=4096, help="roots per search launch")
    ap.add_argument("--dir", default="selfplay_rounds", help="where round_<k>.pt go")
    ap.add_argument("--save-datasets", default=None, metavar="DIR", help="write each round's dataset to DIR/round_<k>.npz")
    ap.add_argument("--window", type=int, default=1, help="train on this round and the saved datasets of the K-1 before it")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if args.window < 1 or (args.window > 1 and not args.save_datasets):
        ap.error("--window K needs K >= 1, and --save-datasets for K > 1")
    from citadels_self_play_b200 import Engine, arena, selfplay, sharding
    from citadels_self_play_b200.engine import DATASET_KEYS
    from citadels_self_play_b200.value_model import load_checkpoint
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if distributed:   # rank 0 trains while the others wait at the model's broadcast: allow a long round
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(hours=6))
    rank, world = (dist.get_rank(), dist.get_world_size()) if distributed else (0, 1)
    if rank == 0:
        os.makedirs(args.dir, exist_ok=True)
        if args.save_datasets:
            os.makedirs(args.save_datasets, exist_ok=True)
    player = arena.deep(args.iterations, args.depth, args.weight)
    current = load_model(args.init)
    per_game = 256 if args.mode == "root" else 2048
    # every rank records with the same room, so the records it keeps do not depend on its rank
    room = args.max_records or arena.rank_block(args.games, 0, world)[1] * per_game
    rounds = []
    eng = Engine(capacity=args.capacity, device=local)
    # Rank 0 trains on more than its own records (the other ranks', the window's saved rounds): they are pooled in an engine of
    # their own, reserved for the round's known sizes.  One process with --window 1 trains where it recorded, as it always did.
    pooled = rank == 0 and (world > 1 or args.window > 1)
    train_eng = Engine(capacity=1, device=local) if pooled else eng
    t0 = time.perf_counter()
    try:
        for k in range(1, args.rounds + 1):
            r0 = time.perf_counter()
            # every round plays new deals: round k's recorded games and head-to-head deals do not overlap any other round's
            first_gid = k * 10_000_000
            rec = selfplay.record_arena(args.games, [player] * 6, record_seats=range(6), models=[current], mode=args.mode,
                                        threshold=args.threshold, engine=eng, seed=args.seed, first_gid=first_gid, max_records=room)
            counts, gather_s = {key: [rec["info"][key]] for key in selfplay.COUNT_KEYS}, 0.0
            window = [os.path.join(args.save_datasets, "round_%d.npz" % j) for j in range(max(1, k - args.window + 1), k)]
            if pooled:   # room for every rank's records (record_arena's default of 16 option slots per record) and the window's
                sizes = [_file_sizes(p) for p in window]
                train_eng.dataset_reserve(world * room + sum(r for r, _ in sizes), 16 * world * room + sum(s for _, s in sizes))
            if distributed:
                dist.barrier()
            g0 = time.perf_counter()
            if pooled:   # rank 0's own records first, device to device
                own = eng.dataset_tensors("cuda:%d" % local)
                train_eng.dataset_append(*(own[key] for key in DATASET_KEYS))
                del own
            if distributed:
                counts = selfplay.gather_dataset(train_eng, dst=0)
                gather_s = time.perf_counter() - g0
                if rank == 0:   # the pooled copy of rank 0's records has dropped none: its drops are the recording engine's
                    for key in ("dropped_trees", "dropped_records"):
                        counts[key][0] = rec["info"][key]
            best = history = train_idx = val_idx = None
            if rank == 0:
                if args.save_datasets:
                    selfplay.save_dataset(train_eng, os.path.join(args.save_datasets, "round_%d.npz" % k))
                for path in window:
                    selfplay.load_dataset(train_eng, path)
                data = train_eng.dataset_read()
                train_idx, val_idx = selfplay.split_by_game(data["origin"], args.val_fraction, seed=args.seed + k, rows=data["row"])
                if args.label == "winner":   # errored games have no outcome to learn from
                    keep = data["origin"]["winner"] >= 0
                    ok = set(data["row"][keep].tolist())
                    train_idx = [r for r in train_idx if int(r) in ok]
                    val_idx = [r for r in val_idx if int(r) in ok]
                history = {}
                folder = os.path.join(args.dir, "round_%d" % k)
                best = selfplay.train_on_dataset(train_eng, train_idx, val_idx, args.label, epochs=args.epochs, lr=args.lr, gamma=args.gamma,
                                                 batch_size=args.batch_size, model=current, seed=args.seed + k, parent_folder=folder,
                                                 history=history)
                new = load_checkpoint(os.path.join(folder, "best_model.pt"))
                torch.save(new.state_dict(), os.path.join(args.dir, "round_%d.pt" % k))
            else:
                new = copy.deepcopy(current)
            if distributed:   # rank 0's new model to every rank
                for t in new.state_dict().values():
                    buf = t.to("cuda:%d" % local)
                    dist.broadcast(buf, 0)
                    t.copy_(buf.cpu())
            h2h = arena.head_to_head(args.h2h_games, new, current, player=player, engine=eng, seed=args.seed,
                                     first_gid=first_gid + 5_000_000)
            h2h_phase = [p["phase_ms"] for p in h2h.pop("passes")]
            total = {key: sum(v) for key, v in counts.items()}
            searches = sharding.reduce_sum([int(rec["searches"].sum())], "cuda:%d" % local if distributed else "cpu")[0]
            if rank == 0:
                rnd = dict(round=k, games=args.games, records=total["records"], option_slots=total["option_slots"],
                           dropped_trees=total["dropped_trees"], dropped_records=total["dropped_records"],
                           records_per_game=total["records"] / max(1, args.games), searches=searches, record_stats=rec["stats"],
                           record_phase_ms=rec["phase_ms"], train_rows=len(train_idx), val_rows=len(val_idx), best_eval_loss=best,
                           train_losses=history["train_losses"], eval_losses=history["eval_losses"], head_to_head=h2h,
                           head_to_head_phase_ms=h2h_phase, wall_s=time.perf_counter() - r0)
                if distributed:
                    rnd.update(world=world, rank_records=counts["records"], gather_s=gather_s)
                rounds.append(rnd)
                print(json.dumps(dict(round=k, records=total["records"], dropped_records=total["dropped_records"], best_eval_loss=best,
                                      sign_test=h2h["sign_test"], a=h2h["a"], b=h2h["b"])), flush=True)
            current = new
    finally:
        eng.close()
        train_eng.close()
    if rank == 0:
        out = dict(gpu=gpu_info(local), init=args.init, label=args.label, mode=args.mode, threshold=args.threshold,
                   iterations=args.iterations, depth=args.depth, weight=args.weight, epochs=args.epochs, lr=args.lr,
                   batch_size=args.batch_size, seed=args.seed, rounds=rounds, wall_s=time.perf_counter() - t0)
        if distributed:
            out["world"] = world
        d = os.path.dirname(os.path.abspath(args.out))
        os.makedirs(d, exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
