"""The self-play loop on one GPU: play with model N, record, train model N+1 on the records, play N+1 against N.

    python tools/self_play.py --init init:1 --rounds 2 --games 256 --h2h-games 256 --out selfplay.json

Each round records an arena of the current model (default: six deep seats on value-model slot 0, root mode, winner labels; see
citadels_self_play_b200/selfplay.py for why deep seats are recorded that way), splits the records by game, trains from the
dataset on the device starting from the current model, saves <--dir>/round_<k>.pt and plays arena.head_to_head(new, previous).
--init is a state_dict (.pt), a .npz of sd_* tensors or init:SEED (tools/head_to_head.load_model).  Writes one JSON file: per
round the record and drop counts, records per game, the arena's per-phase CUDA-event times (record included), the loss curves,
the head-to-head result; wall time; the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from arena_experiment import gpu_info
from head_to_head import load_model


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
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    from citadels_self_play_b200 import Engine, arena, selfplay
    from citadels_self_play_b200.value_model import load_checkpoint
    torch.cuda.set_device(0)
    os.makedirs(args.dir, exist_ok=True)
    player = arena.deep(args.iterations, args.depth, args.weight)
    current = load_model(args.init)
    per_game = 256 if args.mode == "root" else 2048
    max_records = args.max_records or args.games * per_game
    rounds = []
    eng = Engine(capacity=args.capacity, device=0)
    t0 = time.perf_counter()
    try:
        for k in range(1, args.rounds + 1):
            r0 = time.perf_counter()
            # every round plays new deals: round k's recorded games and head-to-head deals do not overlap any other round's
            first_gid = k * 10_000_000
            rec = selfplay.record_arena(args.games, [player] * 6, record_seats=range(6), models=[current], mode=args.mode,
                                        threshold=args.threshold, engine=eng, seed=args.seed, first_gid=first_gid, max_records=max_records)
            data = eng.dataset_read()
            train_idx, val_idx = selfplay.split_by_game(data["origin"], args.val_fraction, seed=args.seed + k, rows=data["row"])
            if args.label == "winner":   # errored games have no outcome to learn from
                keep = data["origin"]["winner"] >= 0
                ok = set(data["row"][keep].tolist())
                train_idx = [r for r in train_idx if int(r) in ok]
                val_idx = [r for r in val_idx if int(r) in ok]
            history = {}
            folder = os.path.join(args.dir, "round_%d" % k)
            best = selfplay.train_on_dataset(eng, train_idx, val_idx, args.label, epochs=args.epochs, lr=args.lr, gamma=args.gamma,
                                             batch_size=args.batch_size, model=current, seed=args.seed + k, parent_folder=folder,
                                             history=history)
            new = load_checkpoint(os.path.join(folder, "best_model.pt"))
            torch.save(new.state_dict(), os.path.join(args.dir, "round_%d.pt" % k))
            h2h = arena.head_to_head(args.h2h_games, new, current, player=player, engine=eng, seed=args.seed,
                                     first_gid=first_gid + 5_000_000)
            h2h_phase = [p["phase_ms"] for p in h2h.pop("passes")]
            info = rec["info"]
            rounds.append(dict(round=k, games=args.games, records=info["records"], option_slots=info["option_slots"],
                               dropped_trees=info["dropped_trees"], dropped_records=info["dropped_records"],
                               records_per_game=info["records"] / max(1, args.games), searches=int(rec["searches"].sum()),
                               record_stats=rec["stats"], record_phase_ms=rec["phase_ms"], train_rows=len(train_idx), val_rows=len(val_idx),
                               best_eval_loss=best, train_losses=history["train_losses"], eval_losses=history["eval_losses"],
                               head_to_head=h2h, head_to_head_phase_ms=h2h_phase, wall_s=time.perf_counter() - r0))
            print(json.dumps(dict(round=k, records=info["records"], dropped_records=info["dropped_records"], best_eval_loss=best,
                                  sign_test=h2h["sign_test"], a=h2h["a"], b=h2h["b"])), flush=True)
            current = new
    finally:
        eng.close()
    out = dict(gpu=gpu_info(0), init=args.init, label=args.label, mode=args.mode, threshold=args.threshold, iterations=args.iterations,
               depth=args.depth, weight=args.weight, epochs=args.epochs, lr=args.lr, batch_size=args.batch_size, seed=args.seed,
               rounds=rounds, wall_s=time.perf_counter() - t0)
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
