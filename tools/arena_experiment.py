"""The README's win-rate experiment (compare_to_random.py) at a useful size, on the device arena (arena.play_arena).

    python tools/arena_experiment.py --games 10000 --out result.json
    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29512 tools/arena_experiment.py --out result.json

Three configurations, each seat 0 deep MCCFR with the reference's trained checkpoint (tests/golden/value_best_model.npz), seat 1
pure MCCFR, seats 2-5 random:  deep(2000, depth 100) vs pure(2000),  deep(200, depth 10) vs pure(200),  deep(200, depth 10) vs
pure(2000).  Per configuration: wins and win rates with Wilson 99 % intervals, the README's 100-game counts and a chi-square test
of them against the measured rates, wall seconds, games/s and the CUDA-event time of the advance / search / apply phases.
Also times arena.play_games_batched (host-driven game steps, batched searches) against play_arena on the same small experiment
in the same process.  The GPU's name and power limit are read in the same run.  Writes one JSON file (rank 0)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

# the README's charts (images/*.png of the reference): winners of 100 games per seat
CONFIGS = [
    dict(name="deep2000_d100_vs_pure2000", deep=(2000, 100), pure=2000, readme_counts=[24, 36, 5, 7, 9, 19]),
    dict(name="deep200_d10_vs_pure200", deep=(200, 10), pure=200, readme_counts=[35, 12, 14, 10, 12, 17]),
    dict(name="deep200_d10_vs_pure2000", deep=(200, 10), pure=2000, readme_counts=[34, 24, 7, 12, 9, 14]),
]


def readme_chi2(counts, rates):
    """Pearson chi-square of the README's 100 games against the measured rates taken as the true distribution (5 dof)."""
    from scipy.stats import chi2
    counts = np.asarray(counts, dtype=np.float64)
    exp = counts.sum() * np.asarray(rates, dtype=np.float64)
    stat = float((((counts - exp) ** 2) / exp).sum())
    return dict(statistic=stat, dof=5, p_value=float(chi2.sf(stat, 5)))


def gpu_info(device):
    info = dict(name=torch.cuda.get_device_name(device), power_limit_w=None)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in q.stdout.strip().split(",")]
        info.update(power_limit_w=float(pl), max_sm_clock_mhz=float(clk))
    except Exception as ex:   # report what could not be read rather than guess it
        info["query_error"] = repr(ex)
    return info


def load_checkpoint():
    from citadels_self_play_b200.value_model import ValueOnlyNN
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with np.load(os.path.join(root, "tests", "golden", "value_best_model.npz")) as f:
        sd = {k[3:]: torch.from_numpy(f[k]) for k in f.files if k.startswith("sd_")}
    m = ValueOnlyNN(418, 512)
    m.load_state_dict(sd)
    return m.eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=10000)
    ap.add_argument("--configs", default="all", help="comma-separated configuration names, or 'all'")
    ap.add_argument("--seed", type=int, default=20261020)
    ap.add_argument("--capacity", type=int, default=4096, help="roots per search launch")
    ap.add_argument("--compare-games", type=int, default=64)
    ap.add_argument("--compare-iterations", type=int, default=200)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if distributed:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = (dist.get_rank(), dist.get_world_size()) if distributed else (0, 1)
    from citadels_self_play_b200 import Engine, arena, sharding
    from citadels_self_play_b200.arena import wilson
    model = load_checkpoint()
    eng = Engine(capacity=args.capacity, device=local)
    eng.set_value_model(model)
    out = dict(gpu=gpu_info(local), world=world, games_per_config=args.games, seed=args.seed,
               checkpoint="tests/golden/value_best_model.npz (the reference's pretrain/best_model.pt)",
               checkpoint_note="It is not known whether the README's charts were made with this checkpoint.",
               readme_note="README counts: 100 games per configuration, read off images/*.png of the reference; hardware unspecified.",
               configs=[])
    names = [c["name"] for c in CONFIGS] if args.configs == "all" else args.configs.split(",")
    for ci, cfg in enumerate(CONFIGS):
        if cfg["name"] not in names:
            continue
        seats = [arena.deep(cfg["deep"][0], cfg["deep"][1], 5.0), arena.pure(cfg["pure"])] + [arena.random_seat()] * 4
        if distributed:
            dist.barrier()
        t0 = time.perf_counter()
        # game ids by position in CONFIGS: a configuration plays the same games however it is selected
        r = arena.play_arena(args.games, seats=seats, engine=eng, seed=args.seed, first_gid=ci * 10_000_000)
        wall = sharding.reduce_max([time.perf_counter() - t0], "cuda:%d" % local if distributed else "cpu")[0]
        ph = r["phase_ms"]
        phases = sharding.reduce_max([ph["advance"], ph["search"], ph["apply"]], "cuda:%d" % local if distributed else "cpu")
        st = r["stats"]
        decided = st["games"] - st["errors"]
        rates = [w / decided if decided else 0.0 for w in st["wins"]]
        out["configs"].append(dict(
            name=cfg["name"], seats=[list(s) for s in seats], games=st["games"], errors=st["errors"], wins=st["wins"],
            win_rates=rates, wilson99=[wilson(w, decided) for w in st["wins"]],
            mean_points=[p / st["games"] for p in st["points_sum"]], mean_steps=st["steps"] / st["games"],
            searches_rank0=int(r["searches"].sum()), max_searches_in_a_game_rank0=int(r["searches"].max()),
            readme_counts=cfg["readme_counts"], readme_chi2_vs_measured=readme_chi2(cfg["readme_counts"], rates),
            wall_s=wall, games_per_s=st["games"] / wall,
            phase_ms_max_over_ranks=dict(advance=phases[0], search=phases[1], apply=phases[2])))
        if rank == 0:
            print(json.dumps(out["configs"][-1]), flush=True)
    if rank == 0 and args.compare_games > 0:
        # the same small experiment both ways: seat 1 pure MCCFR, every other seat random (play_games_batched's seat 0 is random
        # without a model).  The two drivers draw the random seats' moves from different streams, so only the time is compared.
        # Each timed call sets up its engines as a caller would (play_games_batched makes its search engine, the arena a fresh
        # engine); one untimed call of each before loads modules and makes the facade's default engine.
        n, it = args.compare_games, args.compare_iterations
        seats = [arena.random_seat(), arena.pure(it)] + [arena.random_seat()] * 4

        def run_arena(k, gid0):
            e = Engine(capacity=max(1, k), device=local)
            try:
                return e.arena(k, seats, seed=args.seed, first_gid=gid0)
            finally:
                e.close()
        arena.play_games_batched(2, None, seed=args.seed, first_gid=60_000_000, pure_iterations=it)
        run_arena(2, 60_000_000)
        t0 = time.perf_counter()
        wb = arena.play_games_batched(n, None, seed=args.seed, first_gid=50_000_000, pure_iterations=it)
        t_b = time.perf_counter() - t0
        t0 = time.perf_counter()
        ra = run_arena(n, 50_000_000)
        t_a = time.perf_counter() - t0
        out["driver_comparison"] = dict(games=n, seats=[list(s) for s in seats], play_games_batched_s=t_b, play_arena_s=t_a,
                                        speedup=t_b / t_a, play_games_batched_wins=wb, play_arena_wins=ra["stats"]["wins"])
        print(json.dumps(out["driver_comparison"]), flush=True)
    eng.close()
    if rank == 0:
        d = os.path.dirname(os.path.abspath(args.out))
        os.makedirs(d, exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
