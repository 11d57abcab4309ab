#!/usr/bin/env python
"""bench.py -- env steps/sec of batched 6-player random playouts (BASELINE.json metric, configs[1]) and MCCFR iterations/sec.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--games G] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: G independent preset games per GPU, dealt on the device from
(seed, global game id) and played uniformly at random to terminal by the fused playout kernel.
  value      weak scaling: every rank plays G games per step (rank r owns global ids [(step*world + r)*G, ...)), no collective
             on the step path; one all-reduce of the outcome histogram after the timed region
  strong     the same K steps with G games IN TOTAL, G/world per rank (BASELINE configs[1]: "1M playouts sharded over 1/2/4/8")
  e2e        the same metric through the reference-facing calls with HOST buffers (ctd_load_states + ctd_playout_slots)
  mccfr      secondary metric: pure / deep MCCFR iterations/s (configs[2], [3]), 2000-iteration data generation (configs[4]),
             device-event, wall-clock and host-buffer end-to-end figures; classic-eight figures (the ruleset north_star names)
  cpu_baseline / --impl reference    the reference's own loops timed on the box's host cores: the REAL reference when
             oracle/_ref (its byte-compiled modules, oracle/build_ref.py) travelled with the repo -- kind "reference" --,
             otherwise the oracle's Python port -- kind "port"
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
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

BYTES_PER_STEP = 512          # SURVEY.md 8(d): read + write of the 256 B packed playout record per env step
BYTES_PER_ITER = 2048         # SURVEY.md 8(d): nominal bytes per MCCFR iteration
SEED = 0xC17ADE15
METRIC = "env steps/sec (batched 6p random playouts)"
RULESETS = ["preset", "classic", "random-ruleset"]


def _traffic(games_per_launch):
    """DRAM bytes per launch of the playout kernel from the committed ncu capture, scaled by games per launch."""
    for name in ("r02_playout_traffic.json", "r01_playout_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            t = json.load(open(p))
            return (t["dram_bytes_read"] + t["dram_bytes_write"]) * (games_per_launch / t["games"]), "profiles/" + name
        except Exception:
            continue
    return None, None


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------- CPU arm
# Workers run in a process pool on every host core (multiprocessing, fork).  kind "reference": oracle/_ref, the REAL
# reference byte-compiled from /root/reference (oracle/build_ref.py), driven by its own `random`; kind "port": the oracle.
def _w_ref_playouts(args):
    seed, n = args
    from oracle import ref_loop
    s, g, t, _ = ref_loop.playouts(n, seed)
    return s, t


def _w_ref_pure(args):
    seed, n, iters = args
    from oracle import ref_loop
    it, _, t = ref_loop.pure_mccfr(n, seed, iters)
    return it, t


def _w_ref_deep(args):
    seed, n, iters = args
    from oracle import ref_loop
    it, _, t = ref_loop.deep_mccfr(n, seed, iters)
    return it, t


def _w_port_playouts(args):
    seed, gid0, n, ruleset = args
    from oracle import citadels_oracle as O
    steps = 0
    t0 = time.perf_counter()
    for i in range(n):
        steps += O.playout(seed, gid0 + i, ruleset)[2]
    return steps, time.perf_counter() - t0


def _w_port_pure(args):
    seed, gid0, n, iters = args
    from oracle import mccfr_oracle as M
    from oracle.philox import PhiloxChance
    its = 0
    t0 = time.perf_counter()
    for i in range(n):
        g, _ = M.make_root(seed, gid0 + i, 0, 0, 20)
        if g.terminal:
            continue
        g.chance = PhiloxChance(seed, gid0 + i, stream=1)
        M.Node(g, g.player).cfr_train(iters)
        its += iters
    return its, time.perf_counter() - t0


def _pool_run(fn, jobs):
    """-> (units, seconds) over a fork pool with one process per job, all running at once.  Seconds = the slowest worker's own
    timed region (interpreter start-up, `import torch` and, for the MCCFR legs, root construction are outside it)."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(len(jobs)) as pool:
        res = pool.map(fn, jobs, chunksize=1)
    return sum(r[0] for r in res), max(r[1] for r in res)


def ref_available():
    try:
        from oracle import ref_loop
        return ref_loop.available()
    except Exception:
        return False


def cpu_playouts(games_per_core, cores, salt=0, ruleset=0, kind=None):
    """The reference's random-playout loop (run_utils.py:37-41) on `cores` processes.  -> (env_steps, wall_seconds, kind)"""
    kind = kind or ("reference" if ref_available() and ruleset == 0 else "port")
    if kind == "reference":
        s, w = _pool_run(_w_ref_playouts, [(1000 + salt * cores + c, games_per_core) for c in range(cores)])
    else:
        s, w = _pool_run(_w_port_playouts, [(SEED, 10_000_000 + (salt * cores + c) * games_per_core, games_per_core, ruleset)
                                            for c in range(cores)])
    return s, w, kind


def cpu_mccfr(roots_per_core, cores, iters=200, deep=False, kind=None):
    """run_mccfr(game, max_iterations=200) / CFRNode(...).cfr_pred(200, 10) on near-terminal roots, all host cores."""
    kind = kind or ("reference" if ref_available() else "port")
    if kind == "reference":
        it, w = _pool_run(_w_ref_deep if deep else _w_ref_pure, [(2000 + c, roots_per_core, iters) for c in range(cores)])
    else:
        if deep:
            return None
        it, w = _pool_run(_w_port_pure, [(SEED, 10_000 + c * roots_per_core, roots_per_core, iters) for c in range(cores)])
    return it, w, kind


def run_reference_arm(args, rank, world, emit):
    """The reference's own CPU implementation of the path on this box's host cores: K timed steps (after W warm-up steps) of
    `--ref-games-per-core` games per core each, the loop at run_utils.py:37-41."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_core = max(1, args.ref_games_per_core)
    kind = "reference" if ref_available() and args.ruleset == 0 else "port"
    for w in range(args.warmup):
        cpu_playouts(max(1, per_core // 10), cores, salt=100 + w, ruleset=args.ruleset, kind=kind)
    tot_steps, tot_wall = 0, 0.0
    for k in range(args.steps):
        s, w, _ = cpu_playouts(per_core, cores, salt=k, ruleset=args.ruleset, kind=kind)
        tot_steps += s
        tot_wall += w
    v = tot_steps / tot_wall
    what = ("the unmodified reference (oracle/_ref: its modules byte-compiled from /root/reference), random.seed per worker"
            if kind == "reference" else "oracle port (oracle/_ref not present)")
    sample = "%d games per step (%d per core x %d cores) of the %s random playout, %s" % (
        per_core * cores, per_core, cores, RULESETS[args.ruleset], what)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "env steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "%s 6p random playouts to terminal (BASELINE configs[1]), bounded CPU sample" % RULESETS[args.ruleset],
                       "sample": sample},
            "cpu_baseline": {"value": v, "unit": "env steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "env steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if kind == "reference":   # the port next to it, and the two MCCFR loops, as extra keys
        ps, pw, _ = cpu_playouts(per_core, cores, salt=50, ruleset=args.ruleset, kind="port")
        line["port"] = {"value": ps / pw, "unit": "env steps/s", "cores": cores, "kind": "port"}
        it, w, _ = cpu_mccfr(4, cores, kind="reference")
        line["mccfr_pure"] = {"value": it / w, "unit": "iterations/s", "cores": cores, "kind": "reference",
                              "sample": "%d roots x 200 iterations, run_utils.run_mccfr" % (4 * cores)}
        it, w, _ = cpu_mccfr(4, cores, deep=True, kind="reference")
        line["mccfr_deep"] = {"value": it / w, "unit": "iterations/s", "cores": cores, "kind": "reference",
                              "sample": "%d roots x 200 iterations, CFRNode(model=ValueOnlyNN(418,512), device='cpu').cfr_pred(200, 10)" % (4 * cores)}
    emit(line)


# ------------------------------------------------------------------------------------------- GPU arm: MCCFR
def bench_mccfr(args, rank, world, local, torch):
    """Secondary metric.  Returns (ints for all_reduce SUM, floats for all_reduce MAX, dict of rank-0-only extras)."""
    import numpy as np
    from citadels_self_play_b200 import Engine, sharding
    from citadels_self_play_b200.value_model import ValueOnlyNN
    R, IT = args.mccfr_roots, 200
    out = {}

    def status_split(res):
        st = res["status"]
        return [int(((st & 2) != 0).sum()), int(((st & 4) != 0).sum()), int(((st & 16) != 0).sum()), int((st == 1).sum())]

    eng = Engine(capacity=R, device=local)
    eng.make_roots(R, seed=SEED, first_gid=sharding.first_gid(0, rank, world, R), back_lo=0, back_hi=20)
    # -- pure (configs[2]): device events and wall clock
    eng.mccfr(R, iterations=IT, seed=SEED)
    pure_it = pure_ms = pure_wall = 0
    for _ in range(2):
        t0 = time.perf_counter()
        o = eng.mccfr(R, iterations=IT, seed=SEED)
        pure_wall += time.perf_counter() - t0
        pure_it += int(o["results"]["iterations"].sum())
        pure_ms += o["kernel_ms"]
    split = status_split(o["results"])
    # -- host-buffer end to end: roots in host memory -> ctd_load_roots -> ctd_mccfr -> result records on the host
    roots, knows, used, gids = eng.store_roots(R)
    eng.load_roots(roots, knows, used, gids)
    eng.mccfr(R, iterations=IT, seed=SEED)
    t0 = time.perf_counter()
    e2e_it = 0
    for _ in range(2):
        eng.load_roots(roots, knows, used, gids)
        e2e_it += int(eng.mccfr(R, iterations=IT, seed=SEED)["results"]["iterations"].sum())
    e2e_wall = time.perf_counter() - t0
    out["e2e_h2d_bytes"] = int(roots.nbytes + knows.nbytes + used.nbytes + gids.nbytes)
    out["e2e_d2h_bytes"] = int(o["results"].nbytes)
    # -- deep (configs[3])
    torch.manual_seed(0)
    eng.set_value_model(ValueOnlyNN(418, 512).eval())
    eng.mccfr_pred(R, iterations=IT, max_depth=10, seed=SEED)
    deep_it = deep_ms = deep_wall = 0
    for _ in range(2):     # the engine's default: fused (one launch, every warp evaluates its own leaves)
        t0 = time.perf_counter()
        o = eng.mccfr_pred(R, iterations=IT, max_depth=10, seed=SEED)
        deep_wall += time.perf_counter() - t0
        deep_it += int(o["results"]["iterations"].sum())
        deep_ms += o["kernel_ms"]
    out["deep_waves"] = int(o["waves"])
    eng.set_value_backend("tcgen05")   # for comparison: waves, leaves batched on the tensor cores
    eng.mccfr_pred(R, iterations=IT, max_depth=10, seed=SEED)
    ow = eng.mccfr_pred(R, iterations=IT, max_depth=10, seed=SEED)
    out["deep_waves_tc"] = int(ow["waves"])
    tc_it, tc_ms = int(ow["results"]["iterations"].sum()), ow["kernel_ms"]
    eng.set_value_backend("fused")
    split = [a + b for a, b in zip(split, status_split(o["results"]))]
    eng.close()
    # -- configs[4]: training-data generation, 2000 iterations, create_a_random_game(100) roots, nodes with >= 200 backprops
    R5 = max(64, R // 4)
    eng = Engine(capacity=R5, device=local)
    eng.make_roots(R5, seed=SEED, first_gid=sharding.first_gid(1, rank, world, R5), back_lo=1, back_hi=100, flavour=1)
    eng.mccfr(R5, iterations=2000, seed=SEED)
    t0 = time.perf_counter()
    o5 = eng.mccfr(R5, iterations=2000, seed=SEED)
    gen_wall = time.perf_counter() - t0
    eng.mccfr_targets(R5, iterations=2000, seed=SEED, threshold=200.0)   # warm-up: the first call loads the kernel and sizes buffers
    t5 = time.perf_counter()
    tg = eng.mccfr_targets(R5, iterations=2000, seed=SEED, threshold=200.0)
    t5 = time.perf_counter() - t5
    split = [a + b for a, b in zip(split, status_split(o5["results"]))]
    gen_it, gen_ms, gen_targets = int(o5["results"]["iterations"].sum()), o5["kernel_ms"], len(tg["meta"])
    eng.close()
    # -- the classic eight (the characters north_star lists): pure MCCFR on as many roots (a Magician's turn expands ~1600 children
    # at once: a few such trees are the tail of a small batch)
    Rc = R
    eng = Engine(capacity=Rc, device=local)
    eng.make_roots(Rc, seed=SEED, first_gid=sharding.first_gid(2, rank, world, Rc), ruleset=1, back_lo=0, back_hi=20)
    eng.mccfr(Rc, iterations=IT, seed=SEED, ruleset=1)
    oc = eng.mccfr(Rc, iterations=IT, seed=SEED, ruleset=1)
    cl_it, cl_ms = int(oc["results"]["iterations"].sum()), oc["kernel_ms"]
    split = [a + b for a, b in zip(split, status_split(oc["results"]))]
    eng.close()
    # -- four times the roots in one call (the shared tree arena holds them: ~1 MB per 200-iteration tree): what the kernel does
    # when every warp slot stays busy to the end
    Rb = 4 * R
    eng = Engine(capacity=Rb, device=local)
    eng.make_roots(Rb, seed=SEED, first_gid=sharding.first_gid(3, rank, world, Rb), back_lo=0, back_hi=20)
    eng.mccfr(Rb, iterations=IT, seed=SEED)
    ob = eng.mccfr(Rb, iterations=IT, seed=SEED)
    big_it, big_ms = int(ob["results"]["iterations"].sum()), ob["kernel_ms"]
    split = [a + b for a, b in zip(split, status_split(ob["results"]))]
    eng.close()
    ints = [pure_it, deep_it, gen_it, gen_targets, e2e_it, cl_it] + split + [tc_it, big_it]
    floats = [pure_ms, deep_ms, gen_ms, t5 * 1e3, pure_wall * 1e3, deep_wall * 1e3, e2e_wall * 1e3, gen_wall * 1e3, cl_ms, tc_ms, big_ms]
    return ints, floats, out


DUMP_MAX_GAMES = 1 << 20      # 40 B per game written (winner, points[6], steps as float32, game id as float64): 40 MiB at most, plus headers


def dump_outputs(eng, out_dir, games, first_gid, ruleset, timed_stats):
    """Writes the last timed step of the headline figure as a caller of Engine.playout receives it, one float32 / float64 .npy
    per array, so that two builds can be compared output for output.  stats_*: the outcome statistics the timed call returned.
    winner, points, steps: per game, from one untimed replay of the same games with per-game outputs; the replay's statistics
    must equal the timed call's.  Above DUMP_MAX_GAMES games, a fixed seeded sample of the games is written (game_id says which)."""
    import numpy as np
    out = eng.playout(games, seed=SEED, first_gid=first_gid, ruleset=ruleset)
    if any(out["stats"][k] != timed_stats[k] for k in out["stats"]):
        raise SystemExit("bench.py: the replay of the last timed step differs from it: %r vs %r" % (out["stats"], timed_stats))
    idx = np.arange(games)
    if games > DUMP_MAX_GAMES:
        idx = np.sort(np.random.default_rng(SEED).choice(games, DUMP_MAX_GAMES, replace=False))
    arrays = {"game_id": (first_gid + idx).astype(np.float64), "winner": out["winner"][idx].astype(np.float32),
              "points": out["points"][idx].astype(np.float32), "steps": out["steps"][idx].astype(np.float32)}
    for k, v in out["stats"].items():
        arrays["stats_" + k] = np.atleast_1d(np.asarray(v, dtype=np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--games", type=int, default=1 << 20, help="games per GPU per step (weak); games in total (strong)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-games-per-core", type=int, default=60)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ruleset", type=int, default=0)
    ap.add_argument("--no-mccfr", action="store_true", help="skip the secondary MCCFR measurement")
    ap.add_argument("--no-classic", action="store_true", help="skip the classic-eight playout figure")
    ap.add_argument("--mccfr-roots", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last weak-scaling step computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the one JSON line and nothing else: library chatter written straight to fd 1 (NCCL prints its
    # version there under NCCL_DEBUG=VERSION) goes to stderr until the line is printed
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(_real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from citadels_self_play_b200 import Engine, sharding
    eng = Engine(capacity=1024, device=local)
    G = args.games
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def gid0(step):  # disjoint global ids per (step, rank)
        return sharding.first_gid(step, rank, world, G)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_playouts(games, first_gid_of, steps, ruleset):
        """K steps of `games` fused playouts on this rank.
        -> (wall s, kernel ms, env steps, errors, wins[6], launches, statistics of the last step)"""
        launches0 = eng.launches
        kernel_ms, env_steps, errors, wins = 0.0, 0, 0, [0] * 6
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            st = eng.playout(games, seed=SEED, first_gid=first_gid_of(k), ruleset=ruleset, outputs=False)["stats"]
            kernel_ms += st["kernel_ms"]
            env_steps += st["steps"]
            errors += st["errors"]
            wins = [a + b for a, b in zip(wins, st["wins"])]
        barrier()
        return time.perf_counter() - t0, kernel_ms, env_steps, errors, wins, eng.launches - launches0, st

    # warm-up (untimed)
    for w in range(args.warmup):
        flush.zero_()
        torch.cuda.synchronize()
        eng.playout(G, seed=SEED, first_gid=gid0(1000 + w), ruleset=args.ruleset, outputs=False)

    # ---- device-resident timing, weak scaling: K steps of G games per rank ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    wall, kernel_ms, env_steps, errors, wins, launches, last_stats = timed_playouts(G, gid0, args.steps, args.ruleset)

    # ---- strong scaling: the same K steps with G games in total, ceil(G / world) per rank ----
    Gs = (G + world - 1) // world
    s_wall, s_kernel_ms, s_steps, _, _, _, _ = timed_playouts(Gs, lambda k: (3000 + k) * G + rank * Gs, args.steps, args.ruleset)

    # ---- end-to-end through the public API with HOST buffers: every step copies G packed game records (256 B each) from
    # pinned host memory into the engine's slots (ctd_load_states), plays them to terminal (ctd_playout_slots) and reads
    # winner + step count of every game back to the host.  The records are made beforehand, untimed (two alternating sets).
    eng_h = Engine(capacity=G, device=local)
    host_sets = []
    for j in range(min(2, max(args.steps, 1))):
        buf = torch.empty((G, 256), dtype=torch.uint8, pin_memory=True).numpy()
        eng_h.reset(G, seed=SEED, first_gid=gid0(2000 + j), ruleset=args.ruleset)
        eng_h.store_states(G, out=buf)
        host_sets.append(buf)
    eng_h.load_states(host_sets[0])
    eng_h.playout_slots(G)                                   # warm-up of this path
    launches_h0 = eng_h.launches
    barrier()
    t1 = time.perf_counter()
    e2e_steps = 0
    for k in range(args.steps):
        eng_h.load_states(host_sets[k % len(host_sets)])      # H2D 256*G bytes
        w_host, s_host = eng_h.playout_slots(G)              # D2H 3*G bytes (int8 winner, uint16 steps per game)
        e2e_steps += int(s_host.sum(dtype="int64"))
    barrier()
    e2e_wall = time.perf_counter() - t1
    e2e_launches = eng_h.launches - launches_h0
    assert (w_host >= 0).all()
    eng_h.close()
    del host_sets
    clocks = sampler.stop() if rank == 0 else None

    # ---- the classic eight (Assassin Thief Magician King Bishop Merchant Architect Warlord -- north_star's list): one extra figure
    classic = None
    if not args.no_classic and args.ruleset == 0:
        eng.playout(G, seed=SEED, first_gid=gid0(5000), ruleset=1, outputs=False)
        c_wall, c_ms, c_steps, c_err, _, _, _ = timed_playouts(G, lambda k: gid0(5001 + k), 2, 1)
        classic = [c_wall, c_ms, c_steps, c_err]

    # ---- secondary metric: MCCFR iterations/s ----
    mccfr = None if args.no_mccfr else bench_mccfr(args, rank, world, local, torch)

    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs, G, gid0(args.steps - 1), args.ruleset, last_stats)

    # ---- the only collectives: outcome statistics and times, after the timed regions ----
    def reduce(vals, op, dtype):
        t = torch.tensor(vals, dtype=dtype, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=op)
        return t.tolist()

    wall, e2e_wall, kernel_ms, s_wall, s_kernel_ms = reduce([wall, e2e_wall, kernel_ms, s_wall, s_kernel_ms], dist.ReduceOp.MAX, torch.float64)
    tot = reduce([env_steps, e2e_steps, errors, launches, s_steps] + wins, dist.ReduceOp.SUM, torch.int64)
    env_steps, e2e_steps, errors, launches, s_steps = [int(x) for x in tot[:5]]
    wins = [int(x) for x in tot[5:]]
    if classic is not None:
        cw, cm = reduce(classic[:2], dist.ReduceOp.MAX, torch.float64)
        cs, ce = [int(x) for x in reduce(classic[2:], dist.ReduceOp.SUM, torch.int64)]
    if mccfr is not None:
        mi = [int(x) for x in reduce(mccfr[0], dist.ReduceOp.SUM, torch.int64)]
        mf = reduce(mccfr[1], dist.ReduceOp.MAX, torch.float64)

    if rank == 0:
        peak, peak_src = _peaks()
        value = env_steps / wall
        per_gpu_kernel = (env_steps / world) / (kernel_ms / 1e3)
        achieved = per_gpu_kernel * BYTES_PER_STEP / 1e9
        traffic, traffic_src = _traffic(G)
        line = {
            "metric": METRIC, "value": value, "unit": "env steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
            "device_ms_per_step": kernel_ms / max(args.steps, 1),   # CUDA events on the engine's stream around the kernel, max over ranks
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "%d %s 6-player games per GPU per step, dealt on device from Philox(seed, gid), "
                                   "uniform-random option to terminal (BASELINE configs[1])" % (G, RULESETS[args.ruleset]),
                       "ruleset": RULESETS[args.ruleset], "games_per_gpu_per_step": G,
                       "l2": "no HBM-resident inputs (games are generated on device); 256 MiB flush between iterations",
                       "parallelism": "games sharded by global id, %d rank(s), no step-path collective" % world},
            "strong": {"scaling": "strong", "games_total_per_step": Gs * world, "games_per_gpu_per_step": Gs,
                       "value": s_steps / s_wall, "unit": "env steps/s", "ms_per_step": 1e3 * s_wall / max(args.steps, 1),
                       "device_ms_per_step": s_kernel_ms / max(args.steps, 1),
                       "note": "BASELINE configs[1] as written: the same number of playouts in total, split over the ranks"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": "%s (ncu, bytes per launch)" % traffic_src,
                         "peak_source": peak_src,
                         "note": "algorithmic 512 B/env step (SURVEY 8(d)); the fused kernel keeps the game in shared "
                                 "memory for its ~420 steps, so the real limiter is the SM front end: instruction fetch / issue (see profiles/README.md)",
                         "kernel_env_steps_per_s_per_gpu": per_gpu_kernel},
            "e2e": {"value": e2e_steps / e2e_wall, "unit": "env steps/s", "h2d_bytes_per_step": 256 * G * world,
                    "d2h_bytes_per_step": 3 * G * world,
                    "path": "Engine.load_states (pinned host records -> HBM) + Engine.playout_slots (winner, steps -> host)"},
            "gpu_launches": launches, "gpu_launches_e2e": e2e_launches, "clocks": clocks,
            "outcomes": {"games": G * args.steps * world, "errors": errors, "wins": wins},
        }
        if classic is not None:
            line["classic"] = {"ruleset": "classic eight (Assassin Thief Magician King Bishop Merchant Architect Warlord)",
                               "value": cs / cw, "unit": "env steps/s", "kernel_env_steps_per_s_per_gpu": (cs / world) / (cm / 1e3),
                               "games_per_gpu_per_step": G, "steps": 2, "errors": ce}
        if mccfr is not None:
            R, R5 = args.mccfr_roots, max(64, args.mccfr_roots // 4)
            ex = mccfr[2]
            line["mccfr"] = {
                "unit": "MCCFR iterations/s (one iteration = one node-step, algorithms/deep_mccfr.py:194-204)",
                "roots_per_gpu": R, "iterations_per_root": 200, "root_step_back": "0..20",
                "pure_it_per_s": mi[0] / (mf[0] / 1e3), "deep_it_per_s": mi[1] / (mf[1] / 1e3),
                "pure_it_per_s_4x_roots": mi[11] / (mf[10] / 1e3), "roots_per_gpu_4x": 4 * R,
                "pure_it_per_s_wall": mi[0] / (mf[4] / 1e3), "deep_it_per_s_wall": mi[1] / (mf[5] / 1e3),
                "deep_vs_pure": (mi[1] / mf[1]) / (mi[0] / mf[0]), "deep_waves": ex["deep_waves"],
                "deep_mode": "fused: one launch, every warp evaluates the leaves of its own tree (fp32)",
                "deep_it_per_s_waves_tcgen05": mi[10] / (mf[9] / 1e3), "deep_waves_tcgen05": ex["deep_waves_tc"],
                "deep_max_depth": 10, "deep_model": "ValueOnlyNN(418,512), torch.manual_seed(0) init",
                "e2e": {"value": mi[4] / (mf[6] / 1e3), "unit": "iterations/s", "h2d_bytes_per_step": ex["e2e_h2d_bytes"] * world,
                        "d2h_bytes_per_step": ex["e2e_d2h_bytes"] * world,
                        "path": "Engine.load_roots (host records, knowledge blocks, used_cards, ids -> HBM) + Engine.mccfr (ctd_mccfr_result records -> host)"},
                "roofline_frac_hbm_2048B_per_it": (mi[0] / world / (mf[0] / 1e3)) * BYTES_PER_ITER / 1e9 / peak,
                "trees_by_status": {"device_memory_exhausted(2)": mi[6], "container_capacity(4)": mi[7], "reference_raises(16)": mi[8],
                                    "terminal_root(1)": mi[9]},
                "trees_with_error_status": mi[6] + mi[7] + mi[8],
                "datagen_2000it": {"roots_per_gpu": R5, "roots": "create_a_random_game(100)", "it_per_s": mi[2] / (mf[2] / 1e3),
                                   "it_per_s_wall": mi[2] / (mf[7] / 1e3), "targets": mi[3], "usefulness_threshold": 200,
                                   "targets_export_ms": mf[3]},
                "classic": {"roots_per_gpu": R, "pure_it_per_s": mi[5] / (mf[8] / 1e3)}}
            if not args.no_cpu_baseline:
                cores = os.cpu_count() or 1
                ci, cw_, kind = cpu_mccfr(6, cores)
                line["mccfr"]["cpu_baseline"] = {"value": ci / cw_, "unit": "iterations/s", "cores": cores, "kind": kind,
                                                 "sample": "%d roots x 200 iterations, run_utils.run_mccfr(game, max_iterations=200)" % (6 * cores)}
                dres = cpu_mccfr(6, cores, deep=True)
                if dres is not None:
                    line["mccfr"]["cpu_baseline_deep"] = {
                        "value": dres[0] / dres[1], "unit": "iterations/s", "cores": cores, "kind": dres[2],
                        "sample": "%d roots x 200 iterations, CFRNode(model=ValueOnlyNN(418,512), device='cpu').cfr_pred(200, 10)" % (6 * cores)}
                    line["mccfr"]["deep_vs_cpu_reference"] = line["mccfr"]["deep_it_per_s"] / (dres[0] / dres[1])
                if kind == "reference":
                    pi, pw, _ = cpu_mccfr(12, cores, kind="port")
                    line["mccfr"]["cpu_port"] = {"value": pi / pw, "unit": "iterations/s", "cores": cores, "kind": "port"}
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            per_core = 300   # ~10 s of work per core for the reference (13.6 k env steps/s/core): pool start-up and imports amortised
            cs_, cw_, kind = cpu_playouts(per_core, cores, ruleset=args.ruleset)
            line["cpu_baseline"] = {"value": cs_ / cw_, "unit": "env steps/s", "cores": cores, "kind": kind,
                                    "sample": "%d %s games (%d per core), %s" % (
                                        per_core * cores, RULESETS[args.ruleset], per_core,
                                        "the unmodified reference's loop run_utils.py:37-41 from oracle/_ref" if kind == "reference"
                                        else "oracle port of run_utils.py:37-41")}
            if kind == "reference":
                ps, pw, _ = cpu_playouts(per_core, cores, ruleset=args.ruleset, kind="port")
                line["cpu_port"] = {"value": ps / pw, "unit": "env steps/s", "cores": cores, "kind": "port"}
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
