"""The reference's evaluation harness (compare_to_random.py:8-37) on the engine.

Seat 0 decides with deep MCCFR (value model at depth 10, 200 iterations), seat 1 with pure MCCFR (2000 iterations),
seats 2-5 uniformly at random; forced moves (one legal option) are played without a search, as in the reference.

  play_games(sim_number, model)           the reference's loop, one game at a time through the facade (same calls, same
                                          order: get_options_from_state -> run_mccfr -> option.carry_out)
  play_games_batched(n_games, model)      the same experiment with every game advanced in lock-step: all games in which
                                          seat 0 (resp. seat 1) has a real choice are searched in ONE ctd_mccfr_pred
                                          (resp. ctd_mccfr) launch, one tree per game, and the live decision
                                          (CFRNode.action_choice(live=True), algorithms/deep_mccfr.py:67-75, with the
                                          role-preference quirk of game/game.py:312-317) is taken from the result records.
  play_arena(n_games, seats, model)       the experiment with any player on any seat (random_seat(), pure(it), deep(it,
                                          depth, weight, model=slot)), every game resident on the device from deal to end
                                          (ctd_arena): the host only loops over decision rounds.  Random seats draw from
                                          Philox stream 4 keyed by the game's step count, so results do not depend on batch
                                          sizes.  models=[...] loads one value model per slot, so deep seats can differ in model.
  head_to_head(n_games, model_a, model_b) two value models against each other: every deal is played twice, with a seat
                                          pattern and with A and B swapped, and the pairs are counted and sign-tested.

Every search of game g at decision number t runs on the Philox stream keyed (seed, g | t << 40), so successive decisions of
one game do not reuse draws.  There is no CPU path: games live in 256-byte records, every transition and every search
runs on the device.
"""
import math
import random

import numpy as np

from .engine import Engine, EngineError, DEFAULT_SEED, RULESET_PRESET
from .layout import KNOW_BYTES, SEAT_RANDOM, SEAT_PURE, SEAT_DEEP, MAX_VALUE_MODELS, SEAT_MODEL_SHIFT
from . import facade as F

Z99 = 2.5758293035489004


def play_games(sim_number, model=None, engine=None, seed=DEFAULT_SEED, first_gid=0, deep_iterations=200,
               pure_iterations=2000, rng=None):
    """compare_to_random.play_games (compare_to_random.py:8-37).  -> winners[6]."""
    rng = rng or random.Random(seed)
    winners = [0] * 6
    for s in range(sim_number):
        game = F.create_game(engine=engine, seed=seed, gid=first_gid + s)
        winner = False
        while not winner:
            pid = game.gamestate.player_id
            if pid == 0 and model is not None and len(game.get_options_from_state()) > 1:
                chosen, _ = F.run_mccfr(game, model, max_iterations=deep_iterations)
            elif pid == 1 and len(game.get_options_from_state()) > 1:
                chosen, _ = F.run_mccfr(game, max_iterations=pure_iterations)
            else:
                chosen = rng.choice(game.get_options_from_state())
            winner = chosen.carry_out(game)
        winners[winner.id] += 1
    return winners


def _live_choice(res, game, options, nprng=None):
    """CFRNode.action_choice(live=True) from one ctd_mccfr_result record: the kernel drew the decision from the tree's own
    chance stream right after the search (cumulative-strategy draw, or the role-preference quirk of game/game.py:312-317 at a
    role-pick root)."""
    d = int(res["live_option"])
    if d == 0:
        raise ValueError("a terminal root has no children (the reference raises ValueError here too)")
    return F.option(d, game)


def search_batch(engine, games, decision_no, model=None, iterations=2000, max_depth=10, weight=5.0):
    """One MCCFR tree per game, all in one launch.  -> ctd_mccfr_result records (numpy structured array)."""
    n = len(games)
    recs = np.stack([np.frombuffer(g._rec.tobytes(), dtype=np.uint8) for g in games])
    knows = np.stack([g._know[g.gamestate.player_id * KNOW_BYTES:(g.gamestate.player_id + 1) * KNOW_BYTES] for g in games])
    used = np.stack([g._used for g in games])
    gids = np.array([F.tree_gid(g.gid, t) for g, t in zip(games, decision_no)], dtype=np.uint64)
    engine.load_roots(recs, knows, used, gids)
    ruleset = int(games[0]._rec["ruleset"])
    seed = games[0].seed
    if model is None:
        out = engine.mccfr(n, iterations=iterations, seed=seed, ruleset=ruleset)
    else:
        engine.set_value_model(model)
        out = engine.mccfr_pred(n, iterations=iterations, max_depth=max_depth, seed=seed, ruleset=ruleset, weight=weight)
    res = out["results"]
    bad = res["status"] & ~np.uint32(1)
    if bad.any():
        raise EngineError("MCCFR status %d in a batched search (2 device memory exhausted, 4 container capacity, 16 the reference "
                          "raises for this root)" % int(bad.max()))
    return res


def play_games_batched(n_games, model=None, engine=None, seed=DEFAULT_SEED, first_gid=0, deep_iterations=200,
                       pure_iterations=2000, max_depth=10, rng=None, ruleset=RULESET_PRESET, stats=None):
    """The arena experiment over `n_games` games advanced in lock-step.  -> winners[6].
    `stats` (optional dict) receives the number of searches and launches."""
    rng = rng or random.Random(seed)
    nprng = np.random.default_rng(seed & 0xFFFFFFFF)
    step_engine = engine or F.default_engine()
    search_engine = Engine(capacity=max(1, n_games), device=step_engine.device)
    games = [F.create_game(engine=step_engine, seed=seed, gid=first_gid + i, ruleset=ruleset) for i in range(n_games)]
    decisions = [0] * n_games
    winners = [0] * 6
    live = list(range(n_games))
    n_search = [0, 0]
    try:
        while live:
            options = {i: games[i].get_options_from_state() for i in live}
            chosen = {}
            for seat, its, mdl in ((0, deep_iterations, model), (1, pure_iterations, None)):
                if seat == 0 and model is None:
                    continue
                idx = [i for i in live if games[i].gamestate.player_id == seat and len(options[i]) > 1]
                if not idx:
                    continue
                res = search_batch(search_engine, [games[i] for i in idx], [decisions[i] for i in idx], mdl, its, max_depth)
                n_search[seat] += len(idx)
                for i, r in zip(idx, res):
                    chosen[i] = _live_choice(r, games[i], options[i], nprng)
                    decisions[i] += 1
            nxt = []
            for i in live:
                opt = chosen[i] if i in chosen else rng.choice(options[i])
                winner = opt.carry_out(games[i])
                if winner:
                    winners[winner.id] += 1
                else:
                    nxt.append(i)
            live = nxt
    finally:
        if stats is not None:
            stats.update(deep_searches=n_search[0], pure_searches=n_search[1], search_launches=search_engine.launches)
        search_engine.close()
    return winners


def random_seat():
    """A seat on random.choice (compare_to_random.py:31)."""
    return (SEAT_RANDOM, 0, 0, 0.0)


def pure(iterations):
    """A seat on run_mccfr(game, max_iterations=iterations): cfr_train."""
    return (SEAT_PURE, int(iterations), 0, 0.0)


def deep(iterations, max_depth=10, weight=5.0, model=0):
    """A seat on run_mccfr(game, model, max_iterations=iterations): cfr_pred(iterations, max_depth) with the value model in the
    engine's slot `model` (CTD_SEAT_DEEP_MODEL)."""
    return (SEAT_DEEP | (int(model) << SEAT_MODEL_SHIFT), int(iterations), int(max_depth), float(weight))


def _seat_kind(kind):
    return int(kind) & 0xFF


def _seat_model(kind):
    return (int(kind) >> SEAT_MODEL_SHIFT) & 0xFF


def default_seats():
    """compare_to_random.py's layout: seat 0 deep(200, depth 10), seat 1 pure(2000), seats 2-5 random."""
    return [deep(200, 10, 5.0), pure(2000)] + [random_seat()] * 4


def rank_block(n_games, rank, world):
    """(first game, number of games) of rank `rank` out of `world`: contiguous blocks of ceil(n_games / world) games."""
    from . import sharding
    per = -(-int(n_games) // int(world))
    first = min(int(n_games), sharding.first_gid(0, rank, world, per))
    return first, min(int(n_games), first + per) - first


def arena_models(seats, model, models, engine):
    """The value models of play_arena's model= / models= as a list for slots 0, 1, ...; ValueError when both are given, when there are
    more than an engine holds, or (without `engine`, whose slots may already be loaded) when a deep seat's slot is not among them."""
    if model is not None:
        if models is not None:
            raise ValueError("pass model= or models=, not both")
        models = [model]
    models = [] if models is None else list(models)
    if len(models) > MAX_VALUE_MODELS:
        raise ValueError("an engine holds %d value models, got %d" % (MAX_VALUE_MODELS, len(models)))
    missing = sorted({_seat_model(s[0]) for s in seats if _seat_kind(s[0]) == SEAT_DEEP} - set(range(len(models))))
    if missing and engine is None:
        raise ValueError("deep seats on value-model slots %s, but models= fills slots [0, %d)" % (missing, len(models)))
    return models


def play_arena(n_games, seats=None, model=None, engine=None, seed=DEFAULT_SEED, first_gid=0, ruleset=RULESET_PRESET,
               max_steps=4096, group=None, models=None, record=None):
    """compare_to_random.play_games with a player per seat, every game on the device (Engine.arena).  Under torch.distributed
    each rank plays its own block of game ids (sharding.first_gid over rank_block's split) and the statistics are summed.
    Without `engine` the games run on torch's current CUDA device (under torchrun: the rank's own GPU after
    torch.cuda.set_device(LOCAL_RANK)); the statistics are reduced on the engine's device.
    models: value models loaded into slots 0 .. len(models) - 1, for the seats deep(..., model=slot); `model` is short for
    models=[model].  Without `engine` every deep seat's slot must be among them.
    record: Engine.arena's recording spec, appending to `engine`'s dataset (selfplay.record_arena).
    -> dict(winners[6] and stats over all ranks; this rank's local_stats, first_gid of its games, their per-game arrays
    winner / points / steps / searches and its phase_ms)."""
    import torch
    import torch.distributed as dist
    from . import sharding
    seats = default_seats() if seats is None else list(seats)
    models = arena_models(seats, model, models, engine)
    dist_on = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank(group) if dist_on else 0
    world = dist.get_world_size(group) if dist_on else 1
    first, count = rank_block(n_games, rank, world)
    own = engine is None
    eng = engine or Engine(capacity=max(1, min(count, 8192)), 
                            device=torch.cuda.current_device() if torch.cuda.is_available() else 0)
    try:
        for slot, m in enumerate(models):
            eng.set_value_model(m, slot=slot)
        out = eng.arena(count, seats, seed=seed, first_gid=first_gid + first, ruleset=ruleset, max_steps=max_steps, record=record)
    finally:
        if own:
            eng.close()
    local = out["stats"]
    dev = "cuda:%d" % eng.device if dist_on and dist.get_backend(group) == "nccl" else "cpu"
    stats = sharding.reduce_stats(local, dev, group=group)
    stats["max_steps"] = int(sharding.reduce_max([local["max_steps"]], dev, group=group)[0])
    out.update(winners=list(stats["wins"]), stats=stats, local_stats=local, first_gid=first_gid + first)
    return out


def wilson(k, n, z=Z99):
    """Wilson score interval of k successes in n trials (default 99 %)."""
    if n == 0:
        return [0.0, 1.0]
    p = k / n
    c = (p + z * z / (2 * n)) / (1 + z * z / n)
    h = z * math.sqrt(p * (1 - p) / n + z * z / (4 * n * n)) / (1 + z * z / n)
    return [max(0.0, c - h), min(1.0, c + h)]


PAIR_KEYS = ("a_both", "b_both", "split", "random", "error")


def swap_pattern(pattern):
    """The seat pattern with A and B exchanged (R, a random seat, stays)."""
    return pattern.translate(str.maketrans("AB", "BA"))


def pair_counts(pattern, winner_ab, winner_ba):
    """Game i was played twice on the same deal: with seat pattern `pattern` (winning seat winner_ab[i]) and with A and B swapped
    (winner_ba[i]); -1 is an errored game.  -> dict of pair counts: a_both (A's seats won both games), b_both, split (A won one,
    B the other), random (a random seat won at least one, neither errored) and error (either game errored)."""
    w = [np.asarray(x, dtype=np.int64) for x in (winner_ab, winner_ba)]
    if w[0].shape != w[1].shape:
        raise ValueError("the two passes have %d and %d games" % (w[0].size, w[1].size))
    # the side of each winning seat, E for an error (index 6)
    side = [np.array(list(p) + ["E"])[np.where(x < 0, 6, x)] for p, x in zip((pattern, swap_pattern(pattern)), w)]
    err = (side[0] == "E") | (side[1] == "E")
    a_both = ~err & (side[0] == "A") & (side[1] == "A")
    b_both = ~err & (side[0] == "B") & (side[1] == "B")
    rnd = ~err & ((side[0] == "R") | (side[1] == "R"))
    split = ~err & ~rnd & ~a_both & ~b_both
    return dict(zip(PAIR_KEYS, (int(x.sum()) for x in (a_both, b_both, split, rnd, err))))


def head_to_head(n_games, model_a, model_b, player=deep(200, 10, 5.0), pattern="ABABAB", engine=None, seed=DEFAULT_SEED,
                 first_gid=0, ruleset=RULESET_PRESET, max_steps=4096, group=None):
    """Value model A against value model B: games (seed, first_gid + i) for i < n_games, each played twice through play_arena
    (models=[model_a, model_b]), once with `pattern` (seat s: A, B or R for a random seat) and once with A and B swapped, so
    that the luck of the deal and of the seats cancels.  A's and B's seats play `player` (a deep() seat) on their own model.
    Under torch.distributed both passes split the games over the ranks alike, each rank pairs its own games and the counts are
    summed.
    -> dict(games (pairs), errors (games), a / b: wins, share of the decided games and its Wilson 99 % interval, random_wins,
    seats and seat_wins of each pass, pairs (pair_counts over all ranks), sign_test (two-sided binomial test of a_both against b_both),
    passes (the two play_arena results))."""
    import torch
    import torch.distributed as dist
    from scipy.stats import binomtest
    from . import sharding
    pattern = str(pattern)
    if len(pattern) != 6 or set(pattern) - set("ABR") or "A" not in pattern or "B" not in pattern:
        raise ValueError("pattern: six seats of A, B or R with at least one A and one B, got %r" % (pattern,))
    kind, its, depth, weight = player
    if _seat_kind(kind) != SEAT_DEEP:
        raise ValueError("player must be a deep() seat")
    swapped = swap_pattern(pattern)

    def seats(p):
        return [deep(its, depth, weight, model="AB".index(c)) if c in "AB" else random_seat() for c in p]
    pass_seats = [seats(pattern), seats(swapped)]
    passes = [play_arena(n_games, s, engine=engine, seed=seed, first_gid=first_gid, ruleset=ruleset, max_steps=max_steps, group=group,
                         models=[model_a, model_b]) for s in pass_seats]
    dist_on = dist.is_available() and dist.is_initialized()
    dev = "cpu"
    if dist_on and dist.get_backend(group) == "nccl":
        dev = "cuda:%d" % (engine.device if engine is not None else torch.cuda.current_device())
    local = pair_counts(pattern, passes[0]["winner"], passes[1]["winner"])
    pairs = dict(zip(PAIR_KEYS, sharding.reduce_sum([local[k] for k in PAIR_KEYS], dev, group=group)))
    st = [r["stats"] for r in passes]
    wins = {c: sum(s["wins"][i] for s, p in zip(st, (pattern, swapped)) for i in range(6) if p[i] == c) for c in "ABR"}
    decided = sum(s["games"] - s["errors"] for s in st)
    n_sign = pairs["a_both"] + pairs["b_both"]
    p_value = float(binomtest(pairs["a_both"], n_sign, 0.5, alternative="two-sided").pvalue) if n_sign else 1.0
    side = {c: dict(wins=wins[c], share=wins[c] / decided if decided else 0.0, wilson99=wilson(wins[c], decided)) for c in "AB"}
    return dict(pattern=pattern, swapped=swapped, games=st[0]["games"], errors=st[0]["errors"] + st[1]["errors"], a=side["A"],
                b=side["B"], random_wins=wins["R"], seats=[[list(x) for x in s] for s in pass_seats], seat_wins=[s["wins"] for s in st],
                pairs=pairs, sign_test=dict(a_both=pairs["a_both"], b_both=pairs["b_both"], p_value=p_value), passes=passes)
