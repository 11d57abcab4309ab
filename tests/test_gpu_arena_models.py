"""Value-model slots in the device arena: deep seats on different models in one ctd_arena call, checked against the same games
played through the facade with each seat searching on its own model; slot independence; arena.head_to_head."""
import numpy as np
import pytest

from tests.test_gpu_arena_device import _pick

pytestmark = pytest.mark.gpu

SEED = 0x5107A5


def _model_a():
    """the reference's trained checkpoint"""
    from tests.test_value_checkpoint import load
    return load()[1]


def _init_model(seed):
    import torch
    from citadels_self_play_b200.value_model import ValueOnlyNN
    torch.manual_seed(seed)
    return ValueOnlyNN(418, 512).eval()


def _mirror(seed, gid, ruleset, seats, models, search_engine, max_steps=4096):
    """compare_to_random.play_games for one game through the facade, a deep seat searching with models[its slot]: a search
    (decision number t of the game) when a search seat has >= 2 options, else the stream-4 pick."""
    from citadels_self_play_b200 import arena, facade as F
    from citadels_self_play_b200.layout import SEAT_RANDOM, SEAT_DEEP
    g = F.create_game(seed=seed, gid=gid, ruleset=ruleset)
    t = 0
    while not g.terminal and int(g._rec["steps"]) < max_steps:
        s = int(g._rec["steps"])
        opts = g.get_options_from_state()
        kind, its, depth, weight = seats[g.gamestate.player_id]
        if arena._seat_kind(kind) != SEAT_RANDOM and len(opts) >= 2:
            model = models[arena._seat_model(kind)] if arena._seat_kind(kind) == SEAT_DEEP else None
            res = arena.search_batch(search_engine, [g], [t], model, its, depth, weight)
            t += 1
            chosen = arena._live_choice(res[0], g, opts)
        else:
            chosen = opts[_pick(seed, gid, s, len(opts))]
        chosen.carry_out(g)
    return g, t


def _same_games(x, y):
    return all(np.array_equal(x[k], y[k]) for k in ("winner", "points", "steps", "searches"))


@pytest.mark.parametrize("backend", ["fused", "fp32", "tcgen05"])
def test_two_models_equal_the_facade(backend):
    """Terminal records (bytes [0, 228)), winners, points, steps and searches per game, exactly; and the games change when B is
    replaced by A, so the comparison can tell the two models apart."""
    from citadels_self_play_b200 import Engine, arena
    A, B = _model_a(), _init_model(7)
    seats = [arena.deep(20, 10, 5.0, model=0), arena.deep(20, 10, 5.0, model=1), arena.random_seat(),
             arena.deep(20, 10, 5.0, model=1), arena.pure(40), arena.random_seat()]
    n, first_gid = 6, 900
    eng, se = Engine(capacity=16), Engine(capacity=4)
    try:
        eng.set_value_backend(backend)
        se.set_value_backend(backend)
        eng.set_value_model(A, slot=0)
        eng.set_value_model(B, slot=1)
        out = eng.arena(n, seats, seed=SEED, first_gid=first_gid)
        finals = eng.store_states(n)
        for i in range(n):
            g, t = _mirror(SEED, first_gid + i, 0, seats, [A, B], se)
            assert finals[i, :228].tobytes() == g._rec.tobytes()[:228], (backend, i)
            assert int(out["winner"][i]) == int(g._rec["winner"]), (backend, i)
            assert [int(x) for x in out["points"][i]] == g.points, (backend, i)
            assert int(out["steps"][i]) == int(g._rec["steps"]), (backend, i)
            assert int(out["searches"][i]) == t, (backend, i)
        assert out["stats"]["errors"] == 0 and sum(out["stats"]["wins"]) == n
        eng.set_value_model(A, slot=1)
        same = eng.arena(n, seats, seed=SEED, first_gid=first_gid)
        assert not (_same_games(out, same) and np.array_equal(finals, eng.store_states(n))), backend
    finally:
        eng.close()
        se.close()


def test_a_slot_is_just_a_slot():
    from citadels_self_play_b200 import Engine, arena
    A = _model_a()

    def seats(k):
        return [arena.deep(20, 10, 5.0, model=k), arena.random_seat(), arena.pure(30), arena.deep(20, 10, 5.0, model=k),
                arena.random_seat(), arena.random_seat()]
    e = Engine(capacity=16)
    try:
        e.set_value_model(A, slot=0)
        e.set_value_model(A, slot=3)
        on0 = e.arena(8, seats(0), seed=SEED, first_gid=300)
        rec0 = e.store_states(8)
        on3 = e.arena(8, seats(3), seed=SEED, first_gid=300)
        rec3 = e.store_states(8)
    finally:
        e.close()
    assert _same_games(on0, on3) and np.array_equal(rec0, rec3) and on0["stats"] == on3["stats"]
    assert on0["searches"].min() > 0


@pytest.mark.parametrize("backend", ["fused", "tcgen05"])
def test_reloading_one_slot_leaves_the_others(backend):
    from citadels_self_play_b200 import Engine, arena
    A, B, C = _model_a(), _init_model(7), _init_model(11)

    def seats(k):
        return [arena.deep(20, 10, 5.0, model=k), arena.random_seat(), arena.deep(20, 10, 5.0, model=k)] + [arena.random_seat()] * 3
    e, fresh = Engine(capacity=16), Engine(capacity=16)
    try:
        for x in (e, fresh):
            x.set_value_backend(backend)
        e.set_value_model(A, slot=0)
        e.set_value_model(B, slot=1)
        before = e.arena(6, seats(0), seed=SEED, first_gid=400)
        e.set_value_model(C, slot=1)
        after = e.arena(6, seats(0), seed=SEED, first_gid=400)
        on_c = e.arena(6, seats(1), seed=SEED, first_gid=400)
        fresh.set_value_model(C)
        want_c = fresh.arena(6, seats(0), seed=SEED, first_gid=400)
    finally:
        e.close()
        fresh.close()
    assert _same_games(before, after) and before["stats"] == after["stats"]
    assert _same_games(on_c, want_c)


def test_head_to_head_of_a_model_with_itself_is_symmetric():
    from citadels_self_play_b200 import arena
    A = _model_a()
    n = 6
    r = arena.head_to_head(n, A, A, player=arena.deep(20, 10, 5.0), seed=SEED, first_gid=1200)
    p, q = r["passes"]
    for k in ("winner", "points", "steps", "searches"):
        assert np.array_equal(p[k], q[k]), k
    assert r["games"] == n and r["errors"] == 0
    assert r["pairs"] == dict(a_both=0, b_both=0, split=n, random=0, error=0)
    assert r["a"]["share"] == 0.5 and r["b"]["share"] == 0.5 and r["a"]["wins"] == r["b"]["wins"] == n
    assert r["sign_test"]["p_value"] == 1.0


def test_head_to_head_counts_are_consistent():
    from citadels_self_play_b200 import arena
    A, B = _model_a(), _init_model(7)
    n = 6
    r = arena.head_to_head(n, A, B, player=arena.deep(20, 10, 5.0), pattern="ABRBAR", seed=SEED, first_gid=1300)
    assert r["games"] == n and sum(r["pairs"].values()) == n
    assert r["pairs"] == arena.pair_counts("ABRBAR", r["passes"][0]["winner"], r["passes"][1]["winner"])
    assert r["seat_wins"] == [x["stats"]["wins"] for x in r["passes"]]
    w1, w2 = r["seat_wins"]
    assert r["a"]["wins"] == w1[0] + w1[4] + w2[1] + w2[3]
    assert r["b"]["wins"] == w1[1] + w1[3] + w2[0] + w2[4]
    assert r["random_wins"] == w1[2] + w1[5] + w2[2] + w2[5]
    decided = 2 * n - r["errors"]
    assert r["a"]["wins"] + r["b"]["wins"] + r["random_wins"] == decided
    assert r["a"]["share"] == r["a"]["wins"] / decided
    lo, hi = r["a"]["wilson99"]
    assert 0.0 <= lo <= r["a"]["share"] <= hi <= 1.0
    assert 0.0 <= r["sign_test"]["p_value"] <= 1.0


def test_model_slot_edge_cases():
    from citadels_self_play_b200 import Engine, EngineError, arena
    from citadels_self_play_b200.layout import SEAT_DEEP, SEAT_PURE, SEAT_RANDOM
    A = _model_a()
    rnd = [arena.random_seat()] * 5
    e = Engine(capacity=16)
    try:
        for slot in (6, -1):
            with pytest.raises(EngineError, match="status 1 "):
                e.set_value_model(A, slot=slot)
        e.set_value_model(A, slot=1)
        # slot 0 is empty: the single-model entry points and a plain deep seat fail as on an engine without a model
        e.make_roots(2, seed=SEED, first_gid=0)
        with pytest.raises(EngineError, match="status 1 "):
            e.mccfr_pred(2, iterations=10, max_depth=2, seed=SEED)
        with pytest.raises(EngineError, match="status 1 "):
            e.value_eval(np.zeros((2, 418), dtype=np.float32))
        bad = [[arena.deep(10)] + rnd,                              # slot 0 holds no model
               [arena.deep(10, model=2)] + rnd,                     # nor does slot 2
               [arena.deep(10, model=6)] + rnd,                     # no such slot
               [(SEAT_PURE | (1 << 8), 10, 0, 0.0)] + rnd,          # model bits on a pure seat
               [(SEAT_RANDOM | (1 << 8), 0, 0, 0.0)] + rnd,         # ... on a random seat
               [(SEAT_DEEP | (1 << 8) | (1 << 16), 10, 2, 5.0)] + rnd,   # a bit above 15
               [(-1, 10, 2, 5.0)] + rnd]
        for seats in bad:
            with pytest.raises(EngineError, match="status 1 "):
                e.arena(4, seats)
        out = e.arena(2, [arena.deep(10, 2, 5.0, model=1)] + rnd, seed=SEED, first_gid=0)
        assert out["stats"]["errors"] == 0 and sum(out["stats"]["wins"]) == 2
    finally:
        e.close()


def test_two_model_groups_launch_per_round_not_per_step():
    from citadels_self_play_b200 import Engine, arena
    e = Engine(capacity=256)
    try:
        e.set_value_model(_model_a(), slot=0)
        e.set_value_model(_init_model(7), slot=1)
        seats = [arena.deep(20, 10, 5.0, model=0), arena.random_seat(), arena.deep(20, 10, 5.0, model=1)] + [arena.random_seat()] * 3
        l0 = e.launches
        out = e.arena(64, seats, seed=SEED, first_gid=0)
        rounds, groups = int(out["searches"].max()) + 1, 2
        # per round: advance, and per group gather, the search (a retry pass when a tree outgrows the shared arena), apply;
        # plus deal and final
        assert e.launches - l0 <= 5 * rounds * groups + 2, (e.launches - l0, rounds)
        assert e.launches - l0 < out["stats"]["steps"] / 20
        assert out["stats"]["errors"] == 0
    finally:
        e.close()
