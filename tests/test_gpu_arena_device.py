"""ctd_arena (Engine.arena / arena.play_arena): every game resident on the device from deal to end, a player per seat.
Checked against the same experiment played through the facade one game and one search at a time."""
import os

import numpy as np
import pytest

from tests.golden_util import GOLDEN

pytestmark = pytest.mark.gpu

SEED = 0xA4E7A5


def _checkpoint():
    from tests.test_value_checkpoint import load
    return load()[1]


def _pick(seed, gid, s, n):
    """The random seats' draw: word s & 3 of Philox block (s >> 2, stream 4, gid), k = (u * n) >> 32."""
    from oracle.philox import philox4x32_10, MASK
    from citadels_self_play_b200.layout import ARENA_STREAM
    r = philox4x32_10(s >> 2, ARENA_STREAM, gid & MASK, gid >> 32, seed & MASK, (seed >> 32) & MASK)
    return (r[s & 3] * n) >> 32


def _mirror(seed, gid, ruleset, seats, model, search_engine, max_steps=4096):
    """compare_to_random.play_games for one game through the facade: one enumeration per step, a search (decision number t of
    the game, tree id facade.tree_gid(gid, t)) when a search seat has >= 2 options, else the stream-4 pick."""
    from citadels_self_play_b200 import arena, facade as F
    from citadels_self_play_b200.layout import SEAT_RANDOM, SEAT_DEEP
    g = F.create_game(seed=seed, gid=gid, ruleset=ruleset)
    t = 0
    while not g.terminal and int(g._rec["steps"]) < max_steps:
        s = int(g._rec["steps"])
        opts = g.get_options_from_state()
        kind, its, depth, weight = seats[g.gamestate.player_id]
        if kind != SEAT_RANDOM and len(opts) >= 2:
            res = arena.search_batch(search_engine, [g], [t], model if kind == SEAT_DEEP else None, its, depth, weight)
            t += 1
            chosen = arena._live_choice(res[0], g, opts)
        else:
            chosen = opts[_pick(seed, gid, s, len(opts))]
        chosen.carry_out(g)
    return g, t


@pytest.mark.parametrize("ruleset,n_games,with_deep", [(0, 8, True), (1, 2, False), (2, 2, False)])
def test_arena_equals_the_facade_mirror(ruleset, n_games, with_deep):
    """Terminal records (bytes [0, 228)), winners, points, steps and searches per game, exactly."""
    from citadels_self_play_b200 import Engine, arena
    model = _checkpoint() if with_deep else None
    seat0 = arena.deep(20, 10, 5.0) if with_deep else arena.pure(40)
    seats = [seat0, arena.pure(40), arena.random_seat(), arena.random_seat(), arena.pure(40), arena.random_seat()]
    first_gid = 700 + 100 * ruleset
    eng, se = Engine(capacity=16), Engine(capacity=4)
    try:
        if model is not None:
            eng.set_value_model(model)
        out = eng.arena(n_games, seats, seed=SEED, first_gid=first_gid, ruleset=ruleset)
        finals = eng.store_states(n_games)
        for i in range(n_games):
            g, t = _mirror(SEED, first_gid + i, ruleset, seats, model, se)
            assert finals[i, :228].tobytes() == g._rec.tobytes()[:228], (ruleset, i)
            assert int(out["winner"][i]) == int(g._rec["winner"]), (ruleset, i)
            assert [int(x) for x in out["points"][i]] == g.points, (ruleset, i)
            assert int(out["steps"][i]) == int(g._rec["steps"]), (ruleset, i)
            assert int(out["searches"][i]) == t, (ruleset, i)
        st = out["stats"]
        assert st["games"] == n_games and st["errors"] == 0 and sum(st["wins"]) == n_games
        assert st["steps"] == int(out["steps"].astype(np.int64).sum())
        assert out["searches"].min() > 0
    finally:
        eng.close()
        se.close()


def test_arena_does_not_depend_on_capacity_or_batching():
    from citadels_self_play_b200 import Engine, arena
    seats = [arena.pure(30), arena.random_seat(), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.pure(20)]
    big, small = Engine(capacity=64), Engine(capacity=3)
    try:
        a = big.arena(16, seats, seed=SEED, first_gid=5000)
        b = small.arena(16, seats, seed=SEED, first_gid=5000)
        c1 = big.arena(8, seats, seed=SEED, first_gid=5000)
        c2 = big.arena(8, seats, seed=SEED, first_gid=5008)
    finally:
        big.close()
        small.close()
    for k in ("winner", "points", "steps", "searches"):
        assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(a[k], np.concatenate([c1[k], c2[k]])), k
    assert a["stats"] == b["stats"]
    assert a["stats"]["wins"] == [x + y for x, y in zip(c1["stats"]["wins"], c2["stats"]["wins"])]
    assert a["stats"]["errors"] == 0


def test_random_arena_matches_the_reference_outcome_distribution():
    """Six random seats over 2^14 preset games against the unmodified reference's games (tests/golden/ref_outcomes_preset.npz),
    with the gates of test_gpu_parity.test_distribution_vs_reference_sample: chi-square (5 dof, 99 %) on the winners, |z| < 3.2 on
    the mean points of every seat and on the mean game length."""
    from citadels_self_play_b200 import Engine, arena
    ref = np.load(os.path.join(GOLDEN, "ref_outcomes_preset.npz"))
    n = 1 << 14
    e = Engine(capacity=64)
    try:
        out = e.arena(n, [arena.random_seat()] * 6, seed=2024, first_gid=0)
    finally:
        e.close()
    st = out["stats"]
    assert st["games"] == n and st["errors"] == 0 and int(out["searches"].max()) == 0
    rw = np.bincount(ref["winner"], minlength=6).astype(np.float64)
    gw = np.asarray(st["wins"], dtype=np.float64)
    nr, ng = rw.sum(), gw.sum()
    pooled = (rw + gw) / (nr + ng)
    chi2 = (((rw - nr * pooled) ** 2) / (nr * pooled)).sum() + (((gw - ng * pooled) ** 2) / (ng * pooled)).sum()
    assert chi2 < 15.09, ("winner distribution", chi2, rw / nr, gw / ng)
    rp, gp = ref["points"].astype(np.float64), out["points"].astype(np.float64)
    z = (gp.mean(0) - rp.mean(0)) / np.sqrt(gp.var(0) / ng + rp.var(0) / nr)
    assert np.all(np.abs(z) < 3.2), ("mean points", z)
    rs, gs = ref["steps"].astype(np.float64), out["steps"].astype(np.float64)
    zs = (gs.mean() - rs.mean()) / np.sqrt(gs.var() / ng + rs.var() / nr)
    assert abs(zs) < 3.2, ("steps", gs.mean(), rs.mean(), zs)


def test_arena_launches_follow_decision_rounds_not_steps():
    from citadels_self_play_b200 import Engine, arena
    e = Engine(capacity=256)
    try:
        l0 = e.launches
        out = e.arena(256, [arena.random_seat()] * 6, seed=SEED, first_gid=0)
        assert e.launches - l0 <= 4
        assert out["stats"]["steps"] > 256 * 200
        seats = [arena.pure(20), arena.random_seat(), arena.pure(20)] + [arena.random_seat()] * 3   # one search group
        l0 = e.launches
        out = e.arena(64, seats, seed=SEED, first_gid=0)
        rounds = int(out["searches"].max()) + 1
        # per round: advance, gather, the search (a retry pass when a tree outgrows the shared arena), apply; plus deal and final
        assert e.launches - l0 <= 5 * rounds + 2, (e.launches - l0, rounds)
        assert e.launches - l0 < out["stats"]["steps"] / 20
    finally:
        e.close()


def test_arena_edge_cases():
    from citadels_self_play_b200 import Engine, EngineError, arena
    from citadels_self_play_b200.layout import STATE_DTYPE
    rnd = [arena.random_seat()] * 6
    e = Engine(capacity=16)
    try:
        out = e.arena(0, rnd)
        assert out["stats"]["games"] == 0 and len(out["winner"]) == 0
        bad = [[(3, 10, 0, 0.0)] + rnd[1:],                  # no such seat kind
               [arena.pure(0)] + rnd[1:],                     # a search seat without iterations
               [arena.deep(20, 10, 5.0)] + rnd[1:]]           # deep seat, but this engine has no value model
        for seats in bad:
            with pytest.raises(EngineError, match="status 1 "):
                e.arena(4, seats)
        with pytest.raises(EngineError, match="status 1 "):
            e.arena(4, rnd, ruleset=3)
        with pytest.raises(EngineError, match="status 1 "):   # beyond the range of the record's steps field
            e.arena(4, [arena.pure(10)] + rnd[1:], max_steps=65536)
        out = e.arena(2, rnd, seed=SEED, first_gid=0, max_steps=65535)
        assert out["stats"]["errors"] == 0 and sum(out["stats"]["wins"]) == 2
        out = e.arena(16, rnd, seed=SEED, first_gid=0, max_steps=20)
        assert (out["winner"] == -1).all() and (out["steps"] == 20).all()
        assert out["stats"]["errors"] == 16 and sum(out["stats"]["wins"]) == 0
        finals = e.store_states(16).view(STATE_DTYPE).reshape(16)
        assert (finals["err"] == 16).all()
    finally:
        e.close()


def test_play_arena_single_process():
    """play_arena without torch.distributed: one rank plays every game; its winners are the engine call's."""
    from citadels_self_play_b200 import Engine, arena
    seats = [arena.random_seat(), arena.pure(20)] + [arena.random_seat()] * 4
    out = arena.play_arena(12, seats=seats, seed=SEED, first_gid=40)
    e = Engine(capacity=32)
    try:
        direct = e.arena(12, seats, seed=SEED, first_gid=40)
    finally:
        e.close()
    assert out["first_gid"] == 40 and np.array_equal(out["winner"], direct["winner"])
    assert out["winners"] == direct["stats"]["wins"] and sum(out["winners"]) == 12
    assert out["stats"]["games"] == 12 and out["stats"]["max_steps"] == int(direct["steps"].max())
