"""The fused playout kernels (ctd_playout.cuh: one game per thread, every thread pulling game ids until none are left) against
the Python oracle, bit-exact, where the kernel's own mechanisms are at work: a thread's second and later games (its CtdWork
re-initialised), ragged and boundary launches, every outcome counter against the per-game rows, records continued from the
middle of their games (ctd_playout_slots), and the host's choice of the preset- / classic-specialised or generic kernel for
continued records (the slots_rs run that ctd_reset, ctd_load_states, ctd_states_dev, ctd_make_roots and ctd_load_roots keep).

The oracle runs on the host cores in one spawn pool per module (not fork: this process holds a CUDA context); its results are
memoised, since several tests compare the same games."""
import multiprocessing as mp
import os
import numpy as np
import pytest

from citadels_self_play_b200.layout import STATE_DTYPE
from tests.golden_util import visible

CAP = 4096                  # Engine.playout / playout_slots default max_steps
MAXSTEPS_FLAG = 16          # CTD_ERR_MAXSTEPS in ctd_state.err (byte 228)
OVERFLOW_FLAG = 1           # CTD_ERR_OVERFLOW: ctd_pack saturated a field, e.g. a score past 127
N_BIG = 1 << 20             # bench.py's batch
BIG_SEED, BIG_GID0 = 0x5EED1A7E, 11 << 32
BUILD_SEED, CONT_SEED = 0xB01D, 0xC0471       # mid-game records are built under one seed and continued under another
STOPS = (0, 40, 150, 400)   # env steps the mid-game batches are played before they are stored
PER_STOP, N_TERMINAL = 256, 64


# ---------------------------------------------------------------------------------------------------- oracle
def oracle_continue(rec, seed, max_steps=CAP):
    """Finish a packed record in the oracle as ctd_playout_slots does: chance keyed by (seed, the record's gid) from the record's
    draw counter, the random-playout loop (run_utils.py:37-41) for at most max_steps steps counted from the record.
    -> (winner, points[6], steps taken, final pack(), final draw counter)."""
    from oracle import citadels_oracle as O
    from oracle.philox import PhiloxChance
    rec = bytes(rec)
    r = np.frombuffer(rec, dtype=STATE_DTYPE)[0]
    chance = PhiloxChance(seed, int(r["gid"]))
    chance.i = int(r["rng_draws"])
    g = O.Game.unpack(rec, chance)
    steps = 0
    while not g.terminal and steps < max_steps:
        opts = g.options()
        i = chance.randbelow(len(opts))
        steps += 1
        if g.apply(opts[i]):
            break
    return g.winner, list(g.points), steps, g.pack(), chance.i


def _oracle_one(key):
    from oracle import citadels_oracle as O
    if key[0] == "play":
        _, seed, gid, ruleset, max_steps = key
        w, pts, steps, g = O.playout(seed, gid, ruleset, max_steps=max_steps)
        fin, draws = g.pack(), g.chance.i
    else:
        _, seed, rec, max_steps = key
        w, pts, steps, fin, draws = oracle_continue(rec, seed, max_steps)
    return int(w), tuple(int(x) for x in pts), int(steps), visible(fin), int(draws)


def _oracle_chunk(keys):
    return [_oracle_one(k) for k in keys]


_MEMO = {}


class Expected:
    """Oracle results of a list of games, as arrays: winner, points (int64), steps, draws, and the final records' visible bytes."""

    def __init__(self, rows):
        self.winner = np.array([r[0] for r in rows], dtype=np.int64)
        self.points = np.array([r[1] for r in rows], dtype=np.int64).reshape(-1, 6)
        self.steps = np.array([r[2] for r in rows], dtype=np.int64)
        self.visible = [r[3] for r in rows]
        self.draws = np.array([r[4] for r in rows], dtype=np.int64)


def _oracle(pool, keys):
    todo = [k for k in dict.fromkeys(keys) if k not in _MEMO]
    if todo:
        per = max(1, min(64, (len(todo) + 63) // 64))          # small chunks: games differ in length by 5x
        chunks = [todo[i:i + per] for i in range(0, len(todo), per)]
        for chunk, res in zip(chunks, pool.map(_oracle_chunk, chunks, chunksize=1)):
            _MEMO.update(zip(chunk, res))
    return Expected([_MEMO[k] for k in keys])


def oracle_games(pool, seed, gids, ruleset, max_steps=CAP):
    return _oracle(pool, [("play", int(seed), int(g), int(ruleset), int(max_steps)) for g in gids])


def oracle_continuations(pool, seed, recs, max_steps=CAP):
    return _oracle(pool, [("cont", int(seed), bytes(r.tobytes()), int(max_steps)) for r in recs])


# ---------------------------------------------------------------------------------------------------- CPU self-test
def test_oracle_continuation_is_the_playout():
    """The continuation helper is the oracle's playout: stop a game after k steps, pack it with its gid and draw counter,
    continue it, and the game ends as O.playout ends it (winner, points, step total, final record); k past the end continues
    by zero steps."""
    from oracle import citadels_oracle as O
    from oracle.philox import PhiloxChance
    rng = np.random.default_rng(7)
    for ruleset in (0, 1, 2):
        for j in range(30):
            seed, gid = 0x1234 + 17 * j, (3 << 32) + 1000 * ruleset + j
            w, pts, total, g_full = O.playout(seed, gid, ruleset)
            k = [0, 1, total - 1, total, total + 5][j] if j < 5 else int(rng.integers(2, total - 1))
            chance = PhiloxChance(seed, gid)
            g = O.new_game(chance, ruleset)
            for _ in range(min(k, total)):
                opts = g.options()
                g.apply(opts[chance.randbelow(len(opts))])
            rec = np.frombuffer(bytearray(g.pack()), dtype=STATE_DTYPE).copy()
            rec["rng_draws"], rec["gid"], rec["steps"] = chance.i, gid, min(k, total)
            cw, cpts, csteps, cfin, cdraws = oracle_continue(rec.tobytes(), seed)
            assert (cw, cpts, min(k, total) + csteps) == (w, pts, total), (ruleset, j, k)
            assert cfin[:228] == g_full.pack()[:228] and cdraws == g_full.chance.i, (ruleset, j, k)
            if k >= total:
                assert csteps == 0 and cfin == g.pack()


# ---------------------------------------------------------------------------------------------------- GPU fixtures
@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as p:
        yield p


@pytest.fixture(scope="module")
def engine():
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=N_BIG)
    yield e
    e.close()


@pytest.fixture
def fresh():
    """An engine that has never written its slots: what it knows about them comes from the test's calls alone."""
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=8192)
    yield e
    e.close()


@pytest.fixture(scope="module")
def big(engine):
    """ctd_playout of N_BIG games per ruleset (a B200 holds 148 x 6 x 256 = 227,328 at once: most threads play several)."""
    cache = {}

    def get(ruleset):
        if ruleset not in cache:
            cache[ruleset] = engine.playout(N_BIG, seed=BIG_SEED + ruleset, first_gid=BIG_GID0, ruleset=ruleset)
        return cache[ruleset]
    return get


def _first_wave():
    """Threads the device can hold at once: a game at an index past this is some thread's second or later game."""
    import torch
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count * getattr(p, "max_threads_per_multi_processor", 2048)


def _play_steps(engine, n, seed, first_gid, ruleset, k, rng):
    """reset, then k env steps through enumerate / step with uniform picks of `rng` -> the stored records."""
    engine.reset(n, seed=seed, first_gid=first_gid, ruleset=ruleset)
    for _ in range(k):
        opts, counts = engine.enumerate(n, stride=256)
        pick = (rng.random(n) * counts).astype(np.int64)
        # a finished game has no option, and its row of opts is not written: step it with 0, which leaves it as it is
        engine.step(np.where(counts > 0, opts[np.arange(n), pick], 0).astype(np.uint64))
    return engine.store_states(n)


@pytest.fixture(scope="module")
def midgame(engine):
    """Records of each ruleset at STOPS steps into their games, PER_STOP each, then N_TERMINAL finished games; "mixed" is all
    three rulesets' records shuffled together."""
    cache = {}

    def get(which):
        if which not in cache:
            if which == "mixed":
                allr = np.concatenate([get(r) for r in (0, 1, 2)])
                cache[which] = allr[np.random.default_rng(5).permutation(len(allr))]
            else:
                rng = np.random.default_rng(100 + which)
                parts = [_play_steps(engine, PER_STOP, BUILD_SEED, (1 << 36) + 10_000 * which + 1000 * i, which, k, rng)
                         for i, k in enumerate(STOPS)]
                engine.reset(N_TERMINAL, seed=BUILD_SEED, first_gid=(1 << 36) + 10_000 * which + 9000, ruleset=which)
                engine.playout_slots(N_TERMINAL)
                parts.append(engine.store_states(N_TERMINAL))
                recs = np.concatenate(parts)
                assert (recs[:, 228] == 0).all() and (recs[:, 227] == which).all()
                cache[which] = recs
        return cache[which]
    return get


# ---------------------------------------------------------------------------------------------------- checks
def _assert_rows(out, exp, idx=None, cap=CAP):
    """Per-game rows of ctd_playout against the oracle (scores saturate to int8 in the rows); games the oracle stops at `cap`
    compare by steps and winner == -1 when `cap` is the 4096 default (the random rulesets' never-ending games), in full
    otherwise."""
    sl = slice(None) if idx is None else idx
    w, p, s = out["winner"][sl].astype(np.int64), out["points"][sl].astype(np.int64), out["steps"][sl].astype(np.int64)
    assert np.array_equal(s, exp.steps), ("steps", np.nonzero(s != exp.steps)[0][:8])
    assert np.array_equal(w, exp.winner), ("winner", np.nonzero(w != exp.winner)[0][:8])
    full = exp.steps < CAP if cap == CAP else np.ones(len(s), dtype=bool)
    want = np.clip(exp.points, -128, 127)
    assert np.array_equal(p[full], want[full]), ("points", np.nonzero((p != want).any(1) & full)[0][:8])


def _continue_and_check(engine, pool, n, seed, max_steps=CAP):
    """playout_slots(n) against the oracle's continuation of each slot as it was: winner, steps, the final record's visible
    bytes, draw counter, step counter and error byte (CTD_ERR_MAXSTEPS when capped, CTD_ERR_OVERFLOW for a score past the
    record's int8); a record that was already finished stays byte-identical."""
    before = engine.store_states(n)
    exp = oracle_continuations(pool, seed, before, max_steps)
    w, s = engine.playout_slots(n, max_steps=max_steps)
    after = engine.store_states(n)
    b, a = before.view(STATE_DTYPE).reshape(n), after.view(STATE_DTYPE).reshape(n)
    assert np.array_equal(s.astype(np.int64), exp.steps), ("steps", np.nonzero(s != exp.steps)[0][:8])
    assert np.array_equal(w.astype(np.int64), exp.winner), ("winner", np.nonzero(w != exp.winner)[0][:8])
    bad = [i for i in range(n) if visible(after[i].tobytes()) != exp.visible[i]]
    assert not bad, ("final record", bad[:8])
    assert np.array_equal(a["rng_draws"].astype(np.int64), exp.draws)
    assert np.array_equal(a["steps"].astype(np.int64), b["steps"].astype(np.int64) + exp.steps)
    capped = (a["gflags"] & 2) == 0
    saturated = ((exp.points < -128) | (exp.points > 127)).any(1)
    assert np.array_equal(a["err"], (np.where(capped, MAXSTEPS_FLAG, 0) | np.where(saturated, OVERFLOW_FLAG, 0)).astype(np.uint8))
    assert (w[capped] == -1).all() and (s[capped] == max_steps).all()
    done = (b["gflags"] & 2) != 0
    assert (s[done] == 0).all() and np.array_equal(after[done], before[done])
    return exp


# ---------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_many_games_per_thread_match_one_game_per_thread(engine, big, ruleset):
    """N_BIG games in one launch (most threads play several, reusing their CtdWork) == the same gids in chunks the persistent
    grid covers with one game per thread at any occupancy: winner, points and steps of every game."""
    import torch
    out = big(ruleset)
    chunk = torch.cuda.get_device_properties(0).multi_processor_count * 256
    for lo in range(0, N_BIG, chunk):
        n = min(chunk, N_BIG - lo)
        part = engine.playout(n, seed=BIG_SEED + ruleset, first_gid=BIG_GID0 + lo, ruleset=ruleset)
        for k in ("winner", "points", "steps"):
            assert np.array_equal(part[k], out[k][lo:lo + n]), (k, lo, np.nonzero(part[k] != out[k][lo:lo + n])[0][:8])


@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_later_games_of_a_thread_vs_oracle(big, pool, ruleset):
    """4096 games past the first wave of threads (each is some thread's second or later game) against O.playout."""
    wave = _first_wave()
    assert wave + 4096 < N_BIG
    idx = np.unique(np.concatenate([np.random.default_rng(ruleset).choice(np.arange(wave, N_BIG - 1), 4095, replace=False),
                                    [N_BIG - 1]]))
    assert len(idx) == 4096
    _assert_rows(big(ruleset), oracle_games(pool, BIG_SEED + ruleset, BIG_GID0 + idx, ruleset), idx)


@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_every_counter_from_the_rows(engine, big, pool, ruleset):
    """Every field of ctd_playout_stats recomputed in int64 from the N_BIG per-game rows; ctd_playout_dev (no per-game outputs,
    bench.py's headline figure) returns the same statistics for the same arguments.  A row saturates a score to int8 while
    the counters hold the score itself (a few random classic games score past 127): such rows take their scores from the
    oracle."""
    out = big(ruleset)
    w, p, s = out["winner"].astype(np.int64), out["points"].astype(np.int64), out["steps"].astype(np.int64)
    clamped = np.nonzero(((p == 127) | (p == -128)).any(1))[0]
    if len(clamped):
        exp = oracle_games(pool, BIG_SEED + ruleset, BIG_GID0 + clamped, ruleset)
        assert np.array_equal(np.clip(exp.points, -128, 127), p[clamped])
        p[clamped] = exp.points
    st = out["stats"]
    ended = w >= 0
    assert st["games"] == N_BIG
    assert st["steps"] == int(s.sum()) and st["steps_sq"] == int((s * s).sum())
    assert st["wins"] == [int(x) for x in np.bincount(w[ended], minlength=6)]
    assert st["points_sum"] == [int(x) for x in p.sum(0)] and st["points_sq"] == [int(x) for x in (p * p).sum(0)]
    assert st["errors"] == int((~ended).sum()) and (s[~ended] == CAP).all()   # only the random rulesets' endless games
    assert ruleset == 2 or st["errors"] == 0
    assert st["max_steps"] == int(s.max())
    dev = engine.playout(N_BIG, seed=BIG_SEED + ruleset, first_gid=BIG_GID0, ruleset=ruleset, outputs=False)["stats"]
    dev.pop("kernel_ms")
    assert dev == st


@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_ragged_and_boundary_launches_vs_oracle(engine, pool, ruleset):
    """Partial warps and blocks (1, 31, 33, 255, 257, 4097 games), gids that cross 2^32, and step caps 1 / 37 / 300 (a capped
    game: steps == cap, winner -1, counted in errors) against the oracle."""
    seed = 0x7A66ED + ruleset
    for n in (1, 31, 33, 255, 257, 4097):
        out = engine.playout(n, seed=seed, first_gid=40_000_000, ruleset=ruleset)
        _assert_rows(out, oracle_games(pool, seed, 40_000_000 + np.arange(n), ruleset))
        assert out["stats"]["games"] == n and out["stats"]["steps"] == int(out["steps"].astype(np.int64).sum())
    gid0 = (1 << 32) - 1500
    out = engine.playout(3000, seed=seed, first_gid=gid0, ruleset=ruleset)
    _assert_rows(out, oracle_games(pool, seed, gid0 + np.arange(3000), ruleset))
    for cap in (1, 37, 300):
        out = engine.playout(4096, seed=seed, first_gid=50_000_000, ruleset=ruleset, max_steps=cap)
        exp = oracle_games(pool, seed, 50_000_000 + np.arange(4096), ruleset, max_steps=cap)
        _assert_rows(out, exp, cap=cap)
        capped = out["winner"] == -1
        assert (out["steps"][capped] == cap).all() and out["stats"]["errors"] == int(capped.sum())
        assert capped.any() and out["stats"]["max_steps"] <= cap


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1, 2, "mixed"])
def test_playout_slots_continues_mid_game_records(fresh, pool, midgame, which):
    """Records stopped 0 / 40 / 150 / 400 steps into their games, and finished ones, continued by ctd_playout_slots under a seed
    of their own (set_seed): per ruleset the specialised kernel runs, mixed the generic one.  The same records again with
    max_steps = 25: steps min(25, remaining), the capped records flagged."""
    recs = midgame(which)
    n = len(recs)
    fresh.load_states(recs)
    fresh.set_seed(CONT_SEED)
    exp = _continue_and_check(fresh, pool, n, CONT_SEED)
    assert (exp.steps > 0).sum() >= n // 2
    fresh.load_states(recs)
    short = _continue_and_check(fresh, pool, n, CONT_SEED, max_steps=25)
    assert np.array_equal(short.steps, np.minimum(25, exp.steps))


@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_bench_e2e_path_at_full_size(engine, big, pool, ruleset):
    """bench.py's e2e figure: reset(2^20) -> store_states -> load_states -> playout_slots(2^20) plays the games playout(2^20)
    plays; 1024 final records past the first wave equal the oracle's."""
    engine.reset(N_BIG, seed=BIG_SEED + ruleset, first_gid=BIG_GID0, ruleset=ruleset)
    engine.load_states(engine.store_states(N_BIG))
    w, s = engine.playout_slots(N_BIG)
    out = big(ruleset)
    assert np.array_equal(w, out["winner"]) and np.array_equal(s, out["steps"])
    wave = _first_wave()
    idx = np.sort(np.random.default_rng(50 + ruleset).choice(np.arange(wave, N_BIG), 1024, replace=False))
    exp = oracle_games(pool, BIG_SEED + ruleset, BIG_GID0 + idx, ruleset)
    fin = engine.store_states(N_BIG)[idx]
    done = exp.steps < CAP
    bad = [int(i) for j, i in enumerate(idx) if done[j] and visible(fin[j].tobytes()) != exp.visible[j]]
    assert not bad, ("final record", bad[:8])
    draws = fin.view(STATE_DTYPE).reshape(-1)["rng_draws"].astype(np.int64)
    assert np.array_equal(draws[done], exp.draws[done])


class _DevBytes:
    """A device address as torch.as_tensor reads it (the CUDA array interface)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = dict(shape=(nbytes,), typestr="|u1", data=(ptr, False), version=3)


SEQUENCES = ("load_cuts_run", "load_extends_run", "load_cuts_then_partial", "states_dev_drops_run", "make_roots", "load_roots")


@pytest.mark.gpu
@pytest.mark.parametrize("seq", SEQUENCES)
def test_kernel_selection_survives_every_way_of_writing_the_slots(fresh, pool, midgame, seq):
    """The preset- and classic-specialised kernels treat every other ruleset's characters as unreachable, so a slot run
    that claimed a ruleset the slots no longer hold would give wrong games.  After each way of writing the slots,
    playout_slots agrees with the oracle on every slot."""
    import torch
    n, seed = 256, 0x5E1EC7
    rng = np.random.default_rng(SEQUENCES.index(seq))

    def pick(ruleset, m):
        recs = midgame(ruleset)
        return recs[np.sort(rng.choice(len(recs), m, replace=False))]
    e = fresh
    if seq == "load_cuts_run":
        e.reset(2 * n, seed=seed, first_gid=7000, ruleset=0)
        e.load_states(pick(1, n), first_slot=0)
        _continue_and_check(e, pool, 2 * n, seed)
    elif seq == "load_extends_run":
        e.reset(n, seed=seed, first_gid=7000, ruleset=0)
        e.load_states(pick(0, n), first_slot=n)
        _continue_and_check(e, pool, 2 * n, seed)
    elif seq == "load_cuts_then_partial":
        e.reset(2 * n, seed=seed, first_gid=7000, ruleset=1)
        e.load_states(pick(2, n // 4), first_slot=n // 2)
        _continue_and_check(e, pool, n // 2, seed)
        _continue_and_check(e, pool, 2 * n, seed)
    elif seq == "states_dev_drops_run":
        e.reset(2 * n, seed=seed, first_gid=7000, ruleset=0)
        ptr = e.states_dev_ptr()
        e.sync()
        src = np.ascontiguousarray(np.concatenate([pick(2, n // 2), pick(1, n // 2)]))
        dst = torch.as_tensor(_DevBytes(ptr, src.nbytes), device="cuda:%d" % e.device)
        dst.copy_(torch.from_numpy(src.reshape(-1)).to(dst.device))
        torch.cuda.synchronize(dst.device)
        assert np.array_equal(e.store_states(n), src)
        _continue_and_check(e, pool, 2 * n, seed)
    elif seq == "make_roots":
        e.reset(2 * n, seed=seed, first_gid=7000, ruleset=0)
        e.make_roots(n, seed=seed + 1, first_gid=8000, ruleset=2, back_lo=0, back_hi=60)
        _continue_and_check(e, pool, n, seed + 1)
    else:
        e.make_roots(n, seed=seed + 1, first_gid=8000, ruleset=2, back_lo=0, back_hi=60)
        roots = e.store_roots(n)
        e.reset(2 * n, seed=seed, first_gid=7000, ruleset=0)
        e.load_roots(*roots)
        _continue_and_check(e, pool, n, seed)
