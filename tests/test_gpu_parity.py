"""GPU parity tests: the CUDA engine, called through the C ABI, against (a) the committed golden
fixtures produced by the real reference and (b) the oracle on fresh seeds.  Integer work: bit-exact."""
import zlib
import numpy as np
import pytest

from tests.golden_util import Traces, visible

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=4096)
    yield e
    e.close()


def _replay(engine, name, with_tape):
    """Replay every golden game in lock-step through ctd_enumerate / ctd_step."""
    T = Traces(name)
    n = len(T)
    if with_tape:
        engine.set_tapes([T.game_tape(g) for g in range(n)])
    else:
        engine.set_tapes(None)
    # golden gids are contiguous
    assert np.all(np.diff(T.gids.astype(np.int64)) == 1)
    engine.reset(n, seed=T.seed, first_gid=int(T.gids[0]), ruleset=T.ruleset)
    lens = np.diff(T.step_off).astype(np.int64)
    maxlen = int(lens.max())
    base = T.step_off[:-1].astype(np.int64)
    checked = 0
    for k in range(maxlen):
        live = np.nonzero(lens > k)[0]
        opts, counts = engine.enumerate(n, stride=64)
        if k % 3 == 0:   # the playout kernel's choice (ctd_lane_count / ctd_lane_select): every k of every state vs this list
            mis = engine.choose_check(n)
            assert not mis[live].any(), ("cooperative chooser differs", name, k, np.nonzero(mis)[0][:5], mis[mis > 0][:5])
        states = engine.store_states(n)
        idx = base[live] + k
        assert np.array_equal(counts[live], T.nopt[idx].astype(np.uint32)), "option count mismatch at step %d" % k
        for g, i in zip(live, idx):
            assert zlib.crc32(visible(states[g].tobytes())) == int(T.state_crc[i]), (name, "state", int(g), k)
            assert zlib.crc32(opts[g, :counts[g]].astype("<u8").tobytes()) == int(T.opts_crc[i]), (name, "opts", int(g), k)
        chosen = np.zeros(n, dtype=np.uint64)
        chosen[live] = opts[live, T.chosen[idx].astype(np.int64)]
        winner = engine.step(chosen)
        ending = live[lens[live] == k + 1]
        assert np.all(winner[ending] >= 0)
        assert np.all(winner[np.setdiff1d(live, ending)] == -1)
        checked += len(live)
    final = engine.store_states(n)
    assert np.array_equal(final[:, :228], T.final[:, :228])
    assert np.all(final[:, 228] == 0), "engine error flags set"
    engine.set_tapes(None)
    return checked


def test_replay_preset_tapes(engine):
    """SURVEY 8(d) parity gate 1: 1000 recorded reference games, state + option list after every step."""
    assert _replay(engine, "preset_traces.npz", True) > 400000


def test_replay_classic_tapes(engine):
    assert _replay(engine, "classic_traces.npz", True) > 100000


def test_replay_random_tapes(engine):
    """Game(preset=False): all 24 characters, random uniques / variants / order / crown (500 recorded reference games)."""
    assert _replay(engine, "random_traces.npz", True) > 150000


@pytest.mark.parametrize("name", ["preset_traces.npz", "classic_traces.npz", "random_traces.npz"])
def test_fused_playout_matches_reference_finals(engine, name):
    """The fused Philox playout kernel reproduces the reference's terminal states for the golden gids."""
    T = Traces(name)
    n = len(T)
    out = engine.playout(n, seed=T.seed, first_gid=int(T.gids[0]), ruleset=T.ruleset)
    assert out["stats"]["errors"] == 0
    assert np.array_equal(out["steps"].astype(np.int64), np.diff(T.step_off))
    assert np.array_equal(out["winner"], T.final[:, 218].view(np.int8))
    assert np.array_equal(out["points"], T.final[:, 220:226].view(np.int8))
    assert out["stats"]["games"] == n and out["stats"]["steps"] == int(np.diff(T.step_off).sum())


def test_fused_playout_vs_oracle_fresh_seeds(engine):
    """Fresh (seed, gid) pairs the fixtures do not cover: CUDA vs the Python oracle, bit-exact outcomes."""
    from oracle import citadels_oracle as O
    for ruleset, seed, gid0, n in ((0, 12345, 7_000_000, 48), (1, 0xDEADBEEFCAFE, 1 << 33, 32), (2, 424242, 9_000_000, 32)):
        out = engine.playout(n, seed=seed, first_gid=gid0, ruleset=ruleset)
        for i in range(n):
            w, pts, steps, _ = O.playout(seed, gid0 + i, ruleset)
            assert (w, pts, steps) == (int(out["winner"][i]), [int(x) for x in out["points"][i]], int(out["steps"][i]))


def test_playout_slots_continues_loaded_states(engine):
    """ctd_playout_slots == finishing the game from a mid-game state (run_utils.py:37-41 tail): 100 steps through enumerate /
    step with the playout's own choice (draw number rng_draws of the game's Philox stream, which the record then counts), then
    the fused kernel finishes the games."""
    from oracle.philox import PhiloxChance
    from citadels_self_play_b200.layout import STATE_DTYPE
    T = Traces("preset_full.npz")
    n, k = len(T), 100
    assert np.diff(T.step_off).min() > k
    out = engine.playout(n, seed=T.seed, first_gid=int(T.gids[0]), ruleset=0)
    engine.set_tapes(None)
    engine.reset(n, seed=T.seed, first_gid=int(T.gids[0]), ruleset=0)
    assert np.array_equal(engine.store_states(n)[:, :228], T.states[T.step_off[:-1], :228])
    for _ in range(k):
        opts, counts = engine.enumerate(n, stride=64)
        states = engine.store_states(n)
        rec = states.view(STATE_DTYPE).reshape(n)
        chosen = np.zeros(n, dtype=np.uint64)
        for g in range(n):
            chance = PhiloxChance(T.seed, int(rec["gid"][g]))
            chance.i = int(rec["rng_draws"][g])
            chosen[g] = opts[g, chance.randbelow(int(counts[g]))]
            rec["rng_draws"][g] = chance.i
        engine.load_states(states)
        engine.step(chosen)
    mid = engine.store_states(n)
    assert np.array_equal(mid[:, :228], T.states[T.step_off[:-1] + k, :228])
    winner, steps = engine.playout_slots(n)
    assert np.array_equal(winner, out["winner"])
    assert np.array_equal(steps.astype(np.int64), out["steps"].astype(np.int64) - k)
    fin = engine.store_states(n)
    assert np.array_equal(fin[:, :228], T.final[:, :228])


def test_determinism_and_sharding_invariance(engine):
    """Results are a pure function of (seed, gid): two shards concatenated == one batch (multi-GPU rule)."""
    a = engine.playout(512, seed=99, first_gid=1000)
    b1 = engine.playout(200, seed=99, first_gid=1000)
    b2 = engine.playout(312, seed=99, first_gid=1200)
    assert np.array_equal(a["winner"], np.concatenate([b1["winner"], b2["winner"]]))
    assert np.array_equal(a["points"], np.concatenate([b1["points"], b2["points"]]))
    assert np.array_equal(a["steps"], np.concatenate([b1["steps"], b2["steps"]]))
    for k in ("games", "steps", "steps_sq", "errors"):
        assert a["stats"][k] == b1["stats"][k] + b2["stats"][k]
    assert a["stats"]["wins"] == [x + y for x, y in zip(b1["stats"]["wins"], b2["stats"]["wins"])]


@pytest.mark.parametrize("fixture,ruleset", [("ref_outcomes_preset.npz", 0), ("ref_outcomes_classic.npz", 1),
                                             ("ref_outcomes_random.npz", 2)])
def test_distribution_vs_reference_sample(engine, fixture, ruleset):
    """SURVEY 8(d) parity gate 2: winner multinomial and per-seat mean score of 2^18 GPU playouts against
    games of the unmodified reference under its own Mersenne Twister (tests/golden/ref_outcomes_*.npz: 20,000 preset
    games, 12,000 each of the classic eight and of Game(preset=False)).
    Two-sample tests at the 99% level (chi-square with 5 dof: 15.09; |z| < 2.576 Bonferroni-relaxed to 3.2
    over the 13 z-tests)."""
    import os
    from tests.golden_util import GOLDEN
    ref = np.load(os.path.join(GOLDEN, fixture))
    n = 1 << 18
    out = engine.playout(n, seed=2024 + ruleset, first_gid=0, ruleset=ruleset)
    st = out["stats"]
    assert st["games"] == n
    # Game(preset=False) under uniform random play has games that never end (every hand and the deck empty, nobody can
    # build: the reference loops forever as well; seed 2026 gid 109177 is one).  The engine stops them at max_steps and
    # flags them; nothing else may be flagged.
    capped = out["steps"] == 4096
    assert st["errors"] == int(capped.sum()) and (out["winner"][capped] == -1).all()
    assert st["errors"] == 0 if ruleset != 2 else st["errors"] <= 3
    rw = np.bincount(ref["winner"], minlength=6).astype(np.float64)
    gw = np.asarray(st["wins"], dtype=np.float64)
    nr, ng = rw.sum(), gw.sum()
    pooled = (rw + gw) / (nr + ng)
    chi2 = (((rw - nr * pooled) ** 2) / (nr * pooled)).sum() + (((gw - ng * pooled) ** 2) / (ng * pooled)).sum()
    assert chi2 < 15.09, ("winner distribution", chi2, rw / nr, gw / ng)
    rp = ref["points"].astype(np.float64)
    gp = out["points"][~capped].astype(np.float64)
    z = (gp.mean(0) - rp.mean(0)) / np.sqrt(gp.var(0) / ng + rp.var(0) / nr)
    assert np.all(np.abs(z) < 3.2), ("mean points", z)
    rs, gs = ref["steps"].astype(np.float64), out["steps"][~capped].astype(np.float64)
    zs = (gs.mean() - rs.mean()) / np.sqrt(gs.var() / ng + rs.var() / nr)
    assert abs(zs) < 3.2, ("steps", gs.mean(), rs.mean(), zs)
    assert abs(gs.std() - rs.std()) < (2.0 if ruleset == 0 else 3.0)


def test_full_size_properties_one_million_games():
    """BASELINE configs[1] at full size (2^20 games): size-independent properties -- determinism, shard invariance of the
    outcome statistics (the multi-GPU rule: rank r plays ids [r*G/N, (r+1)*G/N)), and internal consistency of the counters."""
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=64)
    n = 1 << 20
    a = e.playout(n, seed=0xC17ADE15, first_gid=0, outputs=False)["stats"]
    b = e.playout(n, seed=0xC17ADE15, first_gid=0, outputs=False)["stats"]
    keys = ("games", "steps", "steps_sq", "wins", "points_sum", "points_sq", "errors", "max_steps")
    assert all(a[k] == b[k] for k in keys)
    parts = [e.playout(n // 8, seed=0xC17ADE15, first_gid=r * (n // 8), outputs=False)["stats"] for r in range(8)]
    for k in ("games", "steps", "steps_sq", "errors"):
        assert a[k] == sum(p[k] for p in parts), k
    for k in ("wins", "points_sum", "points_sq"):
        assert list(a[k]) == [sum(p[k][i] for p in parts) for i in range(6)], k
    assert a["max_steps"] == max(p["max_steps"] for p in parts)
    assert a["games"] == n and a["errors"] == 0 and sum(a["wins"]) == n
    mean = a["steps"] / n
    assert 410 < mean < 428 and 244 <= a["max_steps"] < 1200          # reference: 418.6 +- 65.4 steps per game
    out = e.playout(1 << 16, seed=0xC17ADE15, first_gid=0)            # per-game rows agree with the counters
    assert int(out["steps"].astype(np.int64).sum()) == out["stats"]["steps"]
    assert list(np.bincount(out["winner"], minlength=6)) == list(out["stats"]["wins"])
    assert [int(x) for x in out["points"].astype(np.int64).sum(0)] == list(out["stats"]["points_sum"])
    e.close()


def _oracle_outcomes(args):
    seed, gid0, n, ruleset = args
    from oracle import citadels_oracle as O
    return [O.playout(seed, gid0 + i, ruleset)[:3] for i in range(n)]


@pytest.mark.parametrize("ruleset,n", [(0, 4096), (1, 2048), (2, 1024)])
def test_fused_playout_vs_oracle_thousands_of_games(engine, ruleset, n):
    """The three playout kernels (preset-specialised, classic-specialised, generic) against the oracle on thousands of fresh
    games each, bit-exact winner / six scores / step count (the oracle runs on the host cores in a process pool)."""
    import multiprocessing as mp
    import os
    seed, gid0 = 0xABCDEF12 + ruleset, 3_000_000
    out = engine.playout(n, seed=seed, first_gid=gid0, ruleset=ruleset)
    cores = min(16, os.cpu_count() or 1)
    per = (n + cores - 1) // cores
    jobs = [(seed, gid0 + c * per, min(per, n - c * per), ruleset) for c in range(cores) if c * per < n]
    with mp.get_context("spawn").Pool(len(jobs)) as pool:     # not fork: this process holds a CUDA context
        res = [r for chunk in pool.map(_oracle_outcomes, jobs) for r in chunk]
    assert len(res) == n
    ow = np.array([r[0] for r in res], dtype=np.int8)
    op = np.array([r[1] for r in res], dtype=np.int8)
    os_ = np.array([r[2] for r in res], dtype=np.int64)
    capped = os_ >= 4096                        # never-ending games of the random rulesets: both sides stop at the cap
    assert np.array_equal(out["steps"].astype(np.int64)[~capped], os_[~capped])
    assert np.array_equal(out["winner"][~capped], ow[~capped])
    assert np.array_equal(out["points"][~capped], op[~capped])
    assert capped.sum() <= 1 and out["stats"]["errors"] == int(capped.sum())
