"""ctd_arena_record / the engine's dataset / ctd_train_begin_dataset: self-play records taken on the device.  Recording changes no
game, its records equal ctd_mccfr_targets on the same trees searched through the facade, and training from the dataset equals
training from the same rows on the host."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED = 0x5E1F9A


def _checkpoint():
    from tests.test_value_checkpoint import load
    return load()[1]


def _pick(seed, gid, s, n):
    """The random seats' draw: word s & 3 of Philox block (s >> 2, stream 4, gid), k = (u * n) >> 32."""
    from oracle.philox import philox4x32_10, MASK
    from citadels_self_play_b200.layout import ARENA_STREAM
    r = philox4x32_10(s >> 2, ARENA_STREAM, gid & MASK, gid >> 32, seed & MASK, (seed >> 32) & MASK)
    return (r[s & 3] * n) >> 32


def _mirror(seed, gid, ruleset, seats, model, search_engine, thresholds, max_steps=4096):
    """compare_to_random.play_games for one game through the facade, as tests/test_gpu_arena_device._mirror; after every search,
    Engine.mccfr_targets of its tree at each threshold.  -> (game, searches, {t: (seat, steps, {threshold: targets})})."""
    from citadels_self_play_b200 import arena, facade as F
    from citadels_self_play_b200.layout import SEAT_RANDOM, SEAT_DEEP
    g = F.create_game(seed=seed, gid=gid, ruleset=ruleset)
    t = 0
    found = {}
    while not g.terminal and int(g._rec["steps"]) < max_steps:
        s = int(g._rec["steps"])
        opts = g.get_options_from_state()
        kind, its, depth, weight = seats[g.gamestate.player_id]
        if kind != SEAT_RANDOM and len(opts) >= 2:
            res = arena.search_batch(search_engine, [g], [t], model if kind & 0xFF == SEAT_DEEP else None, its, depth, weight)
            found[t] = (g.gamestate.player_id, s, {th: search_engine.mccfr_targets(1, seed=seed, threshold=th) for th in thresholds})
            t += 1
            chosen = arena._live_choice(res[0], g, opts)
        else:
            chosen = opts[_pick(seed, gid, s, len(opts))]
        chosen.carry_out(g)
    return g, t, found


def _by_tree(data):
    """canonical dataset -> {(gid, search): [record indices in canonical order]}"""
    out = {}
    for i, o in enumerate(data["origin"]):
        out.setdefault((int(o["gid"]), int(o["search"])), []).append(i)
    return out


def _same_record(data, i, ref, j):
    m, r = data["meta"][i], ref["meta"][j]
    assert np.array_equal(data["features"][i], ref["features"][j])
    for k in ("node", "n_options", "seat", "role_pick"):
        assert int(m[k]) == int(r[k]), k
    assert np.array_equal(m["node_value"], r["node_value"])
    a, b, k = int(m["option_offset"]), int(r["option_offset"]), int(m["n_options"])
    assert np.array_equal(data["options"][a:a + k], ref["options"][b:b + k])
    assert np.array_equal(data["regrets"][a:a + k], ref["regrets"][b:b + k])


@pytest.mark.parametrize("ruleset", [0, 1, 2])
def test_recording_changes_no_game(ruleset):
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE, RECORD_ROOT
    seats = [arena.deep(20, 10, 5.0), arena.pure(40), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.deep(20, 10, 5.0)]
    e = Engine(capacity=16)
    try:
        e.set_value_model(_checkpoint())
        e.dataset_reserve(200_000, 4_000_000)
        first_gid = 300 + 50 * ruleset
        plain = e.arena(6, seats, seed=SEED, first_gid=first_gid, ruleset=ruleset)
        plain_states = e.store_states(6)
        for mode in (RECORD_TREE, RECORD_ROOT):
            out = e.arena(6, seats, seed=SEED, first_gid=first_gid, ruleset=ruleset, record=([0, 1, 3, 5], mode, 15.0))
            for k in ("winner", "points", "steps", "searches"):
                assert np.array_equal(out[k], plain[k]), (mode, k)
            assert out["stats"] == plain["stats"], mode
            assert e.store_states(6).tobytes() == plain_states.tobytes(), mode
            assert out["phase_ms"]["record"] >= 0.0 and "record" not in plain["phase_ms"]
        assert e.dataset_info()["records"] > 0
    finally:
        e.close()


def test_records_equal_the_reference_path():
    """Each recorded tree's records equal ctd_mccfr_targets of the same search made through the facade: all of them in tree mode,
    node 0's in root mode.  Unrecorded and random seats yield nothing; the origin matches the mirror game."""
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE, RECORD_ROOT
    model = _checkpoint()
    seats = [arena.deep(20, 10, 5.0), arena.pure(40), arena.random_seat(), arena.random_seat(), arena.pure(40), arena.random_seat()]
    recorded = [0, 1, 2]   # seat 4 searches but is not recorded; seat 2 is random
    n, first_gid = 4, 900
    eng, se = Engine(capacity=16), Engine(capacity=4)
    try:
        eng.set_value_model(model)
        data = {}
        for mode in (RECORD_TREE, RECORD_ROOT):
            eng.dataset_reserve(100_000, 2_000_000)
            out = eng.arena(n, seats, seed=SEED, first_gid=first_gid, record=(recorded, mode, 15.0))
            data[mode] = eng.dataset_read()
        for i in range(n):
            g, t_n, found = _mirror(SEED, first_gid + i, 0, seats, model, se, (15.0, 0.0))
            assert int(out["searches"][i]) == t_n
            for mode in (RECORD_TREE, RECORD_ROOT):
                d = data[mode]
                trees = _by_tree(d)
                for t, (seat, step, refs) in found.items():
                    got = trees.get((first_gid + i, t), [])
                    if seat not in recorded:
                        assert got == [], (mode, i, t, seat)
                        continue
                    if mode == RECORD_TREE:
                        ref = refs[15.0]
                        assert len(got) == len(ref["meta"]), (i, t)
                        for j, r in enumerate(got):
                            _same_record(d, r, ref, j)
                    else:
                        ref = refs[0.0]
                        assert len(got) == 1 and int(ref["meta"][0]["node"]) == 0, (i, t)
                        _same_record(d, got[0], ref, 0)
                    for r in got:
                        o = d["origin"][r]
                        assert (int(o["mover"]), int(o["step"])) == (seat, step)
                        assert int(o["winner"]) == int(g._rec["winner"]) == int(out["winner"][i])
                        assert [int(x) for x in o["points"]] == g.points
                        assert int(d["meta"][r]["tree"]) == i
        for mode in (RECORD_TREE, RECORD_ROOT):
            assert set(int(m) for m in data[mode]["origin"]["mover"]) <= set(recorded)
        assert len(data[RECORD_ROOT]["meta"]) > 0 and len(data[RECORD_TREE]["meta"]) > 0
    finally:
        eng.close()
        se.close()


def _canonical(data):
    """the dataset without its physical layout: per record the features, meta without tree / option_offset, origin, option slice"""
    rows = []
    for i in range(len(data["meta"])):
        m = data["meta"][i]
        a, k = int(m["option_offset"]), int(m["n_options"])
        rows.append((data["features"][i].tobytes(), int(m["node"]), k, int(m["seat"]), int(m["role_pick"]), m["node_value"].tobytes(),
                     data["origin"][i].tobytes(), data["options"][a:a + k].tobytes(), data["regrets"][a:a + k].tobytes()))
    return rows


def test_dataset_does_not_depend_on_capacity_or_batching():
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE
    seats = [arena.pure(30), arena.random_seat(), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.pure(20)]
    rec = ([0, 3, 5], RECORD_TREE, 15.0)
    big, small = Engine(capacity=64), Engine(capacity=3)
    try:
        big.dataset_reserve(100_000, 2_000_000)
        small.dataset_reserve(100_000, 2_000_000)
        big.arena(16, seats, seed=SEED, first_gid=5000, record=rec)
        small.arena(16, seats, seed=SEED, first_gid=5000, record=rec)
        a, b = _canonical(big.dataset_read()), _canonical(small.dataset_read())
        big.dataset_clear()
        big.arena(8, seats, seed=SEED, first_gid=5000, record=rec)
        big.arena(8, seats, seed=SEED, first_gid=5008, record=rec)
        c = _canonical(big.dataset_read())
    finally:
        big.close()
        small.close()
    assert len(a) > 0
    assert a == b
    assert a == c


def test_overflow_drops_whole_trees():
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE
    seats = [arena.pure(40), arena.random_seat(), arena.pure(40), arena.random_seat(), arena.random_seat(), arena.random_seat()]
    rec = ([0, 2], RECORD_TREE, 15.0)
    e = Engine(capacity=8)
    try:
        e.dataset_reserve(100_000, 2_000_000)
        e.arena(12, seats, seed=SEED, first_gid=77, record=rec)
        full = e.dataset_read()
        full_info = e.dataset_info()
        assert full_info["dropped_trees"] == 0 and full_info["dropped_records"] == 0
        full_trees = _by_tree(full)
        cap = max(1, full_info["records"] // 3)
        e.dataset_reserve(cap, 4 * cap)
        e.arena(12, seats, seed=SEED, first_gid=77, record=rec)
        part = e.dataset_read()
        info = e.dataset_info()
    finally:
        e.close()
    assert info["records"] <= cap and info["option_slots"] <= 4 * cap
    assert info["dropped_trees"] > 0
    part_trees = _by_tree(part)
    for key, idx in part_trees.items():
        assert len(idx) == len(full_trees[key]), key
    assert info["records"] + info["dropped_records"] == full_info["records"]
    assert len(part_trees) + info["dropped_trees"] == len(full_trees)


@pytest.mark.parametrize("label", ["node_value", "winner"])
def test_training_from_the_dataset_equals_training_from_host_rows(label, tmp_path):
    import torch
    from citadels_self_play_b200 import Engine, arena, selfplay
    from citadels_self_play_b200.layout import RECORD_TREE
    from citadels_self_play_b200.train import train_node_value_only
    from citadels_self_play_b200.value_model import ValueOnlyNN
    seats = [arena.pure(60), arena.random_seat(), arena.pure(60), arena.random_seat(), arena.random_seat(), arena.random_seat()]
    e = Engine(capacity=16)
    try:
        e.dataset_reserve(100_000, 2_000_000)
        out = e.arena(10, seats, seed=SEED, first_gid=11, record=([0, 2], RECORD_TREE, 15.0))
        assert (out["winner"] >= 0).all()
        data = e.dataset_read()
        tr_rows, va_rows = selfplay.split_by_game(data["origin"], 0.3, seed=3, rows=data["row"])
        assert len(tr_rows) > 0 and len(va_rows) > 0
        where = np.empty(len(data["row"]), dtype=np.int64)
        where[data["row"]] = np.arange(len(data["row"]))

        def tuples(rows):
            out = []
            for r in rows:
                i = where[int(r)]
                v = data["meta"][i]["node_value"].astype(np.float64) if label == "node_value" else np.eye(6)[int(data["origin"][i]["winner"])]
                out.append((torch.from_numpy(data["features"][i].copy()), None, torch.from_numpy(np.array(v, dtype=np.float64)), None))
            return out
        torch.manual_seed(5)
        model = ValueOnlyNN(418, 512)
        h_dev, h_host = {}, {}
        b_dev = selfplay.train_on_dataset(e, tr_rows, va_rows, label, epochs=3, lr=1e-3, batch_size=32, model=model, seed=9,
                                          parent_folder=str(tmp_path / "dev"), history=h_dev)
        b_host = train_node_value_only(tuples(tr_rows), tuples(va_rows), 3, 1e-3, batch_size=32, model=model, seed=9, engine=e,
                                       parent_folder=str(tmp_path / "host"), history=h_host)
    finally:
        e.close()
    assert b_dev == b_host
    assert h_dev["train_losses"] == h_host["train_losses"] and h_dev["eval_losses"] == h_host["eval_losses"]
    for k, v in h_host["final_state"].items():
        assert np.array_equal(h_dev["final_state"][k], v), k


def test_deep_tree_trap():
    """At the reference's threshold a deep seat's tree has no records (eval-mode node_value sums to 5 or 1); its roots do."""
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE, RECORD_ROOT
    seats = [arena.deep(30, 10, 5.0)] + [arena.random_seat()] * 5
    e = Engine(capacity=16)
    try:
        e.set_value_model(_checkpoint())
        e.dataset_reserve(100_000, 2_000_000)
        out = e.arena(6, seats, seed=SEED, first_gid=40, record=([0], RECORD_TREE, 15.0))
        assert e.dataset_info()["records"] == 0 and int(out["searches"].sum()) > 0
        out = e.arena(6, seats, seed=SEED, first_gid=40, record=([0], RECORD_ROOT, 15.0))
        info = e.dataset_info()
        data = e.dataset_read()
    finally:
        e.close()
    assert info["records"] == int(out["searches"].sum()) and info["dropped_records"] == 0
    assert (data["meta"]["node"] == 0).all() and (data["origin"]["mover"] == 0).all()
    assert (data["meta"]["node_value"].sum(axis=1) < 15).all()


def test_record_edge_cases():
    from citadels_self_play_b200 import Engine, EngineError, arena
    from citadels_self_play_b200.layout import RECORD_TREE, RECORD_ROOT, LABEL_WINNER, TARGET_META_DTYPE, ORIGIN_DTYPE
    from citadels_self_play_b200.train import Trainer
    seats = [arena.pure(20), arena.random_seat(), arena.pure(20)] + [arena.random_seat()] * 3
    e = Engine(capacity=16)
    try:
        with pytest.raises(EngineError, match="status 1 "):   # no reservation yet
            e.arena(2, seats, seed=SEED, record=([0], RECORD_TREE, 15.0))
        e.dataset_reserve(50_000, 1_000_000)
        e.arena(4, seats, seed=SEED, record=([], RECORD_TREE, 0.0))
        e.arena(4, seats, seed=SEED, record=([1, 3, 4, 5], RECORD_ROOT, 0.0))   # random seats only
        assert e.dataset_info()["records"] == 0
        for bad in (([0], RECORD_TREE, -1.0), ([0], RECORD_TREE, float("nan")), ([0], 2, 15.0), ([6], RECORD_TREE, 15.0)):
            with pytest.raises(EngineError, match="status 1 "):
                e.arena(2, seats, seed=SEED, record=bad)
        e.arena(4, seats, seed=SEED, record=([0, 2], RECORD_ROOT, 15.0))
        info = e.dataset_info()
        n, ns = info["records"], info["option_slots"]
        assert n > 0 and ns >= 2 * n
        lib, h = e._lib, e._h
        f = np.zeros((n + 1, 448), dtype=np.float32)
        m = np.zeros(n + 1, dtype=TARGET_META_DTYPE)
        o = np.zeros(n + 1, dtype=ORIGIN_DTYPE)
        assert lib.ctd_dataset_read(h, 0, n + 1, f.ctypes.data, m.ctypes.data, o.ctypes.data) == 1
        assert lib.ctd_dataset_read(h, n, 1, f.ctypes.data, None, None) == 1
        assert lib.ctd_dataset_read(h, n, 0, None, None, None) == 0
        opt = np.zeros(ns + 1, dtype=np.uint64)
        assert lib.ctd_dataset_read_options(h, 0, ns + 1, opt.ctypes.data, None) == 1
        assert lib.ctd_dataset_read_options(h, 0, ns, opt.ctypes.data, None) == 0
        for idx, label in (([0, n], LABEL_WINNER), ([0, 1], 7)):
            with pytest.raises(EngineError, match="status 1 "):
                Trainer.from_dataset(e, idx, [], label, 8)
        with pytest.raises(EngineError, match="status 1 "):
            Trainer.from_dataset(e, [0], [n + 5], LABEL_WINNER, 8)
        # games stopped at max_steps: winner -1, and a winner label on them is refused
        e.dataset_clear()
        out = e.arena(4, seats, seed=SEED, max_steps=40, record=([0, 2], RECORD_ROOT, 0.0))
        assert (out["winner"] == -1).all()
        data = e.dataset_read()
        assert len(data["origin"]) > 0 and (data["origin"]["winner"] == -1).all()
        with pytest.raises(EngineError, match="status 1 "):
            Trainer.from_dataset(e, [0], [], LABEL_WINNER, 8)
        Trainer.from_dataset(e, [0], [], 0, 8).close()   # node_value labels do not need an outcome
    finally:
        e.close()


def test_recording_launches():
    """Per search of a recorded group: count, reserve, fill (3 launches); per call: the outcome kernel."""
    from citadels_self_play_b200 import Engine, arena
    from citadels_self_play_b200.layout import RECORD_TREE
    seats = [arena.pure(20), arena.random_seat(), arena.pure(20)] + [arena.random_seat()] * 3   # one search group
    e = Engine(capacity=64)
    try:
        e.dataset_reserve(100_000, 2_000_000)
        l0 = e.launches
        plain = e.arena(32, seats, seed=SEED, first_gid=0)
        l1 = e.launches
        out = e.arena(32, seats, seed=SEED, first_gid=0, record=([0], RECORD_TREE, 15.0))
        l2 = e.launches
    finally:
        e.close()
    chunks = int(out["searches"].max())   # capacity holds every game: one chunk per decision round with a search
    assert np.array_equal(out["searches"], plain["searches"])
    assert 0 < (l2 - l1) - (l1 - l0) <= 3 * chunks + 1, (l2 - l1, l1 - l0, chunks)
