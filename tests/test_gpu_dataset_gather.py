"""ctd_dataset_append / Engine.dataset_append, dataset_tensors, save_dataset / load_dataset: datasets recorded by separate engines and
put together equal the dataset of one engine recording every game, and train to the same weights."""
import numpy as np
import pytest

from tests.test_gpu_arena_record import _checkpoint, _same_record, _by_tree

pytestmark = pytest.mark.gpu

SEED = 0x6A7E55
G = 600   # first game id
RECORDED = [0, 1, 3, 5]


def _seats():
    from citadels_self_play_b200 import arena
    return [arena.deep(20, 10, 5.0), arena.pure(40), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.deep(20, 10, 5.0)]


def _recorded(first_gid, n, mode, device=0, reserve=(100_000, 2_000_000)):
    """a new engine on `device` whose dataset holds the records of games [first_gid, first_gid + n) -> (engine, arena result)"""
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=16, device=device)
    e.set_value_model(_checkpoint())
    e.dataset_reserve(*reserve)
    out = e.arena(n, _seats(), seed=SEED, first_gid=first_gid, record=(RECORDED, mode, 15.0))
    return e, out


def _snapshot(e):
    return e.dataset_info(), {k: v.tobytes() for k, v in e.dataset_arrays().items()}


def _assert_split_equals_whole(a, c, shifted_from):
    """a's dataset equals c's record for record in canonical order; records of games >= shifted_from carry their own call's tree
    index, 4 below c's"""
    da, dc = a.dataset_read(), c.dataset_read()
    n = len(dc["meta"])
    assert n > 0 and len(da["meta"]) == n
    assert da["origin"].tobytes() == dc["origin"].tobytes()
    for i in range(n):
        _same_record(da, i, dc, i)
        ta, tc = int(da["meta"][i]["tree"]), int(dc["meta"][i]["tree"])
        assert ta == (tc - 4 if int(dc["origin"][i]["gid"]) >= shifted_from else tc), i
    assert _by_tree(da).keys() == _by_tree(dc).keys()
    ia, ic = a.dataset_info(), c.dataset_info()
    assert (ia["records"], ia["option_slots"]) == (ic["records"], ic["option_slots"])


@pytest.mark.parametrize("mode", ["tree", "root"])
def test_split_equals_whole(mode):
    from citadels_self_play_b200 import selfplay
    code = selfplay.MODES[mode]
    (a, _), (b, _), (c, _) = _recorded(G, 4, code), _recorded(G + 4, 4, code), _recorded(G, 8, code)
    try:
        own = a.dataset_arrays()
        ib = b.dataset_info()
        assert ib["records"] > 0 and a.dataset_info()["records"] > 0
        t = b.dataset_tensors("cuda:0")
        assert t["features"].shape == (ib["records"], 448) and t["options"].shape == (ib["option_slots"],)
        a.dataset_append(*(t[k] for k in ("features", "meta", "origin", "options", "regrets")))
        _assert_split_equals_whole(a, c, G + 4)
        assert a.dataset_info()["dropped_records"] == 0
        # once more from host arrays: A's own records first, then B's
        a.dataset_clear()
        a.dataset_append(**own)
        a.dataset_append(**b.dataset_arrays())
        _assert_split_equals_whole(a, c, G + 4)
        assert b.dataset_info() == ib   # the source is not changed
    finally:
        for e in (a, b, c):
            e.close()


def _train(e, folder):
    import torch
    from citadels_self_play_b200 import selfplay
    from citadels_self_play_b200.value_model import ValueOnlyNN
    d = e.dataset_read()
    tr, va = selfplay.split_by_game(d["origin"], 0.3, seed=3, rows=d["row"])
    where = np.empty(len(d["row"]), dtype=np.int64)
    where[d["row"]] = np.arange(len(d["row"]))
    # winner labels (a root record's node_value can be all zero, which the loss turns into NaN); errored games have none
    decided = d["origin"]["winner"][where] >= 0
    tr, va = tr[decided[tr]], va[decided[va]]
    torch.manual_seed(5)
    h = {}
    best = selfplay.train_on_dataset(e, tr, va, "winner", epochs=3, lr=1e-3, batch_size=32, model=ValueOnlyNN(418, 512), seed=9,
                                     parent_folder=folder, history=h)
    return where[tr], where[va], best, h


def _same_training(x, y):
    assert len(x[0]) > 0 and len(x[1]) > 0
    assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])   # the same records, in canonical order
    assert np.isfinite(x[2]) and x[2] == y[2]
    assert x[3]["train_losses"] == y[3]["train_losses"] and x[3]["eval_losses"] == y[3]["eval_losses"]
    for k, v in y[3]["final_state"].items():
        assert np.array_equal(x[3]["final_state"][k], v), k


@pytest.mark.parametrize("mode", ["tree", "root"])
def test_training_on_the_gathered_dataset_is_bit_identical(mode, tmp_path):
    from citadels_self_play_b200 import selfplay
    code = selfplay.MODES[mode]
    (a, _), (b, _), (c, _) = _recorded(G, 4, code), _recorded(G + 4, 4, code), _recorded(G, 8, code)
    try:
        t = b.dataset_tensors("cuda:0")
        a.dataset_append(t["features"], t["meta"], t["origin"], t["options"], t["regrets"])
        _same_training(_train(a, str(tmp_path / "a")), _train(c, str(tmp_path / "c")))
    finally:
        for e in (a, b, c):
            e.close()


def test_append_is_all_or_nothing():
    from citadels_self_play_b200 import Engine, EngineError
    from citadels_self_play_b200.layout import RECORD_ROOT
    src, _ = _recorded(G, 3, RECORD_ROOT)
    x = src.dataset_arrays()
    src.close()
    n, ns = len(x["meta"]), len(x["options"])
    assert n > 1
    e, _ = _recorded(G + 3, 2, RECORD_ROOT)
    try:
        before = _snapshot(e)
        r0, s0 = before[0]["records"], before[0]["option_slots"]

        def refused(status, **change):
            y = {k: v.copy() for k, v in x.items()}
            y.update(change)
            with pytest.raises(EngineError, match="status %d " % status):
                e.dataset_append(**y)
            assert _snapshot(e) == before

        # too few records, then too few slots
        e.dataset_reserve(r0 + n - 1, s0 + ns)
        e.dataset_append(**_from_snapshot(before))
        before = _snapshot(e)
        refused(3)
        e.dataset_reserve(r0 + n, s0 + ns - 1)
        e.dataset_append(**_from_snapshot(before))
        before = _snapshot(e)
        refused(3)
        e.dataset_reserve(100_000, 2_000_000)
        e.dataset_append(**_from_snapshot(before))
        before = _snapshot(e)
        m = x["meta"].copy()
        m["option_offset"][n - 1] = ns - int(m["n_options"][n - 1]) + 1   # one past the incoming slots
        refused(1, meta=m)
        m = x["meta"].copy()
        m["n_options"][0] = 0
        refused(1, meta=m)
        o = x["origin"].copy()
        o["mover"][1] = 6
        refused(1, origin=o)
        o = x["origin"].copy()
        o["winner"][0] = 7
        refused(1, origin=o)
        lib, h = e._lib, e._h
        assert lib.ctd_dataset_append(h, 1, 1, None, None, None, None, None) == 1
        assert _snapshot(e) == before
        # an empty append does nothing
        e.dataset_append(x["features"][:0], x["meta"][:0], x["origin"][:0], x["options"][:0], x["regrets"][:0])
        assert _snapshot(e) == before
        # and a good one still goes through after all the refusals
        e.dataset_append(**x)
        assert e.dataset_info()["records"] == before[0]["records"] + n
    finally:
        e.close()
    fresh = Engine(capacity=4)
    try:
        with pytest.raises(EngineError, match="status 1 "):
            fresh.dataset_append(**x)
    finally:
        fresh.close()


def _from_snapshot(snap):
    """a _snapshot's arrays back in dataset_arrays' types"""
    from citadels_self_play_b200.layout import TARGET_META_DTYPE, ORIGIN_DTYPE
    b = snap[1]
    return dict(features=np.frombuffer(b["features"], dtype=np.float32).reshape(-1, 448), meta=np.frombuffer(b["meta"], dtype=TARGET_META_DTYPE),
                origin=np.frombuffer(b["origin"], dtype=ORIGIN_DTYPE), options=np.frombuffer(b["options"], dtype=np.uint64),
                regrets=np.frombuffer(b["regrets"], dtype=np.float64))


def test_recording_after_an_append():
    """record, append, record again: each call's records get their own games' outcomes, the appended ones keep theirs"""
    from citadels_self_play_b200.layout import RECORD_ROOT
    seats = _seats()
    other, _ = _recorded(G + 10, 3, RECORD_ROOT)
    appended = other.dataset_read()
    e, first = _recorded(G, 3, RECORD_ROOT)
    try:
        e.dataset_append(**other.dataset_arrays())
        third = e.arena(3, seats, seed=SEED, first_gid=G + 20, record=(RECORDED, RECORD_ROOT, 15.0))
        d = e.dataset_read()
    finally:
        e.close()
        other.close()
    gid = d["origin"]["gid"].astype(np.int64)
    for lo, out in ((G, first), (G + 20, third)):
        sel = np.nonzero((gid >= lo) & (gid < lo + 3))[0]
        assert len(sel) > 0
        for i in sel:
            g = int(gid[i]) - lo
            assert int(d["origin"][i]["winner"]) == int(out["winner"][g])
            assert np.array_equal(d["origin"][i]["points"], out["points"][g])
            assert int(d["meta"][i]["tree"]) == g
    sel = np.nonzero((gid >= G + 10) & (gid < G + 13))[0]
    assert len(sel) == len(appended["meta"]) > 0
    assert d["origin"][sel].tobytes() == appended["origin"].tobytes()
    assert np.array_equal(d["meta"][sel]["tree"], appended["meta"]["tree"])


def test_save_load_round_trip(tmp_path):
    from citadels_self_play_b200 import Engine, selfplay
    from citadels_self_play_b200.layout import RECORD_TREE
    e, _ = _recorded(G, 6, RECORD_TREE)
    f = Engine(capacity=16)
    try:
        path = str(tmp_path / "round_1.npz")
        saved = selfplay.save_dataset(e, path)
        info = e.dataset_info()
        assert saved == dict(records=info["records"], option_slots=info["option_slots"]) and saved["records"] > 0
        f.dataset_reserve(saved["records"] - 1, saved["option_slots"])
        with pytest.raises(ValueError, match="do not fit"):
            selfplay.load_dataset(f, path)
        assert f.dataset_info()["records"] == 0
        f.dataset_reserve(100_000, 2_000_000)
        assert selfplay.load_dataset(f, path) == saved
        de, df = e.dataset_read(), f.dataset_read()
        for k in ("features", "meta", "origin", "row", "options", "regrets"):
            assert de[k].tobytes() == df[k].tobytes(), k
        _same_training(_train(f, str(tmp_path / "f")), _train(e, str(tmp_path / "e")))
    finally:
        e.close()
        f.close()


def test_append_from_another_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    from citadels_self_play_b200.layout import RECORD_ROOT
    (a, _), (b, _), (c, _) = _recorded(G, 4, RECORD_ROOT), _recorded(G + 4, 4, RECORD_ROOT, device=1), _recorded(G, 8, RECORD_ROOT)
    try:
        t = b.dataset_tensors("cuda:1")
        a.dataset_append(t["features"], t["meta"], t["origin"], t["options"], t["regrets"])
        _assert_split_equals_whole(a, c, G + 4)
    finally:
        for e in (a, b, c):
            e.close()
