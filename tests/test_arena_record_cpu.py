"""Self-play recording without a GPU: the header's new constants and record against their Python mirrors, split_by_game, and the
argument checks of selfplay.record_arena / train_on_dataset, which run before any engine exists."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    return open(os.path.join(ROOT, "include", "citadels_b200.h")).read()


def test_header_constants_match_the_mirrors():
    from citadels_self_play_b200 import layout
    src = _header()
    consts = dict((k, int(v)) for k, v in re.findall(r"#define (CTD_(?:RECORD|LABEL)_\w+) (\d+)", src))
    assert consts == dict(CTD_RECORD_TREE=layout.RECORD_TREE, CTD_RECORD_ROOT=layout.RECORD_ROOT,
                          CTD_LABEL_NODE_VALUE=layout.LABEL_NODE_VALUE, CTD_LABEL_WINNER=layout.LABEL_WINNER)
    body = src[src.index("typedef struct ctd_record_origin {"):src.index("} ctd_record_origin;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b(?:u?int\d+_t)\s+(\w+)(?:\[(\d+)\])?;", body)
    assert [f[0] for f in fields] == list(layout.ORIGIN_DTYPE.names)
    for name, cnt in fields:
        shape = layout.ORIGIN_DTYPE[name].shape
        assert (shape[0] if shape else 1) == (int(cnt) if cnt else 1), name
    from citadels_self_play_b200 import _lib
    assert [f[0] for f in _lib.RecordOpts._fields_] == ["seat_mask", "mode", "threshold"] and ctypes.sizeof(_lib.RecordOpts) == 16


def test_origin_size_matches_the_library():
    import __graft_entry__
    __graft_entry__.build()
    from citadels_self_play_b200 import _lib, layout
    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.ctd_sizeof.restype = ctypes.c_uint32
    assert lib.ctd_sizeof(9) == layout.ORIGIN_DTYPE.itemsize == 24


def _origin(gids_searches):
    from citadels_self_play_b200.layout import ORIGIN_DTYPE
    o = np.zeros(len(gids_searches), dtype=ORIGIN_DTYPE)
    for i, (g, t) in enumerate(gids_searches):
        o[i]["gid"], o[i]["search"] = g, t
    return o


def test_split_by_game():
    from citadels_self_play_b200.selfplay import split_by_game
    rng = np.random.default_rng(0)
    recs = [(int(g), int(t)) for g in range(100, 140) for t in range(int(rng.integers(1, 6))) for _ in range(int(rng.integers(1, 4)))]
    phys = rng.permutation(len(recs))             # physical order is arbitrary
    origin = _origin([recs[i] for i in phys])
    tr, va = split_by_game(origin, 0.25, seed=7)
    assert tr.dtype == np.uint32 and len(tr) + len(va) == len(origin)
    assert not set(tr.tolist()) & set(va.tolist())
    gtr, gva = set(origin["gid"][tr].tolist()), set(origin["gid"][va].tolist())
    assert not gtr & gva and len(gtr) + len(gva) == 40 and len(gva) == 10
    # canonical order: (gid, search), then row
    key = [(int(origin[r]["gid"]), int(origin[r]["search"]), int(r)) for r in tr]
    assert key == sorted(key)
    tr2, va2 = split_by_game(origin, 0.25, seed=7)
    assert np.array_equal(tr, tr2) and np.array_equal(va, va2)
    assert not np.array_equal(va, split_by_game(origin, 0.25, seed=8)[1])
    # the same records given sorted, with their physical rows, split alike
    order = np.lexsort((np.arange(len(origin)), origin["search"], origin["gid"]))
    tr3, va3 = split_by_game(origin[order], 0.25, seed=7, rows=order)
    assert np.array_equal(tr, tr3) and np.array_equal(va, va3)
    assert len(split_by_game(origin, 0.0, seed=1)[1]) == 0
    one = _origin([(5, 0), (5, 1)])
    assert len(split_by_game(one, 0.9, seed=1)[0]) == 2   # a game always stays for training
    with pytest.raises(ValueError):
        split_by_game(origin, 1.0, seed=1)


def test_argument_errors_come_before_any_engine(monkeypatch):
    from citadels_self_play_b200 import arena, selfplay

    class NoEngine:
        def __init__(self, *a, **k):
            raise AssertionError("an engine was created")
    monkeypatch.setattr(selfplay, "Engine", NoEngine)
    seats = [arena.pure(10)] + [arena.random_seat()] * 5
    for kw in (dict(mode="leaf"), dict(mode=2), dict(threshold=-1.0), dict(threshold=float("nan")), dict(record_seats=[6]),
               dict(seats=seats[:5]), dict(seats=[arena.deep(10)] + seats[1:]), dict(max_records=0)):
        args = dict(n_games=4, seats=seats, record_seats=[0])
        args.update(kw)
        with pytest.raises(ValueError):
            selfplay.record_arena(**args)
    for kw in (dict(label="policy"), dict(label=3), dict(train_idx=[]), dict(batch_size=0), dict(epochs=-1), dict()):
        args = dict(engine=None, train_idx=[0, 1], val_idx=[2])
        args.update(kw)
        with pytest.raises(ValueError):
            selfplay.train_on_dataset(**args)
