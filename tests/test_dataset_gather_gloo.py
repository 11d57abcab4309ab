"""selfplay.gather_dataset / save_dataset / load_dataset on CPU: two gloo ranks, each with a numpy stand-in for the engine's dataset
that implements dataset_info / dataset_arrays / dataset_append the way ctd_dataset_append does (capacity check, option offsets
rebased, tree and origin kept)."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from citadels_self_play_b200.engine import DATASET_KEYS
from citadels_self_play_b200.layout import TARGET_META_DTYPE, ORIGIN_DTYPE


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _records(rank, n):
    """n records of made-up data, game ids in a block of the rank's own, option spans laid end to end"""
    rng = np.random.RandomState(7 + rank)
    ks = rng.randint(1, 6, size=n)
    meta = np.zeros(n, dtype=TARGET_META_DTYPE)
    meta["tree"] = rng.randint(0, 50, size=n)
    meta["node"] = np.arange(n)
    meta["n_options"] = ks
    meta["option_offset"] = np.concatenate([[0], np.cumsum(ks)[:-1]]) if n else []
    meta["node_value"] = rng.rand(n, 6)
    origin = np.zeros(n, dtype=ORIGIN_DTYPE)
    origin["gid"] = 1000 * rank + np.arange(n) // 3
    origin["search"] = np.arange(n) % 3
    origin["mover"] = rng.randint(0, 6, size=n)
    origin["winner"] = rng.randint(-1, 6, size=n)
    ns = int(ks.sum())
    return dict(features=rng.rand(n, 448).astype(np.float32), meta=meta, origin=origin,
                options=rng.randint(1, 1 << 40, size=ns).astype(np.uint64), regrets=rng.rand(ns))


class FakeEngine:
    """The dataset side of Engine, in host memory."""
    device = 0

    def __init__(self, max_records, max_slots, data=None, dropped=(0, 0)):
        self.cap = (max_records, max_slots)
        self.data = data or _records(0, 0)
        self.dropped = dropped
        self.appends = 0

    def dataset_info(self):
        return dict(records=len(self.data["meta"]), option_slots=len(self.data["options"]), dropped_trees=self.dropped[0],
                    dropped_records=self.dropped[1], max_records=self.cap[0], max_option_slots=self.cap[1])

    def dataset_arrays(self):
        return {k: v.copy() for k, v in self.data.items()}

    def dataset_append(self, features, meta, origin, options, regrets):
        from citadels_self_play_b200 import EngineError
        n, ns = len(meta), len(options)
        if len(self.data["meta"]) + n > self.cap[0] or len(self.data["options"]) + ns > self.cap[1]:
            raise EngineError("ctd_dataset_append: status 3")
        meta = np.array(meta, dtype=TARGET_META_DTYPE)
        meta["option_offset"] += np.uint32(len(self.data["options"]))
        new = dict(features=np.asarray(features).reshape(n, -1), meta=meta, origin=np.asarray(origin, dtype=ORIGIN_DTYPE),
                   options=np.asarray(options, dtype=np.uint64), regrets=np.asarray(regrets))
        self.data = {k: np.concatenate([self.data[k], new[k]]) for k in DATASET_KEYS}
        self.appends += 1


SIZES = (5, 8)   # records of rank 0 and rank 1


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from citadels_self_play_b200 import selfplay
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = {}
    try:
        # dst 0 with room for everything
        e = FakeEngine(100, 1000, _records(rank, SIZES[rank]), dropped=(rank + 1, 10 * rank))
        out["counts"] = selfplay.gather_dataset(e, dst=0)
        out["dst0"] = (e.data, e.appends)
        # dst 1
        e = FakeEngine(100, 1000, _records(rank, SIZES[rank]))
        selfplay.gather_dataset(e, dst=1)
        out["dst1"] = (e.data, e.appends)
        # dst 0 without room for rank 1's records: both ranks raise, nothing moves
        e = FakeEngine(SIZES[0] + SIZES[1] - 1 if rank == 0 else 100, 1000, _records(rank, SIZES[rank]))
        try:
            selfplay.gather_dataset(e, dst=0)
            out["small"] = None
        except ValueError as x:
            out["small"] = str(x)
        out["small_appends"] = e.appends
        dist.barrier()
    finally:
        dist.destroy_process_group()
    q.put((rank, out))


def _same(a, b):
    for k in DATASET_KEYS:
        assert np.array_equal(a[k], b[k]), k


def _merged(first, second):
    """second's records after first's, offsets rebased"""
    m = second["meta"].copy()
    m["option_offset"] += np.uint32(len(first["options"]))
    s = dict(second, meta=m)
    return {k: np.concatenate([first[k], s[k]]) for k in DATASET_KEYS}


def test_two_rank_gather():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        got = dict(q.get(timeout=180) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    assert all(p.exitcode == 0 for p in procs)
    r0, r1 = _records(0, SIZES[0]), _records(1, SIZES[1])
    for rank in range(world):
        c = got[rank]["counts"]
        assert c["records"] == list(SIZES) and c["option_slots"] == [len(r0["options"]), len(r1["options"])]
        assert c["dropped_trees"] == [1, 2] and c["dropped_records"] == [0, 10]
    # dst 0: its records, then rank 1's with their offsets rebased (tree and origin kept); rank 1 unchanged
    data, appends = got[0]["dst0"]
    assert appends == 1
    _same(data, _merged(r0, r1))
    for i in range(SIZES[1]):
        m, src = data["meta"][SIZES[0] + i], r1["meta"][i]
        o, k = int(m["option_offset"]), int(m["n_options"])
        assert int(m["tree"]) == int(src["tree"])
        assert np.array_equal(data["options"][o:o + k], r1["options"][int(src["option_offset"]):int(src["option_offset"]) + k])
    assert got[1]["dst0"][1] == 0
    _same(got[1]["dst0"][0], r1)
    # dst 1: rank 1's records, then rank 0's
    _same(got[1]["dst1"][0], _merged(r1, r0))
    assert got[0]["dst1"][1] == 0
    _same(got[0]["dst1"][0], r0)
    # no room: the same ValueError on both ranks, nothing appended
    assert got[0]["small"] is not None and got[0]["small"] == got[1]["small"]
    assert "do not fit" in got[0]["small"]
    assert got[0]["small_appends"] == 0 and got[1]["small_appends"] == 0


def test_single_process_gather_is_a_no_op():
    import torch.distributed as dist
    from citadels_self_play_b200 import selfplay
    assert not dist.is_initialized()
    d = _records(0, 4)
    e = FakeEngine(10, 100, d, dropped=(2, 3))
    c = selfplay.gather_dataset(e)
    assert c == dict(records=[4], option_slots=[len(d["options"])], dropped_trees=[2], dropped_records=[3])
    assert e.appends == 0
    _same(e.data, d)


def test_npz_round_trip(tmp_path):
    from citadels_self_play_b200 import selfplay
    src = FakeEngine(10, 100, _records(1, 6))
    path = str(tmp_path / "round_1.npz")
    assert selfplay.save_dataset(src, path) == dict(records=6, option_slots=len(src.data["options"]))
    dst = FakeEngine(20, 200, _records(0, 3))
    assert selfplay.load_dataset(dst, path) == dict(records=6, option_slots=len(src.data["options"]))
    _same(dst.data, _merged(_records(0, 3), src.data))
    empty = FakeEngine(10, 100)
    selfplay.load_dataset(empty, path)
    _same(empty.data, src.data)
    small = FakeEngine(8, 200, _records(0, 3))
    with pytest.raises(ValueError, match="do not fit"):
        selfplay.load_dataset(small, path)
    assert small.appends == 0
    np.savez(str(tmp_path / "other.npz"), format_version=np.int64(99), **src.data)
    with pytest.raises(ValueError, match="format"):
        selfplay.load_dataset(empty, str(tmp_path / "other.npz"))
