"""bench.py --dump-outputs: the last timed step of the headline figure, written so that two builds can be compared output for
output.  The CPU tests drive the writer with a stand-in engine; the GPU test runs bench.py and checks the dump against the oracle."""
import os
import subprocess
import sys
import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _FakeEngine:
    """Stands in for Engine.playout(outputs=True): per-game outputs that are a function of the game id."""

    def playout(self, n, seed, first_gid, ruleset):
        gid = first_gid + np.arange(n, dtype=np.int64)
        winner = (gid % 6).astype(np.int8)
        points = ((gid[:, None] + np.arange(6)) % 40).astype(np.int8)
        steps = (300 + gid % 200).astype(np.uint16)
        return dict(winner=winner, points=points, steps=steps, stats=dict(games=n, steps=int(steps.sum()), wins=[1] * 6))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_every_game_or_a_fixed_sample(tmp_path, monkeypatch):
    eng = _FakeEngine()
    stats = eng.playout(40, bench.SEED, 1000, 0)["stats"]
    bench.dump_outputs(eng, str(tmp_path / "all"), 40, 1000, 0, dict(stats, kernel_ms=1.0))
    z = _load(str(tmp_path / "all"))
    assert set(z) == {"game_id", "winner", "points", "steps", "stats_games", "stats_steps", "stats_wins"}
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())
    assert np.array_equal(z["game_id"], 1000 + np.arange(40)) and np.array_equal(z["winner"], np.arange(1000, 1040) % 6)
    assert z["points"].shape == (40, 6) and z["stats_steps"][0] == stats["steps"]

    monkeypatch.setattr(bench, "DUMP_MAX_GAMES", 16)
    for run in ("a", "b"):
        bench.dump_outputs(eng, str(tmp_path / run), 40, 1000, 0, stats)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert all(np.array_equal(a[k], b[k]) for k in a)                      # the same sample every run
    gid = a["game_id"].astype(np.int64)
    assert len(gid) == 16 and np.all(np.diff(gid) > 0) and 1000 <= gid[0] and gid[-1] < 1040
    assert np.array_equal(a["winner"], gid % 6) and np.array_equal(a["steps"], 300 + gid % 200)


def test_dump_refuses_a_replay_that_differs_from_the_timed_step(tmp_path):
    eng = _FakeEngine()
    stats = dict(eng.playout(8, bench.SEED, 0, 0)["stats"], steps=1)
    with pytest.raises(SystemExit, match="differs"):
        bench.dump_outputs(eng, str(tmp_path), 8, 0, 0, stats)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
    assert r.returncode == 2 and "error" in r.stderr


@pytest.mark.gpu
def test_bench_dump_is_what_the_engine_plays(tmp_path):
    """A small bench run: the dump holds the last timed step's games (ids of step K-1), equal to the oracle's playouts."""
    from oracle import citadels_oracle as O
    G, K = 4096, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--games", str(G), "--steps", str(K), "--warmup", "1",
                        "--no-mccfr", "--no-classic", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    z = _load(str(tmp_path))
    assert np.array_equal(z["game_id"], (K - 1) * G + np.arange(G))
    assert z["stats_games"][0] == G and z["stats_steps"][0] == z["steps"].astype(np.int64).sum() and z["stats_errors"][0] == 0
    assert np.array_equal(z["stats_wins"], np.bincount(z["winner"].astype(np.int64), minlength=6))
    for i in range(0, G, G // 4):
        w, pts, steps, _ = O.playout(bench.SEED, int(z["game_id"][i]))
        assert (w, pts, steps) == (int(z["winner"][i]), [int(x) for x in z["points"][i]], int(z["steps"][i])), i
