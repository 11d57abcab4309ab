"""GPU parity tests for the MCCFR path (ctd_make_roots / ctd_mccfr through the C ABI)."""
import numpy as np
import pytest

from tests.mccfr_util import MccfrGolden, oracle_preorder, tree_preorder, assert_same_tree

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=512)
    yield e
    e.close()


@pytest.mark.parametrize("name", ["mccfr_preset.npz", "mccfr_preset_deep_back.npz", "mccfr_classic.npz", "mccfr_random.npz", "mccfr_preset_2000it.npz"])
def test_trees_match_reference(engine, name):
    """SURVEY 8(d) parity gate 3: every node of trees grown by the real reference's CFRNode.cfr_train(200) --
    options, regrets, strategies, values (1e-9 relative; the gate asks 1e-5), game record and knowledge block."""
    G = MccfrGolden(name)
    z = G.z
    engine.load_roots(z["roots"], z["knows"], z["used"], G.gids)
    out = engine.mccfr(G.n, iterations=G.iterations, seed=G.seed, ruleset=G.ruleset, trees=True)
    for r in range(G.n):
        res = out["results"][r]
        if z["terminal"][r]:
            assert res["status"] == 1
            continue
        assert res["status"] == 0, (name, r, int(res["status"]))
        assert_same_tree(G.nodes(r), tree_preorder(out["trees"][r]), (name, r))
        root = next(G.nodes(r))
        k = root["nchild"]
        assert res["n_children"] == k
        n = min(len(root["R"]), 128)   # ctd_mccfr_result keeps CTD_MCCFR_MAX_RESULT children; the trees above compare every array in full
        assert np.allclose(res["cumulative_regrets"][:n], root["R"][:n], rtol=1e-9, atol=1e-12)
        assert np.allclose(res["cumulative_strategy"][:n], root["C"][:n], rtol=1e-9, atol=1e-12)
        assert np.allclose(res["node_value"], root["V"], rtol=1e-9, atol=1e-12)
        if not res["role_pick"] and k:
            # the full child arrays of a root, however many (ctd_mccfr_root_children; a result record stops at 128)
            o, R, S, C = engine.root_children(r, 0, k)
            assert np.array_equal(o, out["trees"][r].children["desc"][:k])
            assert np.allclose(R, root["R"], rtol=1e-9, atol=1e-12) and np.allclose(C, root["C"], rtol=1e-9, atol=1e-12)
            assert np.allclose(S, root["S"], rtol=1e-9, atol=1e-12)


def test_make_roots_matches_oracle(engine):
    """Device root construction (two-pass replay with knowledge of all six observers) vs the oracle."""
    from oracle import mccfr_oracle as M
    seed, gid0, n = 777, 50_000, 48
    from tests.golden_util import visible
    # (ruleset, back_lo, back_hi, flavour): create_a_close_to_finished_game and create_a_random_game, all three rulesets
    for ruleset, lo, hi, flavour in ((0, 0, 20, 0), (0, 1, 100, 1), (1, 0, 60, 0), (2, 0, 80, 0), (2, 1, 100, 1)):
        steps = engine.make_roots(n, seed=seed, first_gid=gid0, ruleset=ruleset, back_lo=lo, back_hi=hi, flavour=flavour)
        roots, knows, used, gids = engine.store_roots(n)
        for i in range(0, n, 3):
            g, st = M.make_root(seed, gid0 + i, ruleset, lo, hi, flavour)
            assert st == int(steps[i]) and int(gids[i]) == gid0 + i
            assert visible(roots[i].tobytes()) == visible(g.pack())
            assert roots[i, 228] == 0
            if not g.terminal:
                assert knows[i].tobytes() == g.pack_know(g.player)
            assert used[i].tobytes() == bytes(g.used_cards) + b"\xff" * (76 - len(g.used_cards))


def test_mccfr_fresh_roots_vs_oracle(engine):
    from oracle import mccfr_oracle as M
    seed, gid0, n, iters = 4242, 90_000, 12, 200
    engine.make_roots(n, seed=seed, first_gid=gid0, ruleset=0, back_lo=0, back_hi=20)
    roots, knows, used, gids = engine.store_roots(n)
    out = engine.mccfr(n, iterations=iters, seed=seed, trees=True)
    for i in range(n):
        res = out["results"][i]
        if roots[i, 217] & 2:
            assert res["status"] == 1
            continue
        node = M.run_from_root(roots[i], knows[i], used[i], seed, int(gids[i]), iters)
        assert res["status"] == 0
        assert_same_tree(oracle_preorder(node), tree_preorder(out["trees"][i]), ("fresh", i))
        assert int(res["rng_draws"]) == node.game.chance.i


def _oracle_root_summary(args):
    """(root R, C, V, number of nodes, draws) of one oracle tree -- runs in a worker process."""
    root, know, used, seed, gid, iters = args
    from oracle import mccfr_oracle as M
    node = M.run_from_root(root, know, used, seed, gid, iters)
    return (np.asarray(node.R, dtype=float).ravel(), np.asarray(node.C, dtype=float).ravel(), np.asarray(node.V, dtype=float),
            sum(1 for _ in node.walk()), node.game.chance.i)


@pytest.mark.parametrize("ruleset,n", [(0, 192), (1, 64), (2, 64)])
def test_mccfr_hundreds_of_fresh_roots_vs_oracle(engine, ruleset, n):
    """The search kernels (preset-specialised and generic) on hundreds of fresh roots: tree size, number of chance draws
    and the root's regrets / cumulative strategy / values against the oracle (process pool on the host cores)."""
    import multiprocessing as mp
    import os
    seed, gid0, iters = 31415 + ruleset, 120_000, 200
    engine.make_roots(n, seed=seed, first_gid=gid0, ruleset=ruleset, back_lo=0, back_hi=40)
    roots, knows, used, gids = engine.store_roots(n)
    res = engine.mccfr(n, iterations=iters, seed=seed, ruleset=ruleset)["results"]
    live = [i for i in range(n) if not (roots[i, 217] & 2)]
    assert all(res[i]["status"] == 1 for i in range(n) if i not in live)
    jobs = [(roots[i], knows[i], used[i], seed, int(gids[i]), iters) for i in live]
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as pool:      # not fork: this process holds a CUDA context
        want = pool.map(_oracle_root_summary, jobs, chunksize=2)
    for i, (R, C, V, nodes, draws) in zip(live, want):
        r = res[i]
        # every non-terminal root completes, as in the reference (run-away hypothetical games of the random rulesets -- cities
        # of 40 districts, purses of thousands -- included: csrc/ctd_engine.cuh container capacities)
        assert r["status"] == 0 and int(r["n_nodes"]) == nodes and int(r["rng_draws"]) == draws, (ruleset, i)
        k = min(len(R), 60 if r["role_pick"] else 128)
        assert np.allclose(r["cumulative_regrets"][:k], R[:k], rtol=1e-9, atol=1e-12), (ruleset, i)
        assert np.allclose(r["cumulative_strategy"][:k], C[:k], rtol=1e-9, atol=1e-12), (ruleset, i)
        assert np.allclose(r["node_value"], V, rtol=1e-9, atol=1e-12), (ruleset, i)


def test_roots_the_fixed_pool_refused_now_complete(engine):
    """The two preset roots of the 8-GPU driver run of round 1 that ended with status 2 (more than 8 nodes per iteration:
    gids 11543 and 14440 under seed 0xC17ADE15, roots stepped back 0..20) and neighbours, against the oracle."""
    from oracle import mccfr_oracle as M
    seed = 0xC17ADE15
    for gid0 in (11540, 14436):
        engine.make_roots(8, seed=seed, first_gid=gid0, back_lo=0, back_hi=20)
        roots, knows, used, gids = engine.store_roots(8)
        out = engine.mccfr(8, iterations=200, seed=seed, trees=True)
        assert int(out["results"]["n_nodes"].max()) > 2112          # what the fixed pool of round 1 held
        for i in range(8):
            assert out["results"][i]["status"] in (0, 1)
            if out["results"][i]["n_nodes"] > 2112:
                node = M.run_from_root(roots[i], knows[i], used[i], seed, int(gids[i]), 200)
                assert_same_tree(oracle_preorder(node), tree_preorder(out["trees"][i]), ("big", gid0 + i))


def test_roots_the_knowledge_block_refused_now_complete(engine):
    """Two Game(preset=False) roots whose hypothetical games collect more than 32 hand-knowledge entries (status 4 while the
    knowledge block held 32 of them), against the oracle."""
    from oracle import mccfr_oracle as M
    seed = 0xC17ADE15
    for gid in (7003168, 7006460):
        engine.make_roots(1, seed=seed, first_gid=gid, ruleset=2, back_lo=0, back_hi=20)
        roots, knows, used, gids = engine.store_roots(1)
        out = engine.mccfr(1, iterations=200, seed=seed, ruleset=2, trees=True)
        assert out["results"][0]["status"] == 0
        tv = out["trees"][0]
        assert int(tv.nodes["know"]["n_hk"].max()) > 32
        node = M.run_from_root(roots[0], knows[0], used[0], seed, int(gids[0]), 200)
        assert_same_tree(oracle_preorder(node), tree_preorder(tv), ("busy seer", gid))


def test_exhausted_arena_is_retried(engine, monkeypatch):
    """Tree memory: with the first arena squeezed to a sliver most trees find it exhausted; the engine searches them again from
    further arenas and the call returns the same trees as an unconstrained run."""
    n = 96
    engine.make_roots(n, seed=99, first_gid=7000, back_lo=0, back_hi=20)
    want = engine.mccfr(n, iterations=200, seed=99)["results"]
    monkeypatch.setenv("CTD_ARENA0_BYTES", str(24 << 20))
    got = engine.mccfr(n, iterations=200, seed=99)["results"]
    monkeypatch.delenv("CTD_ARENA0_BYTES")
    assert (got["status"] <= 1).all()
    for f in ("status", "n_nodes", "rng_draws", "n_children", "cumulative_regrets", "cumulative_strategy", "node_value"):
        assert np.array_equal(got[f], want[f]), f


def test_result_records_keep_nothing_of_an_earlier_call(engine):
    """A record's arrays hold the root's first children only (all 60 entries at a role pick); everything after them, and every
    array of a root without children, is zero, whatever the same slots held in the previous call."""
    n = 64
    engine.make_roots(n, seed=808, first_gid=3000, back_lo=0, back_hi=300, flavour=1)
    before = engine.mccfr(n, iterations=50, seed=808)["results"]
    engine.make_roots(n, seed=909, first_gid=4000, back_lo=0, back_hi=20)
    res = engine.mccfr(n, iterations=50, seed=909)["results"]

    def used(r):
        k = min(int(r["n_children"]), 128)
        return k, (60 if r["role_pick"] else k) if k else 0
    assert any(used(a)[1] > used(b)[1] for a, b in zip(before, res))   # the earlier call left longer arrays in some slots
    for i, r in enumerate(res):
        k, na = used(r)
        assert not r["options"][k:].any(), (i, "options")
        for f in ("cumulative_regrets", "strategy", "cumulative_strategy"):
            assert not r[f][na:].any(), (i, f)


@pytest.mark.parametrize("backend", ["fused", "fp32", "tcgen05"])
def test_exhausted_arena_is_retried_deep(engine, monkeypatch, backend):
    """The same for deep MCCFR on each backend: a retry pass of fewer than 1024 trees runs as one group, its model evaluated over
    every root's row with the pending mask picking the retried trees' leaves (tests/test_gpu_value_waves.py: more than 1024)."""
    from citadels_self_play_b200.value_model import ValueOnlyNN
    import torch
    n = 96
    engine.make_roots(n, seed=99, first_gid=7000, back_lo=0, back_hi=20)
    torch.manual_seed(0)
    engine.set_value_model(ValueOnlyNN(418, 512).eval())
    engine.set_value_backend(backend)
    try:
        want = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=99)["results"]
        monkeypatch.setenv("CTD_ARENA0_BYTES", str(24 << 20))
        got = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=99)["results"]
        monkeypatch.delenv("CTD_ARENA0_BYTES")
    finally:
        engine.set_value_backend("fused")      # back to the default
    assert (got["status"] <= 1).all()
    for f in ("status", "n_nodes", "rng_draws", "n_children", "live_option", "cumulative_regrets", "cumulative_strategy", "node_value"):
        assert np.array_equal(got[f], want[f]), f


# ---------------------------------------------------------------- deep MCCFR (config 4)
def _model(seed=0, randomize_bn=False):
    import torch
    from citadels_self_play_b200.value_model import ValueOnlyNN
    torch.manual_seed(seed)
    m = ValueOnlyNN(418, 512).eval()
    if randomize_bn:   # exercise the BatchNorm folding with non-trivial statistics
        with torch.no_grad():
            for bn in (m.bn1, m.bn2):
                bn.running_mean.normal_(0, 0.3)
                bn.running_var.uniform_(0.5, 2.0)
                bn.weight.uniform_(0.5, 1.5)
                bn.bias.normal_(0, 0.2)
    return m


@pytest.mark.parametrize("backend", ["tcgen05", "fp32"])
@pytest.mark.parametrize("randomize_bn", [False, True])
def test_value_kernel_vs_torch_fp32(engine, randomize_bn, backend):
    """ValueOnlyNN forward + square_and_normalize * 5: both kernel families (tcgen05 tensor cores with 3xTF32 split
    precision; fp32 CUDA cores) vs torch fp32 on the CPU (the reference's own arithmetic), tolerance 1e-5 relative
    (north_star)."""
    from citadels_self_play_b200.value_model import reference_value
    m = _model(3, randomize_bn)
    engine.set_value_model(m)
    engine.set_value_backend(backend)
    engine.make_roots(256, seed=11, first_gid=0, back_lo=0, back_hi=300)
    feats = engine.encode(256)
    got = engine.value_eval(feats)
    want = reference_value(m, feats)
    # fp32 CUDA cores: 1e-5 relative elementwise.  Tensor cores: 1e-5 of the output scale (5); the residual is the
    # tcgen05 instruction's internal summation, see profiles/r01_value_tc_accuracy.md
    if backend == "fp32":
        assert np.allclose(got, want, rtol=1e-5, atol=1e-6), np.abs(got - want).max()
    else:
        assert np.abs(got - want).max() <= 1e-5 * 5.0, np.abs(got - want).max()
    assert np.allclose(got.sum(1), 5.0, rtol=1e-5)
    x = np.random.RandomState(1).randn(300, 418).astype(np.float32)      # arbitrary (not integer) inputs, ragged M
    assert np.abs(engine.value_eval(x) - reference_value(m, x)).max() <= 1e-5 * 5.0
    engine.set_value_backend("fused")      # back to the default


def test_encoder_vs_oracle(engine):
    """Game.encode_game on device vs the oracle, exact (small integers in fp32)."""
    from oracle import citadels_oracle as O
    n = 96
    engine.make_roots(n, seed=21, first_gid=500, back_lo=0, back_hi=400)
    roots, knows, used, gids = engine.store_roots(n)
    feats = engine.encode(n)
    for i in range(n):
        g = O.Game.unpack(roots[i].tobytes())
        g.unpack_know(knows[i], used[i])
        want = np.asarray(g.encode_game(5 if g.state == 0 else None), dtype=np.float32)
        assert np.array_equal(feats[i], want), i


@pytest.mark.parametrize("backend", ["tcgen05", "fused"])
@pytest.mark.parametrize("name", ["deep_mccfr_preset.npz", "deep_mccfr_classic.npz", "deep_mccfr_random.npz"])
def test_deep_trees_match_reference(engine, name, backend):
    """Config 4: deep MCCFR, 200 iterations, value model at depth 10 -- every node against the real reference's
    cfr_pred trees (preset eight, classic eight, random 24-character rulesets).  Structure, options, game records and
    knowledge exact; regrets / strategies / values to 1e-5 of each array's scale (gate 3), the slack being fp32
    summation order in the value model (torch CPU GEMV vs the kernel)."""
    G = MccfrGolden(name)
    z = G.z
    engine.set_value_model(_model(0))
    engine.set_value_backend(backend)
    engine.load_roots(z["roots"], z["knows"], z["used"], G.gids)
    out = engine.mccfr_pred(G.n, iterations=G.iterations, max_depth=int(z["max_depth"]), seed=G.seed, ruleset=G.ruleset,
                            trees=True)
    engine.set_value_backend("fused")      # back to the default
    assert out["waves"] >= 2 if backend != "fused" else out["waves"] == 1   # fused: one launch, every warp evaluates its own leaves
    for r in range(G.n):
        if z["terminal"][r]:
            assert out["results"][r]["status"] == 1
            continue
        assert out["results"][r]["status"] == 0
        assert_same_tree(G.nodes(r), tree_preorder(out["trees"][r]), ("deep", r), norm_rtol=1e-5)



def test_fused_deep_mccfr_equals_the_batched_fp32_path(engine):
    """Fused deep MCCFR (one launch, per-warp leaf evaluation) and the wave scheduler with the fp32 batch kernel run the same
    fp32 arithmetic term for term: identical trees, bit for bit, on 256 fresh roots."""
    n = 256
    engine.set_value_model(_model(5, randomize_bn=True))
    engine.make_roots(n, seed=1234, first_gid=40_000, back_lo=0, back_hi=60)
    engine.set_value_backend("fp32")
    a = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=1234)
    engine.set_value_backend("fused")
    b = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=1234)
    engine.set_value_backend("fused")      # back to the default
    assert a["waves"] > 2 and b["waves"] == 1
    for f in ("status", "n_nodes", "rng_draws", "n_children", "live_option", "node_value", "cumulative_regrets", "cumulative_strategy"):
        assert np.array_equal(a["results"][f], b["results"][f]), f


# ---------------------------------------------------------------- training targets (BASELINE configs[4])
@pytest.mark.parametrize("name", ["mccfr_preset.npz", "mccfr_preset_2000it.npz", "mccfr_classic.npz"])
def test_training_targets_match_reference(engine, name):
    """CFRNode.get_all_targets() of the real reference (tuple format of generate_test_data.py:25) vs ctd_mccfr_targets:
    features and option encodings exact, node values and regret rows to 1e-9."""
    from citadels_self_play_b200 import Engine
    G = MccfrGolden(name)
    z = G.z
    engine.load_roots(z["roots"], z["knows"], z["used"], G.gids)
    engine.mccfr(G.n, iterations=G.iterations, seed=G.seed, ruleset=G.ruleset)
    t = engine.mccfr_targets(G.n, iterations=G.iterations, seed=G.seed, ruleset=G.ruleset)
    assert len(t["meta"]) == int(z["t_off"][-1])
    assert np.array_equal(np.bincount(t["meta"]["tree"], minlength=G.n), np.diff(z["t_off"]))
    assert np.array_equal(t["features"], z["t_feat"])
    assert np.array_equal(t["meta"]["n_options"], z["t_k"])
    assert np.allclose(t["meta"]["node_value"], z["t_val"], rtol=1e-12)
    assert np.allclose(t["regrets"], z["t_dist"], rtol=1e-9, atol=1e-12)
    tuples = Engine.targets_as_tuples(t)
    got = np.concatenate([x[1][0].numpy() for x in tuples]) if tuples else np.zeros((0, 131), np.float32)
    assert got.shape == z["t_opts"].shape
    assert np.array_equal(got, z["t_opts"])
    if tuples:
        mi, oi, nv, dd = tuples[0]
        assert mi.shape == (418,) and oi.shape[0] == 1 and oi.shape[2] == 131 and nv.shape == (6,) and dd.shape == (oi.shape[1],)
