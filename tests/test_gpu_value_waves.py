"""Batched leaf evaluation and the deep-MCCFR wave scheduler at the sizes they really run at.

A. A float64 reference of the value model (on the engine's own folded fp32 weights) and a per-element bound on the rounding error
   of an fp32 evaluation; the bound is checked on the CPU against two fp32 evaluations, torch and numpy.
B. The batch kernels (ctd_k_value_mlp, and ctd_k_linear_tc_tma x3 + ctd_k_value_head) through Engine.value_eval against that
   reference at the batch sizes the scheduler produces, around the 16-row and 128-row tiles; a row's value must not depend on
   the batch it is in.
C. The wave scheduler with two groups of trees on two streams (n >= 1024), retry passes of more than 1024 trees, and the arena's
   value-model slots through the two-group path.
"""
import json

import numpy as np
import pytest

from tests.test_gpu_mccfr import _model

U = 2.0 ** -24          # unit roundoff of fp32
CAPACITY = 4100         # engine slots: the largest batch of B; C's calls up to 2048 roots and the 2048-game arena
BATCH_SIZES = (1, 2, 15, 16, 17, 31, 127, 128, 129, 255, 257, 513, 1023, 1024, 1025, CAPACITY)
INPUTS = ("roots", "normal", "wide", "tf32", "zeros")
MODELS = ("init", "bn", "trained")
# a kernel's max / p99 error against float64 may be this many times torch fp32's on the same rows.  fp32 rounds to nearest once
# per fma, as torch does (measured 0.9 - 1.7x over the sweeps on a B200).  The tcgen05 accumulator truncates once per MMA
# instruction at the accumulator's magnitude (ctd_value_tc.cuh), so its errors share a sign and grow with K instead of partly
# cancelling: measured 1.6 - 4.7x, the max 1.1e-5 at weight 5 that profiles/r01_value_tc_accuracy.md documents.  What the gate
# is for stays far outside either factor: one TF32 pass is ~1e-3 off, a lost 32-wide K slice more.
SENSITIVITY = dict(fp32=4.0, tcgen05=8.0)
SEARCH_FIELDS = ("status", "n_nodes", "rng_draws", "n_children", "live_option", "node_value", "cumulative_regrets",
                 "cumulative_strategy")


# ---------------------------------------------------------------- A. float64 reference and error bound
def _pad448(x, dtype):
    out = np.zeros((len(x), 448), dtype=dtype)
    out[:, :np.shape(x)[1]] = x
    return out


def _forward64(arrs, x):
    """fc4's output y [M, 6] in float64 from the folded fp32 weights, and e [M, 6], a bound on |y computed in fp32 - y|.
    Per layer l of fan-in K: magnitudes m = |W|^T |h| + |b|, errors e_l = |W|^T e_(l-1) + (K + 1) 2u m (K products, the bias,
    one rounding each; 2u rather than u for the tensor cores' accumulator, which truncates, ctd_value_tc.cuh).  ReLU is
    1-Lipschitz and adds nothing; a unit whose pre-activation lies below -e is zero either way and passes on no error.
    A worst case over every sign: looser than the errors seen by some orders of magnitude (test_batch_kernels_vs_float64's
    sensitivity gate is the close one)."""
    h = _pad448(x, np.float64)
    e = np.zeros_like(h)
    w1t, b1, w2t, b2, w3t, b3, w4t, b4 = [np.asarray(a, dtype=np.float64) for a in arrs]
    for layer, (w, b) in enumerate(((w1t, b1), (w2t, b2), (w3t, b3), (w4t, b4))):
        aw = np.abs(w)
        e = e @ aw + (w.shape[0] + 1) * 2 * U * (np.abs(h) @ aw + np.abs(b))
        h = h @ w + b
        if layer < 3:
            e = np.where(h + e < 0, 0.0, e)
            h = np.maximum(h, 0.0)
    return h, e


def ref64(arrs, x, weight):
    """weight * y^2 / sum(y^2) of value_model.fold(model)'s fp32 weights, evaluated in float64."""
    y, _ = _forward64(arrs, x)
    y2 = y * y
    return weight * y2 / y2.sum(1, keepdims=True)


def bound64(arrs, x, weight):
    """Per element: how far an fp32 evaluation of the same weights may lie from ref64.
    p_j = y_j^2 / S moves by sum_k (2 |y_k| / S) |delta_jk - p_j| e_k to first order, doubled for the higher orders; the output
    stage adds nine roundings of at most u relative to p_j <= 1 (six squares and sums, the division, the product with the
    weight; counted as ten)."""
    y, e = _forward64(arrs, x)
    y2 = y * y
    s = y2.sum(1, keepdims=True)
    p = y2 / s
    c = 2 * np.abs(y) / s * e
    dp = c * (1 - 2 * p) + p * c.sum(1, keepdims=True)     # = sum_k c_k |delta_jk - p_j|
    return 2 * weight * dp + weight * 10 * U


def torch32(arrs, x, weight):
    """The yardstick: a plain torch fp32 Linear stack on the same folded weights, then square_and_normalize * weight in fp32."""
    import torch
    import torch.nn.functional as F
    t = [torch.from_numpy(np.asarray(a)) for a in arrs]
    h = torch.from_numpy(_pad448(x, np.float32))
    with torch.no_grad():
        for layer in range(4):
            h = F.linear(h, t[2 * layer].T, t[2 * layer + 1])
            if layer < 3:
                h = torch.relu(h)
        y2 = h * h
        return (np.float32(weight) * (y2 / y2.sum(1, keepdim=True))).numpy()


def numpy32(arrs, x, weight):
    h = _pad448(x, np.float32)
    for layer in range(4):
        h = h @ arrs[2 * layer] + arrs[2 * layer + 1]
        if layer < 3:
            h = np.maximum(h, np.float32(0))
    y2 = h * h
    return np.float32(weight) * (y2 / y2.sum(1, keepdims=True))


def _inputs(kind, n, seed=0, roots=None):
    """n rows of input class `kind`: encoded root features (given), N(0, 1), +-10^U(-4, 3) within one row (the three-term
    TF32 split at full stretch), N(0, 1) rounded to TF32 (the split's residual terms are zero), all zero (biases only)."""
    rs = np.random.RandomState(seed)
    if kind == "roots":
        return roots[rs.permutation(len(roots))[:n]].astype(np.float32)
    if kind == "normal":
        return rs.randn(n, 418).astype(np.float32)
    if kind == "wide":
        return (np.where(rs.rand(n, 418) < 0.5, -1.0, 1.0) * 10.0 ** rs.uniform(-4, 3, (n, 418))).astype(np.float32)
    if kind == "tf32":
        x = rs.randn(n, 418).astype(np.float32)
        return (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)     # 10 explicit mantissa bits
    if kind == "zeros":
        return np.zeros((n, 418), dtype=np.float32)
    raise ValueError(kind)


def _make_model(name):
    if name == "init":
        return _model(3)
    if name == "bn":
        return _model(5, randomize_bn=True)
    from tests.test_value_checkpoint import load
    return load()[1]


def _stats(err):
    return float(err.max()), float(np.quantile(err, 0.99))


@pytest.mark.parametrize("model_name", MODELS)
def test_the_bound_holds_for_fp32_on_the_cpu(model_name):
    """Every element of two fp32 evaluations (torch's Linear stack, numpy's matmul) lies within bound64 of ref64, for every input
    class of the GPU sweeps and both reward weights: a bound that is too tight fails here before it judges a kernel."""
    from citadels_self_play_b200.value_model import fold
    from tests.test_value_checkpoint import load
    arrs = fold(_make_model(model_name))
    roots = load()[0]["features"].astype(np.float32)       # 1000 encoded game states
    for kind in INPUTS:
        x = _inputs(kind, 1000, seed=7, roots=roots)
        for weight in (5.0, 1.0):
            ref, bnd = ref64(arrs, x, weight), bound64(arrs, x, weight)
            assert np.all(np.isfinite(ref)) and np.all(bnd > 0)
            for name, got in (("torch", torch32(arrs, x, weight)), ("numpy", numpy32(arrs, x, weight))):
                err = np.abs(got.astype(np.float64) - ref)
                ratio = float((err / bnd).max())
                print(json.dumps(dict(model=model_name, inputs=kind, weight=weight, yardstick=name, max_err=float(err.max()),
                                      bound_median=float(np.median(bnd)), worst_err_over_bound=ratio)))
                assert ratio <= 1.0, (model_name, kind, weight, name, ratio)


# ---------------------------------------------------------------- B. the batch kernels against float64
@pytest.fixture(scope="module")
def engine():
    from citadels_self_play_b200 import Engine
    e = Engine(capacity=CAPACITY)
    yield e
    e.close()


@pytest.fixture(scope="module")
def root_features(engine):
    """Encoded features of CAPACITY real roots, the three rulesets in equal parts."""
    parts = []
    for ruleset in (0, 1, 2):
        n = (CAPACITY + 2) // 3
        engine.make_roots(n, seed=515 + ruleset, first_gid=30_000, ruleset=ruleset, back_lo=0, back_hi=300)
        parts.append(engine.encode(n))
    return np.concatenate(parts)[:CAPACITY]


_cache = {}


def _sweep_reference(model_name, kind, roots):
    """(folded weights, inputs [CAPACITY], ref64 and bound64 at weight 1, torch fp32 p) of one model and input class."""
    key = (model_name, kind)
    if key not in _cache:
        from citadels_self_play_b200.value_model import fold
        arrs = fold(_make_model(model_name))
        x = _inputs(kind, CAPACITY, seed=11, roots=roots)
        _cache[key] = (arrs, x, ref64(arrs, x, 1.0), bound64(arrs, x, 1.0), torch32(arrs, x, 1.0))
    return _cache[key]


@pytest.mark.gpu
@pytest.mark.parametrize("weight", [5.0, 1.0])
@pytest.mark.parametrize("kind", INPUTS)
@pytest.mark.parametrize("model_name", MODELS)
@pytest.mark.parametrize("backend", ["fp32", "tcgen05"])
def test_batch_kernels_vs_float64(engine, root_features, backend, model_name, kind, weight):
    """value_eval on the first M rows for every M of BATCH_SIZES.  Hard gate: every element within bound64.  Sensitivity gate:
    max and p99 of |got - ref64| over the sweep at most SENSITIVITY[backend] times torch fp32's on the same rows (floor:
    u * weight), which a degraded split or a lost K slice would break long before the worst-case bound does."""
    arrs, x, ref1, bnd1, t1 = _sweep_reference(model_name, kind, root_features)
    engine.set_value_model(_make_model(model_name))
    engine.set_value_backend(backend)
    ref, bnd = weight * ref1, weight * bnd1
    yard = np.float32(weight) * t1
    errs, yard_errs, worst = [], [], 0.0
    for m in BATCH_SIZES:
        got = engine.value_eval(x[:m], weight=weight).astype(np.float64)
        err = np.abs(got - ref[:m])
        over = err > bnd[:m]
        assert not over.any(), (backend, model_name, kind, weight, m, "rows", np.unique(np.nonzero(over)[0])[:8].tolist(),
                                float((err / bnd[:m]).max()))
        worst = max(worst, float((err / bnd[:m]).max()))
        errs.append(err.ravel())
        yard_errs.append(np.abs(yard[:m].astype(np.float64) - ref[:m]).ravel())
    k_max, k_p99 = _stats(np.concatenate(errs))
    t_max, t_p99 = _stats(np.concatenate(yard_errs))
    floor = U * weight
    rep = dict(backend=backend, model=model_name, inputs=kind, weight=weight, worst_err_over_bound=worst, max_err=k_max,
               p99_err=k_p99, torch_max_err=t_max, torch_p99_err=t_p99, max_ratio=k_max / max(t_max, floor),
               p99_ratio=k_p99 / max(t_p99, floor))
    print("value_waves_sweep " + json.dumps(rep))
    assert rep["max_ratio"] <= SENSITIVITY[backend] and rep["p99_ratio"] <= SENSITIVITY[backend], rep


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["fp32", "tcgen05"])
def test_a_row_does_not_depend_on_its_batch(engine, root_features, backend):
    """Bit for bit: row i of a batch of 1025 == the same row alone == the same row at another offset of a batch of another size,
    for rows on both sides of the 16-row (fp32) and 128-row (tcgen05) tile boundaries.  The wave scheduler relies on it: a
    retry pass evaluates a tree's leaves in batches other than the first pass's."""
    engine.set_value_model(_model(5, randomize_bn=True))
    engine.set_value_backend(backend)
    rs = np.random.RandomState(3)
    x = np.concatenate([root_features[:700], rs.randn(325, 418).astype(np.float32)])
    x = x[rs.permutation(len(x))]
    full = engine.value_eval(x)
    for i in (0, 1, 14, 15, 16, 17, 126, 127, 128, 129, 255, 256, 511, 512, 1023, 1024):
        alone = engine.value_eval(x[i:i + 1])
        assert np.array_equal(alone[0], full[i]), (backend, i, "alone")
        size = 129 + 97 * (i % 7)
        at = (i * 37 + 5) % size
        other = rs.randn(size, 418).astype(np.float32)
        other[at] = x[i]
        assert np.array_equal(engine.value_eval(other)[at], full[i]), (backend, i, "at", at, "of", size)


# ---------------------------------------------------------------- C. the wave scheduler past 1024 trees
@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 2])
@pytest.mark.parametrize("n", [1024, 1031, 2048])
def test_fused_equals_fp32_waves_in_two_groups(engine, n, ruleset):
    """n >= 1024 roots: the wave scheduler splits the trees into two groups on two streams (1031: groups of 520 and 511).  Fused
    deep MCCFR and the fp32 batch kernel run the same arithmetic term for term, so the trees are identical bit for bit; ruleset 0
    takes the preset-specialised search kernel, ruleset 2 the generic one."""
    engine.set_value_model(_model(5, randomize_bn=True))
    seed = 2718 + n + ruleset
    engine.make_roots(n, seed=seed, first_gid=70_000, ruleset=ruleset, back_lo=0, back_hi=60)
    engine.set_value_backend("fp32")
    a = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=seed, ruleset=ruleset)
    engine.set_value_backend("fused")
    b = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=seed, ruleset=ruleset)
    assert a["waves"] > 2 and b["waves"] == 1
    assert (a["results"]["status"] <= 1).all() and (a["results"]["status"] == 0).any()
    for f in SEARCH_FIELDS:
        assert np.array_equal(a["results"][f], b["results"][f]), (n, ruleset, f)


@pytest.mark.gpu
@pytest.mark.parametrize("ruleset", [0, 2])
def test_tcgen05_two_groups_equal_two_calls_of_one_group(engine, ruleset):
    """1031 roots in one tcgen05 call (two groups of 520 and 511 trees on two streams, each group's leaves in batches of its own)
    == the same roots searched in two calls of 520 and 511 (one group each): trees are functions of (seed, root, gid) and a row's
    value does not depend on its batch, so bit for bit."""
    n, m = 1031, 520
    engine.set_value_model(_model(5, randomize_bn=True))
    engine.set_value_backend("tcgen05")
    seed = 1618 + ruleset
    engine.make_roots(n, seed=seed, first_gid=80_000, ruleset=ruleset, back_lo=0, back_hi=60)
    roots, knows, used, gids = engine.store_roots(n)
    whole = engine.mccfr_pred(n, iterations=200, max_depth=10, seed=seed, ruleset=ruleset)
    parts = []
    for lo, hi in ((0, m), (m, n)):
        engine.load_roots(roots[lo:hi], knows[lo:hi], used[lo:hi], gids[lo:hi])
        parts.append(engine.mccfr_pred(hi - lo, iterations=200, max_depth=10, seed=seed, ruleset=ruleset)["results"])
    engine.set_value_backend("fused")
    want = np.concatenate(parts)
    assert whole["waves"] > 2 and (whole["results"]["status"] <= 1).all()
    for f in SEARCH_FIELDS:
        assert np.array_equal(whole["results"][f], want[f]), (ruleset, f)


RETRY_N, RETRY_ITERATIONS, RETRY_DEPTH, RETRY_CHUNKS = 1152, 50, 3, 64


def _retry_run(e, backend, seed, arena0, monkeypatch):
    e.set_value_backend(backend)
    if arena0 is not None:
        monkeypatch.setenv("CTD_ARENA0_BYTES", str(arena0))
    try:
        return e.mccfr_pred(RETRY_N, iterations=RETRY_ITERATIONS, max_depth=RETRY_DEPTH, seed=seed)["results"]
    finally:
        monkeypatch.delenv("CTD_ARENA0_BYTES", raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["fp32", "tcgen05", "fused"])
def test_a_retry_of_more_than_1024_trees(backend, monkeypatch):
    """The first arena squeezed to RETRY_CHUNKS first chunks: every tree claims its first chunk when it starts, so at least
    RETRY_N - RETRY_CHUNKS = 1088 trees find the arena exhausted and are searched again in one retry pass.  A retry pass indexes
    its feature / pending / prediction rows by root, so it must run as one group of trees: two groups on two streams would
    evaluate, and overwrite, each other's rows.  The results equal the unconstrained run's bit for bit, and the fp32 waves equal
    the fused search."""
    from citadels_self_play_b200 import Engine
    seed = 4242
    e = Engine(capacity=RETRY_N)
    try:
        e.set_value_model(_model(5, randomize_bn=True))
        e.make_roots(RETRY_N, seed=seed, first_gid=90_000, back_lo=1, back_hi=60)
        n0, node_bytes, _ = e.tree_shape(RETRY_ITERATIONS)
        arena0 = RETRY_CHUNKS * n0 * node_bytes
        budget = e.tree_shape(RETRY_ITERATIONS)[2] - (64 << 20)        # ctd_tree_budget: arena bytes per tree
        retry_bytes = budget * 16 * (RETRY_N - RETRY_CHUNKS) + (64 << 20)
        print("value_waves_retry " + json.dumps(dict(backend=backend, trees=RETRY_N, first_arena_bytes=arena0,
                                                     retried_at_least=RETRY_N - RETRY_CHUNKS, retry_arena_bytes=retry_bytes)))
        want = _retry_run(e, backend, seed, None, monkeypatch)
        got = _retry_run(e, backend, seed, arena0, monkeypatch)
        assert (got["status"] <= 1).all() and (got["status"] == 0).sum() >= 1024 + RETRY_CHUNKS   # >= 1024 trees retried
        for f in SEARCH_FIELDS:
            assert np.array_equal(got[f], want[f]), (backend, f, int((got[f] != want[f]).reshape(RETRY_N, -1).any(1).sum()))
        if backend == "fp32":
            fused = _retry_run(e, "fused", seed, None, monkeypatch)
            for f in SEARCH_FIELDS:
                assert np.array_equal(got[f], fused[f]), ("fp32 vs fused", f)
    finally:
        e.close()


@pytest.mark.gpu
def test_arena_model_slots_through_two_groups(engine):
    """2048 arena games, deep seats on value-model slots 1 (four seats) and 0 (one), one random seat: in the first decision
    rounds slot 1's search group holds well over 1024 games, so its searches take the two-group path with sp.model = 1.  The fp32
    waves and the fused search give identical games and final records."""
    from citadels_self_play_b200 import arena
    from tests.test_value_checkpoint import load
    n, seed = 2048, 0x5EA7
    engine.set_value_model(load()[1], slot=0)
    engine.set_value_model(_model(7), slot=1)
    d0, d1 = arena.deep(10, 3, 5.0, model=0), arena.deep(10, 3, 5.0, model=1)
    seats = [d1, d1, d0, d1, d1, arena.random_seat()]
    out = {}
    for backend in ("fp32", "fused"):
        engine.set_value_backend(backend)
        out[backend] = engine.arena(n, seats, seed=seed, first_gid=5000)
        out[backend]["finals"] = engine.store_states(n)
    a, b = out["fp32"], out["fused"]
    assert a["stats"]["errors"] == 0 and sum(a["stats"]["wins"]) == n and a["searches"].min() > 0
    for k in ("winner", "points", "steps", "searches", "finals"):
        assert np.array_equal(a[k], b[k]), k
    assert a["stats"] == b["stats"]
