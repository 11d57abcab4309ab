"""Batch engine: a thin numpy-facing wrapper over the C ABI.  One Engine == one ctd_engine handle ==
`capacity` game slots in HBM on one device."""
import ctypes
import numpy as np

from . import _lib
from .layout import STATE_BYTES, KNOW_BYTES, MCCFR_RESULT_DTYPE, TARGET_META_DTYPE, ORIGIN_DTYPE, TreeView, encode_options

RULESET_PRESET, RULESET_CLASSIC, RULESET_RANDOM = 0, 1, 2
ROOTS_CLOSE_TO_FINISHED, ROOTS_RANDOM_GAME = 0, 1
DEFAULT_SEED = 0xC17ADE15


class EngineError(RuntimeError):
    pass


class Engine:
    def __init__(self, capacity=1024, device=0):
        self._lib = _lib.load()
        h = ctypes.c_void_p()
        st = self._lib.ctd_create(int(device), int(capacity), ctypes.byref(h))
        self._h = h
        if st != 0:
            msg = self._lib.ctd_last_error(h).decode() if h else "ctd_create failed"
            raise EngineError("ctd_create: status %d (%s)" % (st, msg))
        self.capacity = int(capacity)
        self.device = int(device)
        self._model_arrays = {}
        self._ds_cap = None   # (max_records, max_option_slots) of the dataset's reservation

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ctd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what, allow=()):
        if st != 0 and st not in allow:
            raise EngineError("%s: status %d (%s)" % (what, st, self._lib.ctd_last_error(self._h).decode()))
        return st

    # ---- state ----
    def reset(self, n, seed=DEFAULT_SEED, first_gid=0, ruleset=RULESET_PRESET):
        self._check(self._lib.ctd_reset(self._h, n, seed, first_gid, ruleset), "ctd_reset")

    def set_seed(self, seed):
        self._check(self._lib.ctd_set_seed(self._h, seed), "ctd_set_seed")

    def load_states(self, states, first_slot=0):
        a = np.ascontiguousarray(states, dtype=np.uint8).reshape(-1, STATE_BYTES)
        self._check(self._lib.ctd_load_states(self._h, first_slot, len(a), a.ctypes.data), "ctd_load_states")

    def store_states(self, n, first_slot=0, out=None):
        a = np.empty((n, STATE_BYTES), dtype=np.uint8) if out is None else out
        assert a.dtype == np.uint8 and a.shape == (n, STATE_BYTES) and a.flags.c_contiguous
        self._check(self._lib.ctd_store_states(self._h, first_slot, n, a.ctypes.data), "ctd_store_states")
        return a

    def states_dev_ptr(self):
        p = ctypes.c_void_p()
        self._check(self._lib.ctd_states_dev(self._h, ctypes.byref(p)), "ctd_states_dev")
        return p.value

    def set_tapes(self, tapes):
        """tapes: list of uint8 arrays (one per slot) or None to clear."""
        if not tapes:
            self._check(self._lib.ctd_set_tapes(self._h, 0, None, None), "ctd_set_tapes")
            return
        off = np.zeros(len(tapes) + 1, dtype=np.uint32)
        off[1:] = np.cumsum([len(t) for t in tapes])
        flat = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.uint8) for t in tapes]))
        if len(flat) == 0:
            flat = np.zeros(1, dtype=np.uint8)
        self._check(self._lib.ctd_set_tapes(self._h, len(tapes), flat.ctypes.data, off.ctypes.data), "ctd_set_tapes")

    # ---- hot path ----
    def enumerate(self, n, stride=128):
        """-> (opts[n, stride] uint64, counts[n] uint32); grows stride until every list fits."""
        while True:
            opts = np.zeros((n, stride), dtype=np.uint64)
            counts = np.zeros(n, dtype=np.uint32)
            st = self._check(self._lib.ctd_enumerate(self._h, n, opts.ctypes.data, counts.ctypes.data, stride),
                             "ctd_enumerate", allow=(3,))
            if st == 0:
                return opts, counts
            stride = int(max(counts.max(), stride * 2))

    def choose_check(self, n):
        """Test hook: cooperative count/select of the playout kernel vs the enumerated list, per slot."""
        mis = np.empty(n, dtype=np.uint32)
        self._check(self._lib.ctd_choose_check(self._h, n, mis.ctypes.data), "ctd_choose_check")
        return mis

    def step(self, chosen):
        c = np.ascontiguousarray(chosen, dtype=np.uint64)
        winner = np.empty(len(c), dtype=np.int8)
        self._check(self._lib.ctd_step(self._h, len(c), c.ctypes.data, winner.ctypes.data), "ctd_step")
        return winner

    def playout(self, n_games, seed=DEFAULT_SEED, first_gid=0, ruleset=RULESET_PRESET, max_steps=4096,
                outputs=True):
        """Fused random playouts of new games.  -> dict(winner, points, steps, stats)."""
        stats = _lib.PlayoutStats()
        if outputs:
            winner = np.empty(n_games, dtype=np.int8)
            points = np.empty((n_games, 6), dtype=np.int8)
            steps = np.empty(n_games, dtype=np.uint16)
            self._check(self._lib.ctd_playout(self._h, n_games, seed, first_gid, ruleset, max_steps, winner.ctypes.data,
                                              points.ctypes.data, steps.ctypes.data, ctypes.byref(stats)), "ctd_playout")
            return dict(winner=winner, points=points, steps=steps, stats=stats_dict(stats))
        ms = ctypes.c_float()
        self._check(self._lib.ctd_playout_dev(self._h, n_games, seed, first_gid, ruleset, max_steps, ctypes.byref(stats),
                                              ctypes.byref(ms)), "ctd_playout_dev")
        d = stats_dict(stats)
        d["kernel_ms"] = ms.value
        return dict(stats=d)

    def arena(self, n_games, seats, seed=DEFAULT_SEED, first_gid=0, ruleset=RULESET_PRESET, max_steps=4096, record=None):
        """Games (seed, first_gid + i) played to the end on the device, one player per seat (ctd_arena).
        seats: six (kind, iterations, max_depth, reward_weight) tuples, kind in layout.SEAT_RANDOM / SEAT_PURE / SEAT_DEEP, a deep
        seat's value-model slot in bits 8..15 of kind (arena.deep(model=)).
        record: None, or (seats, mode, threshold) to append the targets of those seats' searches to the engine's dataset
        (ctd_arena_record; dataset_reserve first): mode layout.RECORD_TREE (CFRNode.get_all_targets(threshold) of every tree) or
        RECORD_ROOT (the position played, threshold not applied).  The games are the same either way.
        -> dict(winner[n] i8 (-1: error), points[n, 6] i8, steps[n] u16, searches[n] u32, stats, phase_ms (with record: + "record"))."""
        if len(seats) != 6:
            raise ValueError("ctd_arena takes one player per seat (6), got %d" % len(seats))
        arr = (_lib.ArenaSeat * 6)(*[_lib.ArenaSeat(int(k), int(it), int(d), float(wt)) for k, it, d, wt in seats])
        winner = np.empty(n_games, dtype=np.int8)
        points = np.empty((n_games, 6), dtype=np.int8)
        steps = np.empty(n_games, dtype=np.uint16)
        searches = np.empty(n_games, dtype=np.uint32)
        stats = _lib.PlayoutStats()
        ms = (ctypes.c_float * 4)()
        args = (self._h, n_games, seed, first_gid, ruleset, arr, max_steps, winner.ctypes.data, points.ctypes.data, steps.ctypes.data,
                searches.ctypes.data, ctypes.byref(stats))
        if record is None:
            self._check(self._lib.ctd_arena(*args, ms), "ctd_arena")
        else:
            rec_seats, mode, threshold = record
            mask = 0
            for s in rec_seats:
                mask |= 1 << int(s)
            opts = _lib.RecordOpts(mask, int(mode), float(threshold))
            self._check(self._lib.ctd_arena_record(*args, ctypes.byref(opts), ms), "ctd_arena_record")
        phase_ms = dict(advance=ms[0], search=ms[1], apply=ms[2])
        if record is not None:
            phase_ms["record"] = ms[3]
        return dict(winner=winner, points=points, steps=steps, searches=searches, stats=stats_dict(stats), phase_ms=phase_ms)

    # ---- self-play dataset (filled by arena(record=...)) ----
    def dataset_reserve(self, max_records, max_option_slots):
        """Allocate the engine's dataset in HBM (max_records rows of 448 floats; max_option_slots options / regrets) and clear it."""
        self._ds_cap = None
        self._check(self._lib.ctd_dataset_reserve(self._h, int(max_records), int(max_option_slots)), "ctd_dataset_reserve")
        self._ds_cap = (int(max_records), int(max_option_slots))

    def dataset_clear(self):
        self._check(self._lib.ctd_dataset_clear(self._h), "ctd_dataset_clear")

    def dataset_info(self):
        """-> dict(records, option_slots, dropped_trees, dropped_records, max_records, max_option_slots): trees that did not fit are
        dropped whole; the last two are the reservation's."""
        nr, ns, dt, dr = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self._lib.ctd_dataset_info(self._h, ctypes.byref(nr), ctypes.byref(ns), ctypes.byref(dt), ctypes.byref(dr)),
                    "ctd_dataset_info")
        return dict(records=nr.value, option_slots=ns.value, dropped_trees=dt.value, dropped_records=dr.value,
                    max_records=self._ds_cap[0], max_option_slots=self._ds_cap[1])

    def _dataset_fill(self, n, ns, feats, meta, origin, opts, regs):
        self._check(self._lib.ctd_dataset_read(self._h, 0, n, feats, meta, origin), "ctd_dataset_read")
        self._check(self._lib.ctd_dataset_read_options(self._h, 0, ns, opts, regs), "ctd_dataset_read_options")

    def dataset_arrays(self):
        """The whole dataset in physical order, as dataset_append takes it: features[R, 448] f32, meta[R] (layout.TARGET_META_DTYPE),
        origin[R] (layout.ORIGIN_DTYPE), options[S] u64, regrets[S] f64."""
        info = self.dataset_info()
        n, ns = info["records"], info["option_slots"]
        a = dict(features=np.zeros((n, 448), dtype=np.float32), meta=np.zeros(n, dtype=TARGET_META_DTYPE),
                 origin=np.zeros(n, dtype=ORIGIN_DTYPE), options=np.zeros(ns, dtype=np.uint64), regrets=np.zeros(ns, dtype=np.float64))
        self._dataset_fill(n, ns, *(a[k].ctypes.data for k in DATASET_KEYS))
        return a

    def dataset_tensors(self, device):
        """dataset_arrays as torch tensors on CUDA device `device`, copied device to device: features[R, 448] f32, meta[R, 72] and
        origin[R, 24] u8 (the bytes of the two records), options[S] u64, regrets[S] f64."""
        import torch
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError("dataset_tensors fills CUDA tensors, got device %r" % (device,))
        info = self.dataset_info()
        n, ns = info["records"], info["option_slots"]
        t = dict(features=torch.empty((n, 448), dtype=torch.float32, device=dev),
                 meta=torch.empty((n, TARGET_META_DTYPE.itemsize), dtype=torch.uint8, device=dev),
                 origin=torch.empty((n, ORIGIN_DTYPE.itemsize), dtype=torch.uint8, device=dev),
                 options=torch.empty(ns, dtype=torch.uint64, device=dev), regrets=torch.empty(ns, dtype=torch.float64, device=dev))
        torch.cuda.current_stream(dev).synchronize()   # the engine writes on its own stream: nothing of torch's may still use the memory
        self._dataset_fill(n, ns, *(t[k].data_ptr() for k in DATASET_KEYS))
        return t

    def dataset_append(self, features, meta, origin, options, regrets):
        """Append records after the dataset's own (ctd_dataset_append), from numpy arrays or torch CUDA tensors on any device, laid
        out as dataset_arrays / dataset_tensors return them (features with 418 columns are zero-padded to 448; meta and origin may
        also be their raw bytes).  option_offset indexes `options` and is rebased; tree and origin are kept.  All or nothing:
        EngineError with status 3 when the reservation is too small, 1 for a malformed record, and the dataset is unchanged."""
        arrs = [_append_input(x, k) for x, k in zip((features, meta, origin, options, regrets), DATASET_KEYS)]
        (f, nf), (m, n), (o, no), (x, ns), (r, nr) = arrs
        if nf != n or no != n or nr != ns:
            raise ValueError("dataset_append: %d feature rows, %d metas, %d origins, %d options, %d regrets" % (nf, n, no, ns, nr))
        tensors = [a for a, _ in arrs if not isinstance(a, np.ndarray)]
        for d in {t.device for t in tensors}:
            import torch
            torch.cuda.current_stream(d).synchronize()   # the producing work must be complete: the engine copies on its own stream
        ptr = [a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr() for a in (f, m, o, x, r)]
        self._check(self._lib.ctd_dataset_append(self._h, n, ns, *ptr), "ctd_dataset_append")

    def dataset_read(self):
        """Every record of the dataset in canonical order (origin gid, search, then pre-order within the tree): features[R, 418] f32,
        meta[R] (tree: the game's index in its arena call; option_offset into options / regrets), origin[R] (layout.ORIGIN_DTYPE),
        row[R] (the record's physical row, what train_on_dataset's indices name), and every option slot: options[S] u64, regrets[S]
        f64.  Engine.targets_as_tuples accepts the result as it is."""
        a = self.dataset_arrays()
        origin = a["origin"]
        # a tree's records are consecutive in pre-order, so the physical row orders them within (gid, search)
        row = np.lexsort((np.arange(len(origin)), origin["search"], origin["gid"])).astype(np.int64)
        return dict(features=a["features"][row, :418], meta=a["meta"][row], origin=origin[row], row=row, options=a["options"],
                    regrets=a["regrets"])

    def playout_slots(self, n, max_steps=4096):
        winner = np.empty(n, dtype=np.int8)
        steps = np.empty(n, dtype=np.uint16)
        self._check(self._lib.ctd_playout_slots(self._h, n, max_steps, winner.ctypes.data, steps.ctypes.data),
                    "ctd_playout_slots")
        return winner, steps

    # ---- MCCFR ----
    def make_roots(self, n, seed=DEFAULT_SEED, first_gid=0, ruleset=RULESET_PRESET, back_lo=0, back_hi=20,
                   flavour=ROOTS_CLOSE_TO_FINISHED):
        """CFR roots on the device: run_utils.create_a_close_to_finished_game (default flavour) or
        run_utils.create_a_random_game (ROOTS_RANDOM_GAME: games[-m], m in [back_lo, back_hi], the searching player fixed
        before the forced moves are skipped).  -> root_step[n]"""
        steps = np.empty(n, dtype=np.uint32)
        self._check(self._lib.ctd_make_roots(self._h, n, seed, first_gid, ruleset, back_lo, back_hi, flavour,
                                             steps.ctypes.data), "ctd_make_roots")
        return steps

    def load_roots(self, roots, knows, used_cards, gids):
        r = np.ascontiguousarray(roots, dtype=np.uint8).reshape(-1, STATE_BYTES)
        k = np.ascontiguousarray(knows, dtype=np.uint8).reshape(-1, KNOW_BYTES)
        u = np.ascontiguousarray(used_cards, dtype=np.uint8).reshape(-1, 76)
        g = np.ascontiguousarray(gids, dtype=np.uint64)
        assert len(r) == len(k) == len(u) == len(g)
        self._check(self._lib.ctd_load_roots(self._h, len(r), r.ctypes.data, k.ctypes.data, u.ctypes.data, g.ctypes.data),
                    "ctd_load_roots")

    def store_roots(self, n):
        r = np.empty((n, STATE_BYTES), dtype=np.uint8)
        k = np.empty((n, KNOW_BYTES), dtype=np.uint8)
        u = np.empty((n, 76), dtype=np.uint8)
        g = np.empty(n, dtype=np.uint64)
        self._check(self._lib.ctd_store_roots(self._h, n, r.ctypes.data, k.ctypes.data, u.ctypes.data, g.ctypes.data),
                    "ctd_store_roots")
        return r, k, u, g

    def tree_shape(self, iterations, ruleset=RULESET_PRESET, n_roots=1):
        """-> (nodes in a tree's first chunk, bytes per node, bytes of the arena a search of n_roots trees starts with)."""
        n0, nb, ab = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_uint64()
        self._lib.ctd_mccfr_tree_shape(iterations, ruleset, n_roots, ctypes.byref(n0), ctypes.byref(nb), ctypes.byref(ab))
        return n0.value, nb.value, ab.value

    def export_trees(self, n, first=0):
        """The trees of the last mccfr()/mccfr_pred() call, roots [first, first+n) -> [TreeView]."""
        sizes = np.zeros(n, dtype=np.uint64)
        self._check(self._lib.ctd_mccfr_export(self._h, first, n, sizes.ctypes.data, None, 0), "ctd_mccfr_export")
        total = int(sizes.sum())
        buf = np.zeros(max(total, 1), dtype=np.uint8)
        self._check(self._lib.ctd_mccfr_export(self._h, first, n, sizes.ctypes.data, buf.ctypes.data, total), "ctd_mccfr_export")
        off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        return [TreeView(buf[int(off[i]):int(off[i + 1])]) for i in range(n)]

    def root_children(self, tree, first, count):
        """Children [first, first+count) of the root of tree `tree` -> (options u64, R, s, C float64)."""
        o = np.zeros(count, dtype=np.uint64)
        r, s_, c = (np.zeros(count, dtype=np.float64) for _ in range(3))
        self._check(self._lib.ctd_mccfr_root_children(self._h, tree, first, count, o.ctypes.data, r.ctypes.data, s_.ctypes.data,
                                                      c.ctypes.data), "ctd_mccfr_root_children")
        return o, r, s_, c

    def mccfr(self, n_roots, iterations=200, seed=DEFAULT_SEED, ruleset=RULESET_PRESET, trees=False):
        """CFRNode(...).cfr_train(iterations) on the loaded/made roots.  -> dict(results, trees, kernel_ms)"""
        res = np.zeros(n_roots, dtype=MCCFR_RESULT_DTYPE)
        ms = ctypes.c_float()
        self._check(self._lib.ctd_mccfr(self._h, n_roots, seed, iterations, ruleset, res.ctypes.data, ctypes.byref(ms)),
                    "ctd_mccfr")
        return dict(results=res, trees=self.export_trees(n_roots) if trees else None, kernel_ms=ms.value)

    def mccfr_continue(self, n_roots, more_iterations, seed=DEFAULT_SEED, ruleset=RULESET_PRESET):
        """Root-parallel mode only: `more_iterations` further iterations on the trees of the last mccfr() call."""
        res = np.zeros(n_roots, dtype=MCCFR_RESULT_DTYPE)
        ms = ctypes.c_float()
        self._check(self._lib.ctd_mccfr_continue(self._h, n_roots, seed, more_iterations, ruleset, res.ctypes.data, ctypes.byref(ms)),
                    "ctd_mccfr_continue")
        return dict(results=res, kernel_ms=ms.value)

    def root_set(self, regrets, strategy, values):
        """Root-parallel mode only: overwrite the roots' cumulative_regrets / cumulative_strategy [n, stride] and node_value [n, 6]."""
        r = np.ascontiguousarray(regrets, dtype=np.float64)
        c = np.ascontiguousarray(strategy, dtype=np.float64)
        v = np.ascontiguousarray(values, dtype=np.float64)
        assert r.shape == c.shape and v.shape == (len(r), 6)
        self._check(self._lib.ctd_mccfr_root_set(self._h, len(r), r.shape[1], r.ctypes.data, c.ctypes.data, v.ctypes.data),
                    "ctd_mccfr_root_set")

    def set_value_model(self, model, slot=0):
        """model: a ValueOnlyNN(418, 512) in eval mode (reference state_dict layout), loaded into value-model slot `slot` (0 ..
        layout.MAX_VALUE_MODELS - 1).  mccfr_pred and value_eval use slot 0; an arena's deep seat uses the slot of arena.deep(model=)."""
        from .value_model import fold
        arrs = fold(model)
        self._check(self._lib.ctd_set_value_model_slot(self._h, int(slot), *[a.ctypes.data for a in arrs]), "ctd_set_value_model_slot")
        self._model_arrays[int(slot)] = arrs   # the folded weights of every loaded slot

    def set_value_backend(self, backend):
        """'fp32' (CUDA cores, leaves batched in waves), 'tcgen05' (tensor cores, 3xTF32 split precision, waves) or 'fused' (the
        default: deep MCCFR in one launch, every warp evaluates its own leaves in fp32; value_eval stays on the tensor cores)."""
        b = {"fp32": 0, "tcgen05": 1, "fused": 2}[backend]
        self._check(self._lib.ctd_set_value_backend(self._h, b), "ctd_set_value_backend")

    def value_eval(self, features, weight=5.0):
        f = np.zeros((len(features), 448), dtype=np.float32)
        f[:, :np.shape(features)[1]] = features
        out = np.empty((len(f), 6), dtype=np.float32)
        self._check(self._lib.ctd_value_eval(self._h, len(f), f.ctypes.data, weight, out.ctypes.data), "ctd_value_eval")
        return out

    def encode(self, n, cfr_role_pick=True):
        """Game.encode_game of roots [0,n); cfr_role_pick: role-pick states seen by "player 5" as inside CFRNode."""
        f = np.empty((n, 448), dtype=np.float32)
        self._check(self._lib.ctd_encode(self._h, n, 1 if cfr_role_pick else 0, f.ctypes.data), "ctd_encode")
        return f[:, :418]

    def mccfr_pred(self, n_roots, iterations=200, max_depth=10, seed=DEFAULT_SEED, ruleset=RULESET_PRESET, weight=5.0,
                   trees=False):
        """CFRNode(..., model).cfr_pred(iterations, max_depth) on the loaded/made roots."""
        res = np.zeros(n_roots, dtype=MCCFR_RESULT_DTYPE)
        ms, waves = ctypes.c_float(), ctypes.c_uint32()
        self._check(self._lib.ctd_mccfr_pred(self._h, n_roots, seed, iterations, max_depth, ruleset, weight, res.ctypes.data,
                                             ctypes.byref(ms), ctypes.byref(waves)), "ctd_mccfr_pred")
        return dict(results=res, trees=self.export_trees(n_roots) if trees else None, kernel_ms=ms.value, waves=waves.value)

    def mccfr_targets(self, n_roots, iterations=200, seed=DEFAULT_SEED, ruleset=RULESET_PRESET, threshold=15.0):
        """CFRNode.get_all_targets() for every tree of the last mccfr()/mccfr_pred() call with the same arguments.
        -> dict(features[R,418] f32, meta[R], options[S] u64, regrets[S] f64)."""
        nr, ns = ctypes.c_uint32(0), ctypes.c_uint32(0)
        self._check(self._lib.ctd_mccfr_targets(self._h, n_roots, seed, iterations, ruleset, threshold, ctypes.byref(nr),
                                                ctypes.byref(ns), None, None, None, None), "ctd_mccfr_targets")
        feats = np.zeros((nr.value, 448), dtype=np.float32)
        meta = np.zeros(nr.value, dtype=TARGET_META_DTYPE)
        opts = np.zeros(max(ns.value, 1), dtype=np.uint64)
        regs = np.zeros(max(ns.value, 1), dtype=np.float64)
        if nr.value:
            self._check(self._lib.ctd_mccfr_targets(self._h, n_roots, seed, iterations, ruleset, threshold, ctypes.byref(nr),
                                                    ctypes.byref(ns), feats.ctypes.data, meta.ctypes.data, opts.ctypes.data,
                                                    regs.ctypes.data), "ctd_mccfr_targets")
        return dict(features=feats[:, :418], meta=meta, options=opts[:ns.value], regrets=regs[:ns.value])

    @staticmethod
    def targets_as_tuples(t):
        """The reference's pickle format (generate_test_data.py:25, train_from_scratch.py): a list of
        (model_input float32[418], options_input float32[1,K,131], node_value float64[6], decision_dist float64[K])."""
        import torch
        out = []
        for i, m in enumerate(t["meta"]):
            o, k = int(m["option_offset"]), int(m["n_options"])
            out.append((torch.from_numpy(t["features"][i].copy()),
                        torch.from_numpy(encode_options(t["options"][o:o + k])).unsqueeze(0),
                        torch.from_numpy(np.array(m["node_value"])), torch.from_numpy(t["regrets"][o:o + k].copy())))
        return out

    def sync(self):
        self._check(self._lib.ctd_sync(self._h), "ctd_sync")

    @property
    def launches(self):
        return int(self._lib.ctd_launch_count(self._h))


DATASET_KEYS = ("features", "meta", "origin", "options", "regrets")
# per input of dataset_append: (numpy dtypes, torch dtype names, bytes per item)
_APPEND_TYPES = dict(features=((np.float32,), ("float32",), 4 * 448),
                     meta=((TARGET_META_DTYPE, np.uint8), ("uint8",), TARGET_META_DTYPE.itemsize),
                     origin=((ORIGIN_DTYPE, np.uint8), ("uint8",), ORIGIN_DTYPE.itemsize),
                     options=((np.uint64, np.int64), ("uint64", "int64"), 8),
                     regrets=((np.float64,), ("float64",), 8))


def _append_input(a, key):
    """One input of Engine.dataset_append -> (contiguous numpy array or CUDA tensor, item count); features of 418 columns padded."""
    np_types, t_types, item = _APPEND_TYPES[key]
    if isinstance(a, np.ndarray) or not hasattr(a, "data_ptr"):
        a = np.ascontiguousarray(a)
        if key == "features" and a.ndim == 2 and a.shape[1] == 418:
            a = np.pad(a, ((0, 0), (0, 448 - 418)))
        ok, nbytes = any(a.dtype == np.dtype(t) for t in np_types), a.nbytes
    else:
        if not a.is_cuda:
            raise ValueError("dataset_append takes numpy arrays or CUDA tensors, got a tensor on %s" % a.device)
        if key == "features" and a.dim() == 2 and a.shape[1] == 418:
            import torch
            a = torch.nn.functional.pad(a, (0, 448 - 418))
        a = a.contiguous()
        ok, nbytes = str(a.dtype).replace("torch.", "") in t_types, a.numel() * a.element_size()
    if key == "features" and (len(a.shape) != 2 or a.shape[1] != 448):
        ok = False
    if not ok or nbytes % item:
        raise ValueError("dataset_append: %s of dtype %s and shape %s is not what dataset_arrays returns"
                         % (key, a.dtype, tuple(a.shape)))
    return a, nbytes // item


def stats_dict(s):
    return dict(games=int(s.games), steps=int(s.steps), steps_sq=int(s.steps_sq), wins=[int(x) for x in s.wins],
                points_sum=[int(x) for x in s.points_sum], points_sq=[int(x) for x in s.points_sq],
                errors=int(s.errors), max_steps=int(s.max_steps))
