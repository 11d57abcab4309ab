"""Self-play training data from the device arena, and training on it where it lies.

    eng = Engine(capacity=4096)
    out = record_arena(1000, [arena.deep(200)] * 6, record_seats=range(6), models=[model], engine=eng, max_records=300_000)
    data = eng.dataset_read()
    train_idx, val_idx = split_by_game(data["origin"], 0.1, seed=1, rows=data["row"])
    best = train_on_dataset(eng, train_idx, val_idx, "winner", epochs=20, lr=1e-3, model=model)

The arena records the targets of its searches into a dataset the engine keeps in HBM (ctd_arena_record): after each search its
trees are counted, given rows on the device and written out, and each record's game outcome is filled in when the call ends.
Training gathers its rows from that dataset on the device (ctd_train_begin_dataset); only the index lists cross to the device.

On several GPUs (torchrun, one rank per GPU) every rank records its own block of games into its own engine, gather_dataset
appends all of them to one rank's dataset (NCCL: device to device, the records never touch the host) and that rank trains as
above.  The training step is bound by launch latency, so one GPU training on everything is as fast as several sharing the work,
and the semantics stay those of one engine.  save_dataset / load_dataset keep a dataset in an .npz beyond its engine, so a round
can be trained again or appended to a later round's records.

Which records, which labels.  The reference trains on CFRNode.get_all_targets(15) of pure-MCCFR trees, labelled with node_value.
A deep seat's tree is different: in eval mode a node's node_value is written only on its first backprop, so it sums to the reward
weight (5) or to 1 at a terminal and never reaches 15 -- tree mode at the reference's threshold records nothing from it -- and what
it holds is the value model's own prediction, so training on it would distil the model into itself.  Deep seats are therefore
recorded in root mode (the position each search played) and labelled with the game's winner, a single sample of what a pure tree's
node_value estimates.  Those are the defaults here.  Pure seats can use either mode with node_value labels, which gives the
reference's targets on self-play positions instead of random ones.
"""
import math

import numpy as np

from .engine import Engine, DEFAULT_SEED, RULESET_PRESET, DATASET_KEYS
from .layout import RECORD_TREE, RECORD_ROOT, LABEL_NODE_VALUE, LABEL_WINNER, TARGET_META_DTYPE, ORIGIN_DTYPE

MODES = {"tree": RECORD_TREE, "root": RECORD_ROOT}
LABELS = {"node_value": LABEL_NODE_VALUE, "winner": LABEL_WINNER}
DATASET_FORMAT = 1   # save_dataset's .npz layout
COUNT_KEYS = ("records", "option_slots", "dropped_trees", "dropped_records")


def _code(value, names, what):
    if value in names:
        return names[value]
    if value in names.values() and not isinstance(value, bool):
        return int(value)
    raise ValueError("%s must be one of %s, got %r" % (what, sorted(names), value))


def record_arena(n_games, seats, record_seats, models=None, mode="root", threshold=15.0, engine=None, seed=DEFAULT_SEED, first_gid=0,
                 ruleset=RULESET_PRESET, max_steps=4096, max_records=None, max_option_slots=None):
    """arena.play_arena(n_games, seats, models=models) that also records the searches of the seats in `record_seats` (seat indices)
    into the engine's dataset: mode "root" (default: the position each search played) or "tree" (CFRNode.get_all_targets(threshold)
    of each tree).  The games are exactly those play_arena plays.
    Without `engine` a new one is made, its dataset reserved, and the records are read back (out["dataset"], Engine.dataset_read)
    before it closes.  With `engine` the records are appended to its dataset, which stays there for train_on_dataset; max_records
    (and max_option_slots, default 16 per record) given: the dataset is reserved (and cleared) first.  Without a reservation the
    default room is 256 records per game in root mode and 2048 in tree mode.  Trees that do not fit are dropped whole and counted.
    -> play_arena's result plus info (Engine.dataset_info after the call) and dataset (without `engine`)."""
    from . import arena
    code = _code(mode, MODES, "mode")
    rec_seats = [int(s) for s in record_seats]
    if any(s < 0 or s > 5 for s in rec_seats):
        raise ValueError("record_seats are seat indices 0..5, got %r" % (rec_seats,))
    if not (isinstance(threshold, (int, float)) and math.isfinite(threshold) and threshold >= 0):
        raise ValueError("threshold must be a finite number >= 0, got %r" % (threshold,))
    seats = list(seats)
    if len(seats) != 6:
        raise ValueError("one player per seat (6), got %d" % len(seats))
    models = arena.arena_models(seats, None, models, engine)
    if max_records is not None and int(max_records) < 1:
        raise ValueError("max_records must be >= 1")
    own = engine is None
    if own or max_records is not None:
        max_records = int(max_records or max(1, n_games) * (256 if code == RECORD_ROOT else 2048))
        max_option_slots = int(max_option_slots or 16 * max_records)
    eng = engine
    if own:
        import torch
        eng = Engine(capacity=max(1, min(int(n_games), 8192)), device=torch.cuda.current_device() if torch.cuda.is_available() else 0)
    try:
        if max_records is not None:
            eng.dataset_reserve(max_records, max_option_slots)
        out = arena.play_arena(n_games, seats, engine=eng, models=models, seed=seed, first_gid=first_gid, ruleset=ruleset,
                               max_steps=max_steps, record=(rec_seats, code, float(threshold)))
        out["info"] = eng.dataset_info()
        out["dataset"] = eng.dataset_read() if own else None
    finally:
        if own:
            eng.close()
    return out


def _item_bytes(key, n_records, n_slots):
    return {"features": 448 * 4 * n_records, "meta": TARGET_META_DTYPE.itemsize * n_records,
            "origin": ORIGIN_DTYPE.itemsize * n_records, "options": 8 * n_slots, "regrets": 8 * n_slots}[key]


def _from_bytes(key, b, n_records):
    """A received byte buffer (torch CUDA tensor or numpy array) -> the layout dataset_append takes."""
    if isinstance(b, np.ndarray):
        dt = {"features": np.float32, "meta": TARGET_META_DTYPE, "origin": ORIGIN_DTYPE, "options": np.uint64, "regrets": np.float64}
        a = b.view(dt[key])
        return a.reshape(n_records, 448) if key == "features" else a
    import torch
    if key == "features":
        return b.view(torch.float32).view(n_records, 448)
    if key in ("meta", "origin"):
        return b.view(n_records, -1)
    return b.view(torch.int64 if key == "options" else torch.float64)


def gather_dataset(engine, dst=0, group=None):
    """Collective over `group` (default: the default process group): every rank calls it with its own engine.  The datasets of all
    ranks but `dst` are appended to `dst`'s (Engine.dataset_append), in rank order, so that dst holds its own records followed by
    those of the other ranks; their datasets are left as they are.  The ranks' counts and dst's reservation are all_gathered first,
    so every rank reaches the same verdict: when the records or option slots do not fit dst's reservation, every rank raises the
    same ValueError and nothing is appended.  Then one rank at a time sends its physical-order dataset to dst (point to point,
    which bounds dst's staging memory to one rank's records): with NCCL as CUDA tensors (Engine.dataset_tensors), so the records
    never touch the host; with gloo as host arrays (Engine.dataset_arrays).  Game ids of different ranks are disjoint (play_arena's
    rank blocks), so dataset_read's canonical order and split_by_game work on the merged dataset as they are.  A single process:
    nothing to do.  -> dict(records, option_slots, dropped_trees, dropped_records): one entry per rank, as the datasets stood
    before the gather."""
    import torch
    import torch.distributed as dist
    info = engine.dataset_info()
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return {k: [info[k]] for k in COUNT_KEYS}
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if not 0 <= int(dst) < world:
        raise ValueError("dst must be a rank of the group (0 .. %d), got %r" % (world - 1, dst))
    dst = int(dst)
    nccl = dist.get_backend(group) == "nccl"
    dev = torch.device("cuda", engine.device) if nccl else torch.device("cpu")
    mine = torch.tensor([info[k] for k in COUNT_KEYS + ("max_records", "max_option_slots")], dtype=torch.int64, device=dev)
    every = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(every, mine, group=group)
    every = [[int(x) for x in t.tolist()] for t in every]
    counts = {k: [c[i] for c in every] for i, k in enumerate(COUNT_KEYS)}
    recs, slots = counts["records"], counts["option_slots"]
    cap_r, cap_s = every[dst][4], every[dst][5]
    if sum(recs) > cap_r or sum(slots) > cap_s:
        raise ValueError("gather_dataset: %d records and %d option slots over %d ranks do not fit rank %d's reservation of %d and %d"
                         % (sum(recs), sum(slots), world, dst, cap_r, cap_s))
    for src in range(world):
        if src == dst or (recs[src] == 0 and slots[src] == 0) or rank not in (src, dst):
            continue
        sizes = {k: _item_bytes(k, recs[src], slots[src]) for k in DATASET_KEYS}
        if rank == src:
            parts = engine.dataset_tensors(dev) if nccl else engine.dataset_arrays()
            for k in DATASET_KEYS:
                if sizes[k]:
                    p = parts[k]
                    b = p.view(torch.uint8).reshape(-1) if nccl else torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).reshape(-1))
                    dist.send(b, group=group, group_dst=dst)
            if nccl:
                torch.cuda.current_stream(dev).synchronize()   # the sends have read the tensors before they are freed
        else:
            got = {}
            for k in DATASET_KEYS:
                b = torch.empty(sizes[k], dtype=torch.uint8, device=dev)
                if sizes[k]:
                    dist.recv(b, group=group, group_src=src)
                got[k] = _from_bytes(k, b if nccl else b.numpy(), recs[src])
            engine.dataset_append(*(got[k] for k in DATASET_KEYS))
    return counts


def save_dataset(engine, path):
    """The engine's dataset, in physical order, to an .npz (np.savez: `path` gains .npz unless it has it) with its format version:
    features [R, 448] f32, meta [R, 72] and origin [R, 24] as bytes, options [S] u64, regrets [S] f64.  -> dict(records, option_slots)"""
    a = engine.dataset_arrays()
    n = len(a["meta"])
    np.savez(path, format_version=np.int64(DATASET_FORMAT), features=a["features"], meta=a["meta"].view(np.uint8).reshape(n, -1),
             origin=a["origin"].view(np.uint8).reshape(n, -1), options=a["options"], regrets=a["regrets"])
    return dict(records=n, option_slots=len(a["options"]))


def load_dataset(engine, path):
    """Append the records of a save_dataset file to the engine's reserved dataset (Engine.dataset_append: their option offsets are
    rebased, trees and origins kept).  ValueError when the file is not of this format or does not fit the reservation (nothing is
    appended); EngineError when no dataset is reserved.  -> dict(records, option_slots) appended."""
    with np.load(path, allow_pickle=False) as z:
        if "format_version" not in z.files or int(z["format_version"]) != DATASET_FORMAT:
            raise ValueError("%s is not a dataset of format %d (save_dataset)" % (path, DATASET_FORMAT))
        a = {k: z[k] for k in DATASET_KEYS}
    meta, origin = a["meta"].reshape(-1).view(TARGET_META_DTYPE), a["origin"].reshape(-1).view(ORIGIN_DTYPE)
    n, ns = len(meta), len(a["options"])
    info = engine.dataset_info()
    if info["records"] + n > info["max_records"] or info["option_slots"] + ns > info["max_option_slots"]:
        raise ValueError("%s: %d records and %d option slots do not fit the dataset (%d + %d of %d, %d + %d of %d)"
                         % (path, n, ns, info["records"], n, info["max_records"], info["option_slots"], ns, info["max_option_slots"]))
    engine.dataset_append(a["features"], meta, origin, a["options"], a["regrets"])
    return dict(records=n, option_slots=ns)


def split_by_game(origin, val_fraction, seed, rows=None):
    """Training and validation rows of a dataset, split by game so that sibling positions of one game never sit on both sides.
    origin: the records' ctd_record_origin (layout.ORIGIN_DTYPE) in any order; rows: their physical rows (default: origin is in
    physical order, as ctd_dataset_read returns it).  round(val_fraction * games) games, drawn with numpy's default_rng(seed), go
    to validation; at least one game stays for training.  Deterministic.
    -> (train_rows, val_rows) uint32, physical rows in canonical order (gid, search, row)."""
    o = np.asarray(origin)
    if not 0.0 <= float(val_fraction) < 1.0:
        raise ValueError("val_fraction must be in [0, 1), got %r" % (val_fraction,))
    rows = np.arange(len(o), dtype=np.int64) if rows is None else np.asarray(rows, dtype=np.int64)
    if rows.shape != (len(o),):
        raise ValueError("rows must give one physical row per record")
    order = np.lexsort((rows, o["search"], o["gid"]))
    games = np.unique(o["gid"])
    n_val = min(int(round(float(val_fraction) * len(games))), max(0, len(games) - 1))
    val_games = np.random.default_rng(seed).permutation(games)[:n_val]
    is_val = np.isin(o["gid"][order], val_games)
    sorted_rows = rows[order]
    return sorted_rows[~is_val].astype(np.uint32), sorted_rows[is_val].astype(np.uint32)


def train_on_dataset(engine, train_idx, val_idx, label="winner", epochs=10, lr=1e-3, gamma=1.0, batch_size=64, model=None,
                     seed=DEFAULT_SEED, parent_folder="selfplay", history=None, verbose=False):
    """train_node_value_only's epoch loop (StepLR(300, gamma), <parent_folder>/best_model.pt at the best evaluation loss) on rows
    train_idx / val_idx of `engine`'s dataset, gathered on the device.  label: "winner" (default: one-hot of the game's winner; an
    errored game's record is refused) or "node_value" (the tree's node_value, the reference's target -- for pure-seat records; see
    the module notes).  model: the ValueOnlyNN(418, 512) to start from (default: a freshly initialised one).  With the same rows,
    labels, model and seed the result is bit for bit that of train_node_value_only.  -> best evaluation loss."""
    import os
    from .train import Trainer, _epochs
    from .value_model import ValueOnlyNN
    code = _code(label, LABELS, "label")
    train_idx = np.asarray(train_idx).reshape(-1)
    val_idx = np.asarray(val_idx).reshape(-1)
    if len(train_idx) == 0:
        raise ValueError("no training rows")
    if not 1 <= int(batch_size) <= 65536:
        raise ValueError("batch_size must be in [1, 65536], got %r" % (batch_size,))
    if int(epochs) < 0:
        raise ValueError("epochs must be >= 0")
    if engine is None:
        raise ValueError("the dataset lives in an engine: pass the engine that recorded it")
    os.makedirs(parent_folder, exist_ok=True)
    model = model or ValueOnlyNN(418, 512)
    tr = Trainer.from_dataset(engine, train_idx, val_idx, code, batch_size)
    try:
        return _epochs(tr, model, int(epochs), lr, gamma, int(batch_size), seed, parent_folder, verbose, history)
    finally:
        tr.close()
