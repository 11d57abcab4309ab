"""Self-play training data from the device arena, and training on it where it lies.

    eng = Engine(capacity=4096)
    out = record_arena(1000, [arena.deep(200)] * 6, record_seats=range(6), models=[model], engine=eng, max_records=300_000)
    data = eng.dataset_read()
    train_idx, val_idx = split_by_game(data["origin"], 0.1, seed=1, rows=data["row"])
    best = train_on_dataset(eng, train_idx, val_idx, "winner", epochs=20, lr=1e-3, model=model)

The arena records the targets of its searches into a dataset the engine keeps in HBM (ctd_arena_record): after each search its
trees are counted, given rows on the device and written out, and each record's game outcome is filled in when the call ends.
Training gathers its rows from that dataset on the device (ctd_train_begin_dataset); only the index lists cross to the device.

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

from .engine import Engine, DEFAULT_SEED, RULESET_PRESET
from .layout import RECORD_TREE, RECORD_ROOT, LABEL_NODE_VALUE, LABEL_WINNER

MODES = {"tree": RECORD_TREE, "root": RECORD_ROOT}
LABELS = {"node_value": LABEL_NODE_VALUE, "winner": LABEL_WINNER}


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
