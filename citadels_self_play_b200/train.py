"""Value-network training on the device: the reference's `train_node_value_only` (algorithms/train.py:13-86).

    best_eval_loss = train_node_value_only(train_data, val_data, epochs, lr, hidden_size, gamma, batch_size=64,
                                           parent_folder="pretrain")

Same arguments, same side effect (`<parent_folder>/best_model.pt`: the state_dict of the epoch with the lowest evaluation
loss, loadable by run_utils.setup_model_for_eval) and same return value.  `train_data` / `val_data` are lists of the reference's
target tuples (model_input float32[418], options_input, node_value float64[6], decision_dist) -- what
datagen.get_mccfr_targets returns.  The model is ValueOnlyNN(418, 512); forward, loss, backward and Adam run in the engine's
kernels (csrc/ctd_train.cuh, dense products on the tcgen05 GEMM); this module is the epoch loop: batch order, StepLR(300, gamma),
best-eval checkpointing.

Chance: initial weights come from torch's default initialisation of the mirror class (pass `model=` or seed torch yourself, as
with the reference); batch order and dropout masks are Philox4x32-10 streams of `seed` (functions below), so a run is a pure
function of its inputs.  tests/golden/gen_train_fixture.py replays the unmodified reference with its DataLoader order and its
dropout routed through the same functions; tests/test_gpu_train.py compares loss curves and weights.
"""
import ctypes
import os
import numpy as np

from .engine import Engine, EngineError, DEFAULT_SEED

KEEP_U32 = 3435973836        # floor(0.8 * 2^32): Dropout(0.2)
STATE_KEYS = ["fc1.weight", "fc1.bias", "bn1.weight", "bn1.bias", "bn1.running_mean", "bn1.running_var", "fc2.weight", "fc2.bias",
              "bn2.weight", "bn2.bias", "bn2.running_mean", "bn2.running_var", "fc3.weight", "fc3.bias", "fc4.weight", "fc4.bias"]


def philox_words(seed, step, layer, e):
    """Word e & 3 of Philox4x32-10(key = seed, counter = (e >> 2, layer | step << 8, 0xD0, 0)) for an array of element indices e
    (uint32) -- the generator of csrc/ctd_train.cuh (ctd_tr_philox_word)."""
    e = np.asarray(e, dtype=np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1 = e >> np.uint64(2), np.full(e.shape, (layer | (step << 8)) & 0xFFFFFFFF, dtype=np.uint64)
    c2, c3 = np.full(e.shape, 0xD0, dtype=np.uint64), np.zeros(e.shape, dtype=np.uint64)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        n0, n2 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m32
        c1, c3, c0, c2 = p1 & m32, p0 & m32, n0, n2
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
    w = e & np.uint64(3)
    return np.where(w == 0, c0, np.where(w == 1, c1, np.where(w == 2, c2, c3))).astype(np.uint64)


def dropout_mask(seed, step, layer, rows, width):
    """keep-mask [rows, width] of dropout layer `layer` (1 or 2) at optimiser step `step` (0-based): element r * width + c."""
    e = np.arange(rows * width, dtype=np.uint64)
    return (philox_words(seed, step, layer, e) < KEEP_U32).reshape(rows, width)


def epoch_permutation(seed, epoch, n):
    """Batch order of epoch `epoch`: Fisher-Yates from the top over arange(n) with draws philox_words(seed, epoch, 14, k)."""
    perm = np.arange(n, dtype=np.uint32)
    if n > 1:
        d = philox_words(seed, epoch, 14, np.arange(n - 1, dtype=np.uint64))
        for k, i in enumerate(range(n - 1, 0, -1)):
            j = int((int(d[k]) * (i + 1)) >> 32)
            perm[i], perm[j] = perm[j], perm[i]
    return perm


class Trainer:
    """Thin wrapper over ctd_train_* (include/citadels_b200.h)."""

    def __init__(self, engine, feats, vals, val_feats, val_vals, batch_size):
        self.e = engine
        self.lib, self.h = engine._lib, engine._h
        f = np.ascontiguousarray(feats, dtype=np.float32).reshape(-1, 418)
        v = np.ascontiguousarray(vals, dtype=np.float64).reshape(-1, 6)
        vf = np.ascontiguousarray(val_feats, dtype=np.float32).reshape(-1, 418)
        vv = np.ascontiguousarray(val_vals, dtype=np.float64).reshape(-1, 6)
        assert len(f) == len(v) and len(vf) == len(vv)
        self.n_train, self.n_val = len(f), len(vf)
        engine._check(self.lib.ctd_train_begin(self.h, len(f), f.ctypes.data, v.ctypes.data, len(vf), vf.ctypes.data if len(vf) else None,
                                               vv.ctypes.data if len(vf) else None, int(batch_size)), "ctd_train_begin")

    @classmethod
    def from_dataset(cls, engine, train_idx, val_idx, label, batch_size):
        """ctd_train_begin_dataset: the rows are records train_idx / val_idx (physical rows) of the engine's dataset, gathered on the
        device; label layout.LABEL_NODE_VALUE or LABEL_WINNER."""
        self = cls.__new__(cls)
        self.e = engine
        self.lib, self.h = engine._lib, engine._h
        ti = np.ascontiguousarray(train_idx, dtype=np.uint32).reshape(-1)
        vi = np.ascontiguousarray(val_idx, dtype=np.uint32).reshape(-1)
        self.n_train, self.n_val = len(ti), len(vi)
        engine._check(self.lib.ctd_train_begin_dataset(self.h, len(ti), ti.ctypes.data, len(vi), vi.ctypes.data if len(vi) else None,
                                                       int(label), int(batch_size)), "ctd_train_begin_dataset")
        return self

    def _ptrs(self, arrs):
        return (ctypes.c_void_p * 16)(*[a.ctypes.data for a in arrs])

    def set_state(self, state_dict):
        arrs = [np.ascontiguousarray(np.asarray(state_dict[k].detach().cpu().numpy() if hasattr(state_dict[k], "detach") else state_dict[k]),
                                     dtype=np.float32) for k in STATE_KEYS]
        if arrs[0].shape != (512, 418):
            raise ValueError("the training kernels are built for ValueOnlyNN(418, 512)")
        self.e._check(self.lib.ctd_train_set_state(self.h, self._ptrs(arrs)), "ctd_train_set_state")

    def get_state(self):
        shapes = [(512, 418), (512,), (512,), (512,), (512,), (512,), (256, 512), (256,), (256,), (256,), (256,), (256,), (128, 256), (128,),
                  (6, 128), (6,)]
        arrs = [np.zeros(s, dtype=np.float32) for s in shapes]
        self.e._check(self.lib.ctd_train_get_state(self.h, self._ptrs(arrs)), "ctd_train_get_state")
        return dict(zip(STATE_KEYS, arrs))

    def get_grads(self):
        """Test hook: the gradients of the last optimiser step, keyed like the state_dict."""
        shapes = [(512, 418), (512,), (512,), (512,), (512,), (512,), (256, 512), (256,), (256,), (256,), (256,), (256,), (128, 256), (128,),
                  (6, 128), (6,)]
        arrs = [np.zeros(s, dtype=np.float32) for s in shapes]
        self.e._check(self.lib.ctd_train_get_grads(self.h, self._ptrs(arrs)), "ctd_train_get_grads")
        return dict(zip(STATE_KEYS, arrs))

    def epoch(self, seed, lr, perm):
        tl, el = ctypes.c_double(), ctypes.c_double()
        p = None if perm is None else np.ascontiguousarray(perm, dtype=np.uint32)
        self.e._check(self.lib.ctd_train_epoch(self.h, seed, float(lr), None if p is None else p.ctypes.data, ctypes.byref(tl), ctypes.byref(el)),
                      "ctd_train_epoch")
        return tl.value, el.value

    def close(self):
        self.lib.ctd_train_end(self.h)


def _stack(data, idx, dtype):
    return np.stack([np.asarray(item[idx].numpy() if hasattr(item[idx], "numpy") else item[idx], dtype=dtype) for item in data])


def train_node_value_only(train_data, val_data, epochs, lr, hidden_size=512, gamma=1.0, batch_size=64, device=None, parent_folder="pretrain",
                          verbose=False, model=None, seed=DEFAULT_SEED, engine=None, history=None):
    """algorithms/train.py:13-86.  -> best evaluation loss; writes <parent_folder>/best_model.pt.
    `model` (optional): a ValueOnlyNN(418, 512) whose weights are the starting point (default: a freshly initialised one, as in
    the reference); `history` (optional dict) receives the per-epoch train / eval losses, learning rates and the final state."""
    from .value_model import ValueOnlyNN
    if hidden_size != 512:
        raise ValueError("the training kernels are built for ValueOnlyNN(418, 512)")
    os.makedirs(parent_folder, exist_ok=True)
    model = model or ValueOnlyNN(418, hidden_size)
    own = engine is None
    eng = engine or Engine(capacity=8, device=0 if device in (None, "cuda", "cuda:0") else int(str(device).split(":")[-1]))
    tr = Trainer(eng, _stack(train_data, 0, np.float32), _stack(train_data, 2, np.float64), _stack(val_data, 0, np.float32),
                 _stack(val_data, 2, np.float64), batch_size)
    try:
        return _epochs(tr, model, epochs, lr, gamma, batch_size, seed, parent_folder, verbose, history)
    finally:
        tr.close()
        if own:
            eng.close()


def _epochs(tr, model, epochs, lr, gamma, batch_size, seed, parent_folder, verbose, history):
    """The epoch loop of train_node_value_only on a trainer that holds its rows: start from `model`'s weights, StepLR(300, gamma),
    <parent_folder>/best_model.pt at every new best evaluation loss.  -> best evaluation loss."""
    import torch
    train_losses, eval_losses, lrs = [], [], []
    best = float("inf")
    tr.set_state(model.state_dict())
    steps_per_epoch = (tr.n_train + batch_size - 1) // batch_size
    for epoch in range(epochs):
        cur_lr = lr * gamma ** (epoch // 300)                         # StepLR(step_size=300, gamma), stepped once per epoch
        tl, el = tr.epoch(seed, cur_lr, epoch_permutation(seed, epoch, tr.n_train))
        train_losses.append(tl)
        eval_losses.append(el)
        lrs.append(lr * gamma ** ((epoch + 1) // 300))                # scheduler.get_last_lr() after scheduler.step()
        if el < best:
            best = el
            sd = {k: torch.from_numpy(v.copy()) for k, v in tr.get_state().items()}
            for bn in ("bn1", "bn2"):
                sd[bn + ".num_batches_tracked"] = torch.tensor((epoch + 1) * steps_per_epoch, dtype=torch.long)
            ordered = {k: sd[k] for k in model.state_dict().keys()}
            torch.save(ordered, os.path.join(parent_folder, "best_model.pt"))
        if verbose:
            print("Epoch %d/%d - Train Loss: %.4f - Eval Loss: %.4f" % (epoch + 1, epochs, tl, el))
    if history is not None:
        history.update(train_losses=train_losses, eval_losses=eval_losses, learning_rates=lrs, final_state=tr.get_state())
    return best
