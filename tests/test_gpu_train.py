"""Value-network training on the device (citadels_self_play_b200.train, csrc/ctd_train.cuh) against the REAL reference's
train_node_value_only (algorithms/train.py:13-86): tests/golden/train_value_net.npz (tests/golden/gen_train_fixture.py) holds, for
8 epochs over 5000 targets with the same initial weights, batch order and dropout masks, the reference's first-step loss and
gradients, its loss curve and its best_model.pt.

What can agree and what cannot.  At EQUAL weights (the first optimiser step) the loss agrees to 1e-6 and every gradient tensor to a
few 1e-3 of its norm -- not tighter, for either side: the loss is KL(t || y^2 / sum y^2), its gradient carries 1 / p, and the rows
that dominate a batch's gradient are the ones where the network puts p ~ 1e-9 on a seat the target gives 0.7 (one such row weighs
as much as thousands of ordinary ones); p there comes from an output y ~ 1e-5 that is a cancelling fp32 sum, so its last bits -- the
summation order of the GEMM -- move the whole batch gradient by ~1e-3.  torch on the CPU against torch on a GPU differs by as
much.  From there Adam (steps of ~lr whatever a gradient's size, lr a third of a typical weight) makes the two runs different
samples of the same training: the curves stay within ~15 % of each other and end in the same place, which is what is gated."""
import json
import os
import numpy as np
import pytest

from tests.golden_util import GOLDEN

pytestmark = pytest.mark.gpu


def _fixture():
    with np.load(os.path.join(GOLDEN, "train_value_net.npz")) as f:
        return {k: f[k] for k in f.files}


def test_first_step_loss_and_gradients_match_the_reference():
    import torch
    from citadels_self_play_b200 import Engine, train as T
    from citadels_self_play_b200.value_model import ValueOnlyNN
    z = _fixture()
    perm = T.epoch_permutation(int(z["seed"]), 0, len(z["train_x"]))[:int(z["batch"])]       # the reference's first batch
    x, v = z["train_x"][perm].astype(np.float32), z["train_v"][perm]
    torch.manual_seed(int(z["init_seed"]))
    eng = Engine(capacity=8)
    tr = T.Trainer(eng, x, v, x[:8], v[:8], int(z["batch"]))
    try:
        tr.set_state(ValueOnlyNN(418, 512).state_dict())
        loss, _ = tr.epoch(int(z["seed"]), 1e-12, None)
        g = tr.get_grads()
    finally:
        tr.close()
        eng.close()
    rep = {"first_loss_rel": abs(loss / float(z["first_loss"]) - 1)}
    for k in ("fc1.weight", "bn1.weight", "bn1.bias", "fc2.weight", "bn2.weight", "bn2.bias", "fc3.weight", "fc3.bias", "fc4.weight", "fc4.bias"):
        if "g_" + k in z:
            rep["g_" + k] = float(np.linalg.norm(g[k] - z["g_" + k]) / np.linalg.norm(z["g_" + k]))
        else:
            probe = g[k].reshape(-1)[z["g_" + k + "_probe_idx"]]
            rep["g_" + k] = float(max(np.linalg.norm(probe - z["g_" + k + "_probe"]) / np.linalg.norm(z["g_" + k + "_probe"]),
                                      np.linalg.norm(g[k].sum(1) - z["g_" + k + "_rowsum"]) / np.linalg.norm(z["g_" + k + "_rowsum"]),
                                      abs(np.sqrt((g[k].astype(np.float64) ** 2).sum()) / float(z["g_" + k + "_norm"]) - 1)))
    # fc1.bias / fc2.bias feed a BatchNorm: their true gradient is zero, both sides hold rounding noise of the same size
    for k in ("fc1.bias", "fc2.bias"):
        rep["g_" + k + "_abs"] = float(np.abs(g[k]).max())
        assert np.abs(g[k]).max() < 1e-5 and float(z["g_" + k + "_norm"]) < 1e-5
    print(json.dumps(rep, indent=1))
    assert rep["first_loss_rel"] <= 1e-5, rep
    assert all(val <= 1e-2 for key, val in rep.items() if key.startswith("g_") and not key.endswith("_abs")), rep


def test_training_run_tracks_the_reference(tmp_path):
    import torch
    from citadels_self_play_b200 import train as T
    from citadels_self_play_b200.value_model import ValueOnlyNN, load_checkpoint
    z = _fixture()
    tr = [(torch.from_numpy(x.astype(np.float32)), None, torch.from_numpy(v), None) for x, v in zip(z["train_x"], z["train_v"])]
    va = [(torch.from_numpy(x.astype(np.float32)), None, torch.from_numpy(v), None) for x, v in zip(z["val_x"], z["val_v"])]
    torch.manual_seed(int(z["init_seed"]))
    hist = {}
    best = T.train_node_value_only(tr, va, epochs=int(z["epochs"]), lr=float(z["lr"]), hidden_size=512, gamma=float(z["gamma"]),
                                   batch_size=int(z["batch"]), parent_folder=str(tmp_path), model=ValueOnlyNN(418, 512), seed=int(z["seed"]),
                                   history=hist)
    tl, el = np.array(hist["train_losses"]), np.array(hist["eval_losses"])
    rep = dict(train_rel=float(np.abs(tl / z["train_losses"] - 1).max()), eval_rel=float(np.abs(el / z["eval_losses"] - 1).max()),
               train_losses=tl.tolist(), eval_losses=el.tolist(), ref_train_losses=z["train_losses"].tolist(),
               ref_eval_losses=z["eval_losses"].tolist(), best_eval=best, ref_best_eval=float(z["best_eval"]))
    print(json.dumps(rep, indent=1))
    assert abs(tl[0] / z["train_losses"][0] - 1) <= 0.03          # the first epoch is three steps from equal weights
    assert rep["train_rel"] <= 0.25 and rep["eval_rel"] <= 0.25, rep
    assert tl[-1] < 0.6 * tl[0] and el[-1] < el[0]               # it learns, like the reference does (0.74 / 1.99, 0.83 / 1.41)
    assert best == el.min()
    # the checkpoint is what run_utils.setup_model_for_eval loads (run_utils.py:11-18): reference keys, eval mode
    m = load_checkpoint(os.path.join(str(tmp_path), "best_model.pt"))
    assert not m.training
    sd = torch.load(os.path.join(str(tmp_path), "best_model.pt"))
    assert list(sd.keys()) == list(ValueOnlyNN(418, 512).state_dict().keys())
    assert int(sd["bn1.num_batches_tracked"]) == int(z["w_bn1.num_batches_tracked"])
