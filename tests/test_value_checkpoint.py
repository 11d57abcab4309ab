"""The reference's trained checkpoint (pretrain/best_model.pt; BatchNorm running_var 3.7e3 .. 6.8e4) through the value path.
tests/golden/value_best_model.npz (tests/golden/gen_value_fixture.py) holds its tensors, 1000 encoded states and what the
reference's own ValueOnlyNN + square_and_normalize give for them in torch fp32 on the CPU."""
import json
import os
import numpy as np
import pytest

from tests.golden_util import GOLDEN


def load():
    import torch
    from citadels_self_play_b200.value_model import ValueOnlyNN
    with np.load(os.path.join(GOLDEN, "value_best_model.npz")) as f:
        z = {k: f[k] for k in f.files}
    m = ValueOnlyNN(418, 512)
    m.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in z.items() if k.startswith("sd_")})   # the reference's state_dict keys
    m.eval()
    return z, m


def test_mirror_model_reproduces_the_reference_checkpoint_outputs():
    """state_dict compatibility on the real checkpoint: the mirror class gives the reference's outputs bit for bit (same torch,
    same CPU), and the BatchNorm folding the kernels rely on is exact to fp64 rounding."""
    import torch
    from citadels_self_play_b200.value_model import fold, reference_value
    z, m = load()
    x = z["features"].astype(np.float32)
    with torch.no_grad():
        assert np.array_equal(m(torch.from_numpy(x)).numpy(), z["raw"])
    assert np.array_equal(reference_value(m, x), z["leaf"])
    w1t, b1, w2t, b2, w3t, b3, w4t, b4 = [a.astype(np.float64) for a in fold(m)]
    xp = np.zeros((len(x), 448))
    xp[:, :418] = x
    h = np.maximum(xp @ w1t + b1, 0)
    h = np.maximum(h @ w2t + b2, 0)
    h = np.maximum(h @ w3t + b3, 0)
    y = h @ w4t + b4
    assert np.abs(y - z["raw"]).max() <= 2e-4 * np.abs(z["raw"]).max()      # fp32 weights after folding vs torch's unfolded fp32


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["tcgen05", "fp32"])
def test_value_kernels_on_the_reference_checkpoint(backend):
    """Both kernel families against torch fp32 on the trained checkpoint.  Two error measures, both printed with the
    test's output: (a) max |diff| relative to the output scale 5 (leaf values are 5 * p, p a
    distribution), (b) elementwise relative error over the entries that are not vanishing (want >= 0.05, i.e. p >= 1 %)."""
    from citadels_self_play_b200 import Engine
    z, m = load()
    x = z["features"].astype(np.float32)
    e = Engine(capacity=1024)
    try:
        e.set_value_model(m)
        e.set_value_backend(backend)
        got = e.value_eval(x)
    finally:
        e.close()
    want = z["leaf"]
    diff = np.abs(got.astype(np.float64) - want)
    big = want >= 0.05
    rep = dict(backend=backend, rows=len(x), max_abs=float(diff.max()), scale_rel=float(diff.max() / 5.0),
               elementwise_rel_max=float((diff[big] / want[big]).max()), elementwise_rel_p99=float(np.quantile(diff[big] / want[big], 0.99)),
               entries_compared_elementwise=int(big.sum()))
    print(json.dumps(rep))
    assert np.allclose(got.sum(1), 5.0, rtol=1e-5)
    assert rep["scale_rel"] <= 1e-5, rep            # north_star's 1e-5, of the output scale
    assert rep["elementwise_rel_max"] <= 1e-4, rep  # elementwise, entries >= 1 % of the mass
