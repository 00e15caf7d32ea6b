"""The reference script's training loop on the drop-in modules, on the GPU (SURVEY J1 / section 8b).

`tests/golden/script_trace.npz` holds the loss curve of the UNMODIFIED reference script (noisynet.py, q_a = q_w = 4,
I = 1 nA, batch 64, --seed 0) over its first 60 steps on a deterministic synthetic dataset, minted in the build
container by oracle/gen_script_trace.py.

  * test_script_equivalent_loop_matches_reference_trace drives the drop-in modules (NoisyConv2d / NoisyLinear /
    QuantMeasure / add_noise_calculate_power in the script's two-call flow, the script's AdamW groups, per-step weight
    clamp, np.random permutation, `input.max()` live ranges of quantize2 / quantize4) through the SAME steps on the
    same data and compares the loss curve with the reference's own.  The generators differ (Philox streams of this
    library vs. ATen's), so the comparison is by windows: mean loss of steps 0-9, 25-34 and 50-59 within 0.12 of the
    reference's, and the same downward trend.
"""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def _windows(losses):
    l = np.asarray(losses, dtype=np.float64)
    return np.array([l[0:10].mean(), l[25:35].mean(), l[50:60].mean()])


def _check_against_trace(losses, trace):
    ref = trace["losses"]
    assert len(losses) == len(ref) == 60 and np.all(np.isfinite(losses))
    w, wr = _windows(losses), _windows(ref)
    assert np.all(np.abs(w - wr) <= 0.12), (w, wr)
    assert w[2] < w[0] - 0.15 and wr[2] < wr[0] - 0.15, (w, wr)          # both learn


def test_script_equivalent_loop_matches_reference_trace(golden):
    from gen_script_trace import synthetic_learnable_cifar
    from noisynet_b200 import ops
    from noisynet_b200.net import NoisyNet, default_args, init_like_reference, make_optimizer, with_quant
    import __graft_entry__ as entry
    entry.build()
    trace = golden("script_trace")
    B, steps = int(trace["batch"]), int(trace["steps"])
    dev = torch.device("cuda:0")
    x, y = synthetic_learnable_cifar(50000, seed=int(trace["data_seed"]))
    train_inputs = torch.from_numpy(x.reshape(50000, 3, 32, 32)).to(dev)          # utils.py:143-153: whole set on the device
    train_labels = torch.from_numpy(y).to(dev)
    torch.manual_seed(0)                                                             # --seed 0 (noisynet.py:314-317)
    np.random.seed(int(trace["np_seed"]))
    a = with_quant(default_args(), 4, 4)
    model = init_like_reference(NoisyNet(a, fused=False, precision="bf16")).to(dev)  # the script's flow: layer, then noise call
    opt = make_optimizer(model, a)                                                   # noisynet.py:1135-1169
    model.train()
    rnd_idx = np.random.permutation(len(train_inputs))                               # noisynet.py:1232-1234
    train_inputs, train_labels = train_inputs[rnd_idx], train_labels[rnd_idx]
    losses = []
    for i in range(steps):
        inp = train_inputs[i * B:(i + 1) * B]
        lab = train_labels[i * B:(i + 1) * B]
        out = model(inp, 0, i)                                                       # :1276 (i < 20: side statistics collected)
        loss = torch.nn.CrossEntropyLoss()(out, lab)                                 # :1278
        opt.zero_grad()                                                              # :1346
        loss.backward()                                                              # :1372
        opt.step()                                                                   # :1520
        model.clamp_weights_()                                                       # :1527-1542
        losses.append(loss.item())
    assert ops.error_flag() == 0
    assert len(model.power[0]) == 20 and len(model.nsr[3]) == 20 and all(np.isfinite(model.power[1]))
    _check_against_trace(losses, trace)
