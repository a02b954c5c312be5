"""The CPU oracle (oracle/voicesplit_oracle.c) against golden vectors produced by the unmodified
reference module (tests/golden/make_golden.py).  Tolerances: the oracle accumulates in double, the
reference in fp32 (oneDNN/MKL), so agreement is at fp32 rounding level."""
import os

import numpy as np

from conftest import ROOT
from oracle import oracle


def test_oracle_matches_reference_goldens(golden):
    out = oracle.forward(golden["state_dict"], golden["dims"], golden["x"], golden["emb"],
                         activation=golden["model_name"], want=("masked", "conv_out", "lstm_out", "dump"),
                         dump_layer=2)
    assert np.abs(out["conv_out"] - golden["conv_out"]).max() < 2e-4
    assert np.abs(out["dump"][:, ::7, :, ::5] - golden["act3_sample"]).max() < 2e-4
    assert np.abs(out["lstm_out"] - golden["lstm_out"]).max() < 2e-4
    # the stress weights amplify the reference's own fp32 rounding: its distance to exact
    # (double) arithmetic reaches ~2e-4 max on the mask; the stated parity tolerance is 1e-3
    assert np.abs(out["mask"] - golden["mask"]).max() < 1e-3
    assert np.abs(out["mask"] - golden["mask"]).mean() < 2e-5
    assert np.abs(out["masked"] - golden["masked"]).max() < 1e-3


def test_activation_matches_torch():
    import torch
    import torch.nn.functional as F
    x = np.concatenate([np.linspace(-30, 30, 2001), [19.99, 20.0, 20.01, 0.0, -0.0]]).astype(np.float32)
    xt = torch.from_numpy(x)
    ref = (xt * torch.tanh(F.softplus(xt))).numpy()      # reference utils/generic_utils.py:399
    assert np.abs(oracle.activation(x, "mish") - ref).max() < 2e-6
    assert np.array_equal(oracle.activation(x, "relu"), np.maximum(x, 0))


def test_oracle_matches_live_reference_train_shape():
    """A shape that is not in the case_*.npz goldens, against the reference's mask stored by
    tests/golden/make_reference_checks_golden.py."""
    from voicesplit_b200 import synth
    dims = synth.make_dims(29, 12, 20, 28)
    sd = synth.make_state_dict(dims, 77, "stress")
    x, emb = synth.make_inputs(2, 53, dims, 5)
    ref = np.load(os.path.join(ROOT, "tests", "golden", "reference_checks.npz"))["oracle_f29.mask"]
    got = oracle.forward(sd, dims, x, emb)["mask"]
    assert np.abs(got - ref).max() < 1e-3 and np.abs(got - ref).mean() < 2e-5


def test_torch_port_matches_reference_goldens(golden):
    """The multi-threaded CPU baseline (oracle/torch_port.py) against the same golden vectors."""
    from oracle import torch_port
    got = torch_port.forward(golden["state_dict"], golden["x"], golden["emb"], golden["model_name"]).numpy()
    assert np.abs(got - golden["mask"]).max() < 2e-5
