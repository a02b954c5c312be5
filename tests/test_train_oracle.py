"""Pins the TRAINING-mode checker: oracle/torch_port.forward_train (+ torch autograd) - what the GPU gradient tests
(tests/test_gpu_train.py, tests/test_gpu_dp.py) compare the device against - must reproduce the golden vectors produced by the
UNMODIFIED reference modules in `.train()` mode (tests/golden/make_train_golden.py; reference models/voicesplit/model.py:15-89 as
driven by train.py:84,94,108-110): mask, the gradient of every one of the 44 parameters, of x and of the d-vector, and the
BatchNorm buffers after the step.  Both sides run the same ATen kernels in fp32 on a CPU, so agreement is at rounding level; the
bound is relative to each tensor's own scale."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import torch_port
from voicesplit_b200 import synth

CASES = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "train_*.npz")))


def _run_port(model_name, dims, flavour, wseed, iseed, gseed, B, T):
    sd = {}
    for k, v in synth.make_state_dict(dims, wseed, flavour).items():
        t = torch.from_numpy(np.array(v))
        if t.dtype == torch.float32 and "running" not in k:
            t.requires_grad_(True)
        sd[k] = t
    x, emb = synth.make_inputs(B, T, dims, iseed)
    xt, et = torch.from_numpy(x).requires_grad_(True), torch.from_numpy(emb).requires_grad_(True)
    mask = torch_port.forward_train(sd, xt, et, model_name)
    gw = np.random.default_rng(gseed).standard_normal((B, T, dims["num_freq"])).astype(np.float32)
    (mask * torch.from_numpy(gw)).sum().backward()
    return mask.detach().numpy(), sd, xt.grad.numpy(), et.grad.numpy()


def _close(got, want, what, rel=2e-4):
    scale = max(float(np.abs(want).max()), 1e-30)
    err = float(np.abs(got - want).max())
    assert err <= rel * scale + 1e-7, (what, err, scale)


def test_fixtures_exist():
    assert len(CASES) == 3


@pytest.mark.parametrize("path", CASES, ids=lambda p: os.path.basename(p)[6:-4])
def test_forward_train_matches_the_reference_in_train_mode(path):
    z = np.load(path)
    d = [int(v) for v in z["dims"]]
    dims = synth.make_dims(*d)
    mask, sd, gx, gemb = _run_port(str(z["model_name"]), dims, str(z["flavour"]), int(z["wseed"]), int(z["iseed"]), int(z["gseed"]),
                                   int(z["B"]), int(z["T"]))
    _close(mask, z["mask"], "mask", rel=2e-5)
    _close(gx, z["grad_x"], "grad_x")
    _close(gemb, z["grad_emb"], "grad_emb")
    seen = 0
    # a conv bias in front of a batch-statistics BatchNorm has an analytically zero gradient: both sides hold rounding noise there,
    # judged on the scale of the layer's weight gradient (same rule as tests/test_gpu_train.py)
    conv_bias = {f"conv.{i}.bias": f"conv.{i}.weight" for i in (1, 5, 9, 13, 17, 21, 25, 28)}
    wscale = {}
    for k in z.files:
        if k.startswith("grad.") or k.startswith("gradsample."):
            wscale[k.split(".", 1)[1]] = float(np.abs(z[k]).max())
    for k in z.files:
        if k.startswith("grad."):
            name = k[5:]
            g = sd[name].grad.numpy()
            if name in conv_bias:
                assert np.abs(g - z[k]).max() <= 2e-4 * max(wscale[name], wscale[conv_bias[name]]) + 1e-7, name
            else:
                _close(g, z[k], name)
            seen += 1
        elif k.startswith("gradsample."):
            name = k[11:]
            g = sd[name].grad.numpy()
            _close(g.reshape(-1)[::4], z[k], name)
            s, s2 = z["gradmoments." + name]
            g64 = g.astype(np.float64)
            assert abs(g64.sum() - s) <= 2e-4 * np.sqrt(s2 * g.size) and abs((g64 ** 2).sum() - s2) <= 4e-4 * s2, name
            seen += 1
        elif k.startswith("buf."):
            name = k[4:]
            if "num_batches" in name:
                assert int(sd[name]) == int(z[k]) == 1
            else:
                _close(sd[name].detach().numpy(), z[k], name, rel=1e-5)
    assert seen == 44


def test_forward_train_matches_the_live_reference_on_a_fresh_shape():
    """A shape and seeds that are not in the fixtures, two consecutive steps (the second one starts from updated running buffers),
    against the reference's gradients and buffers stored by tests/golden/make_reference_checks_golden.py (the large weight
    gradients as a strided sample plus the max |g|, sum and sum of squares of the whole tensor)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "reference_checks.npz"))
    stride = int(z["sample_stride"])
    dims = synth.make_dims(29, 12, 20, 28)
    B, T = 2, 26
    sd_np = synth.make_state_dict(dims, 41, "stress")
    sd = {}
    for k, v in sd_np.items():
        t = torch.from_numpy(np.array(v))
        sd[k] = t.requires_grad_(True) if (t.dtype == torch.float32 and "running" not in k) else t
    for step in range(2):
        x, emb = synth.make_inputs(B, T, dims, 50 + step)
        gw = torch.from_numpy(np.random.default_rng(step).standard_normal((B, T, dims["num_freq"])).astype(np.float32))
        for t in sd.values():
            t.grad = None
        (torch_port.forward_train(sd, torch.from_numpy(x), torch.from_numpy(emb)) * gw).sum().backward()
        pre, seen = f"train_f29.step{step}.", 0
        for k in z.files:
            if not k.startswith(pre):
                continue
            kind, name = k[len(pre):].split(".", 1)
            if kind == "grad":
                _close(sd[name].grad.numpy(), z[k], (step, name))
                seen += 1
            elif kind == "gradsample":
                g = sd[name].grad.numpy()
                gmax, s, s2 = z[pre + "gradstats." + name]
                err = float(np.abs(g.reshape(-1)[::stride] - z[k]).max())
                assert err <= 2e-4 * gmax + 1e-7, (step, name, err, gmax)
                g64 = g.astype(np.float64)
                assert abs(np.abs(g64).max() - gmax) <= 2e-4 * gmax + 1e-7, (step, name)
                assert abs(g64.sum() - s) <= 2e-4 * np.sqrt(s2 * g.size) and abs((g64 ** 2).sum() - s2) <= 4e-4 * s2, (step, name)
                seen += 1
            elif kind == "buf":
                if "running" in name:
                    _close(sd[name].detach().numpy(), z[k], (step, name), rel=1e-5)
                else:
                    assert int(sd[name]) == int(z[k]) == step + 1
        assert seen == 36                                   # 44 parameters less the 8 conv biases, analytically zero (see above)
