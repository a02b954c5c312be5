"""Outputs of the UNMODIFIED reference code (CPU, fp32) for the tests that once compared against a live reference tree: the
reference classes' state_dict layouts, its config.json as its own load_config reads it, the GE2E checkpoint's layout, a mask at a
shape that is not in case_*.npz, two training-mode steps at that shape, SiSNR_With_Pit with C = 1, 2, 3 sources and the Q1 loss
chain at another shape.  Needs a checkout of the reference (the path oracle/ref_import.REF_ROOT names):

    python tests/golden/make_reference_checks_golden.py

Writes tests/golden/reference_checks.npz, reference_layouts.json and reference_config.json (the reference's config.json,
byte for byte: the input of tests/test_host.py::test_reference_config_json_builds_module).  Weights and inputs are regenerated from
the seeds below by voicesplit_b200.synth (numpy PCG64) and torch generators in the tests themselves, not stored.
"""
import importlib.util
import json
import os
import re
import shutil
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from voicesplit_b200 import synth  # noqa: E402
from voicesplit_b200.synth import loss_inputs  # noqa: E402

# training-mode gradients with more elements than SAMPLE_ABOVE are stored as every SAMPLE_STRIDE-th element (a prime, so the
# sample walks through every filter tap and gate) plus the float64 sum and sum of squares of the whole tensor
SAMPLE_ABOVE, SAMPLE_STRIDE = 4096, 197
CONV_BIAS = tuple(f"conv.{i}.bias" for i in (1, 5, 9, 13, 17, 21, 25, 28))


def _layout(sd):
    return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]


def layouts(VoiceSplit, VoiceFilter, gu):
    out = {}
    dims = synth.make_dims(33, 16, 24, 40)
    for name, cls in (("VoiceSplit", VoiceSplit), ("VoiceFilter", VoiceFilter)):
        m = cls(gu.AttrDict(synth.make_config_dict(dims)))
        out[name] = {"dims": [33, 16, 24, 40], "state_dict": _layout(m.state_dict()), "n_parameters": len(list(m.parameters()))}
    cfg = os.path.join(ref_import.REF_ROOT, "config.json")
    out["config_json"] = dict(gu.load_config(cfg))
    ck = torch.load(os.path.join(ref_import.REF_ROOT, "notebooks", "embedder.pt"), map_location="cpu")
    out["embedder_checkpoint"] = _layout(ck)
    shutil.copyfile(cfg, os.path.join(HERE, "reference_config.json"))
    return out


def oracle_shape(VoiceSplit, gu):
    """tests/test_oracle.py::test_oracle_matches_live_reference_train_shape"""
    dims = synth.make_dims(29, 12, 20, 28)
    model = VoiceSplit(gu.AttrDict(synth.make_config_dict(dims))).eval()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in synth.make_state_dict(dims, 77, "stress").items()})
    x, emb = synth.make_inputs(2, 53, dims, 5)
    with torch.no_grad():
        return {"oracle_f29.mask": model(torch.from_numpy(x), torch.from_numpy(emb)).numpy()}


def train_shape(VoiceSplit, gu):
    """tests/test_train_oracle.py::test_forward_train_matches_the_live_reference_on_a_fresh_shape: two consecutive steps"""
    dims = synth.make_dims(29, 12, 20, 28)
    B, T = 2, 26
    model = VoiceSplit(gu.AttrDict(synth.make_config_dict(dims)))
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in synth.make_state_dict(dims, 41, "stress").items()})
    model.train()
    out = {}
    for step in range(2):
        x, emb = synth.make_inputs(B, T, dims, 50 + step)
        gw = torch.from_numpy(np.random.default_rng(step).standard_normal((B, T, dims["num_freq"])).astype(np.float32))
        model.zero_grad()
        (model(torch.from_numpy(x), torch.from_numpy(emb)) * gw).sum().backward()
        pre = f"train_f29.step{step}."
        for k, p in model.named_parameters():
            if k in CONV_BIAS:
                continue                                    # analytically zero in front of a batch-statistics BatchNorm
            g = p.grad.numpy()
            if g.size > SAMPLE_ABOVE:
                g64 = g.astype(np.float64)
                out[pre + "gradsample." + k] = g.reshape(-1)[::SAMPLE_STRIDE].copy()
                out[pre + "gradstats." + k] = np.array([np.abs(g64).max(), g64.sum(), (g64 ** 2).sum()])
            else:
                out[pre + "grad." + k] = g.copy()
        for k, v in model.state_dict().items():
            if "running" in k or "num_batches" in k:
                out[pre + "buf." + k] = v.numpy().copy()
    return out


def si_snr(gu):
    """tests/test_dist_cpu.py::test_si_snr_matches_reference_formula and ::test_general_pit_matches_the_live_reference_with_gradients"""
    torch.manual_seed(1)
    est, src = torch.randn(3, 1, 500), torch.randn(3, 1, 500)
    out = {"sisnr_c1.loss": np.float32(gu.SiSNR_With_Pit()(est.clone(), src.clone(), torch.tensor([500, 321, 77])))}
    for C in (2, 3):
        g = torch.Generator().manual_seed(7 + C)
        src = torch.randn(4, C, 400, generator=g)
        mix = torch.randn(4, C, C, generator=g) * 0.3 + torch.eye(C)[torch.randperm(C, generator=g)]
        est0 = torch.einsum("bij,bjl->bil", mix, src) + 0.1 * torch.randn(4, C, 400, generator=g)
        b = est0.clone().requires_grad_(True)
        ref = gu.SiSNR_With_Pit()(b * 1.0, src.clone(), torch.tensor([400, 399, 123, 57]))
        ref.backward()
        out[f"sisnr_c{C}.loss"] = np.float32(ref.detach())
        out[f"sisnr_c{C}.grad"] = b.grad.numpy().copy()
    return out


def loss_chain():
    """tests/test_loss_oracle.py::test_loss_oracle_against_the_live_reference_on_a_fresh_case"""
    spec = importlib.util.spec_from_file_location("_make_loss_golden", os.path.join(HERE, "make_loss_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    apm, gu = gen.load_reference_audio_processor()
    n_fft, hop, win, B, T = 256, 64, 128, 3, 23
    ap = apm.openVoiceFilterAudioProcessor(sample_rate=16000, n_fft=n_fft, num_freq=n_fft // 2 + 1, hop_length=hop, win_length=win, preemphasis=0.97,
                                           power=1.5, min_level_db=-100.0, ref_level_db=20.0, num_mels=40, griffin_lim_iters=60)
    est, tgt, phase = loss_inputs(n_fft, B, T, 77)
    lens = np.array([hop * (T - 1), 1000, 333], dtype=np.int64)
    e = torch.from_numpy(est).requires_grad_(True)
    out = ap.torch_inv_spectrogram(e, torch.from_numpy(phase))
    ref = ap.torch_inv_spectrogram(torch.from_numpy(tgt), torch.from_numpy(phase))
    loss = gu.SiSNR_With_Pit()(out[:, None, :], ref[:, None, :], torch.from_numpy(lens))
    loss.backward()
    return {"loss_f129.loss": np.float32(loss.detach()), "loss_f129.grad_est": e.grad.numpy().copy()}


def main():
    VoiceSplit, VoiceFilter, gu = ref_import.load()
    text, prev = json.dumps(layouts(VoiceSplit, VoiceFilter, gu), indent=1), None
    while text != prev:                                 # one line per list that holds no dict: one state_dict entry per line
        prev = text
        text = re.sub(r"\[\n\s*((?:[^\[\]{}]|\[[^\[\]{}\n]*\])*?)\n\s*\]", lambda m: "[" + re.sub(r",\n\s*", ", ", m.group(1)) + "]", text)
    with open(os.path.join(HERE, "reference_layouts.json"), "w") as f:
        f.write(text + "\n")
    arrays = {**oracle_shape(VoiceSplit, gu), **train_shape(VoiceSplit, gu), **si_snr(gu), **loss_chain()}
    path = os.path.join(HERE, "reference_checks.npz")
    np.savez_compressed(path, torch_version=torch.__version__, sample_stride=SAMPLE_STRIDE, **arrays)
    print(len(arrays), "arrays,", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
