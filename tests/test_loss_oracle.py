"""The loss-chain oracle (oracle/loss_oracle.py) against golden vectors made by the unmodified reference
(tests/golden/make_loss_golden.py): waveforms of the Q1 iSTFT, the Si-SNR loss value and the autograd gradient."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import loss_oracle
from voicesplit_b200.synth import loss_inputs

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "loss_*.npz")))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_loss_oracle_matches_reference(path):
    g = np.load(path)
    n_fft, hop, win, B, T = (int(g[k]) for k in ("n_fft", "hop", "win", "B", "T"))
    est, tgt, phase = loss_inputs(n_fft, B, T, int(g["seed"]))
    r = loss_oracle.loss_and_grad(est, tgt, phase, g["lengths"], n_fft, hop, win, float(g["min_db"]), float(g["ref_db"]), "q1")
    scale = np.abs(g["wav_est"]).max()
    assert np.abs(r["wav_est"] - g["wav_est"]).max() <= 2e-5 * scale        # reference ran in fp32
    assert np.abs(r["wav_tgt"] - g["wav_tgt"]).max() <= 2e-5 * np.abs(g["wav_tgt"]).max()
    assert abs(r["loss"] - float(g["loss"])) <= 2e-4
    gs = np.abs(g["grad_est"]).max()
    assert np.abs(r["grad_est"] - g["grad_est"]).max() <= 2e-4 * gs


def test_corrected_mode_inverts_a_real_stft():
    # the corrected mode is a true inverse: STFT (periodic Hann, centre, reflect) -> dB normalise -> spec2wav gives the signal back
    n_fft, hop, win = 128, 32, 64
    rng = np.random.Generator(np.random.PCG64(5))
    y = torch.from_numpy(rng.standard_normal((2, 32 * 20)) * 0.05)
    D = torch.stft(y, n_fft, hop, win, window=loss_oracle.hann(win, True), center=True, pad_mode="reflect", return_complex=True)  # [B,F,T]
    mag = D.abs().transpose(1, 2)
    spec = torch.clamp((20 * torch.log10(torch.clamp(mag, min=1e-5)) - 20.0) / 100.0, -1, 0) + 1
    w = loss_oracle.spec2wav(spec, torch.angle(D).transpose(1, 2), n_fft, hop, win, mode="corrected")
    assert (w - y).abs().max() < 1e-6 + 1e-3 * y.abs().max()              # only the 1e-5 magnitude floor / clipping differs


def test_lengths_mask_and_q1_differs_from_corrected():
    est, tgt, phase = loss_inputs(64, 2, 20, 3)
    L = 16 * 19
    a = loss_oracle.loss_and_grad(est, tgt, phase, np.array([L, L]), 64, 16, 32, mode="q1")
    b = loss_oracle.loss_and_grad(est, tgt, phase, np.array([L, L // 2]), 64, 16, 32, mode="q1")
    c = loss_oracle.loss_and_grad(est, tgt, phase, np.array([L, L]), 64, 16, 32, mode="corrected")
    assert abs(a["snr"][0] - b["snr"][0]) < 1e-9 and abs(a["snr"][1] - b["snr"][1]) > 1e-3
    assert abs(a["loss"] - c["loss"]) > 1e-2
    # clamp: no gradient where the estimate lies outside [0, 1]
    assert np.all(a["grad_est"][(est < 0) | (est > 1)] == 0)


def test_loss_oracle_against_the_live_reference_on_a_fresh_case():
    """Beyond the loss_*.npz goldens: another shape, against the unmodified reference chain's loss and gradient stored by
    tests/golden/make_reference_checks_golden.py."""
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_checks.npz"))
    ref_loss, ref_grad = float(z["loss_f129.loss"]), z["loss_f129.grad_est"]
    n_fft, hop, win, B, T = 256, 64, 128, 3, 23
    est, tgt, phase = loss_inputs(n_fft, B, T, 77)
    lens = np.array([hop * (T - 1), 1000, 333], dtype=np.int64)
    r = loss_oracle.loss_and_grad(est, tgt, phase, lens, n_fft, hop, win, mode="q1")
    assert abs(r["loss"] - ref_loss) <= 2e-4
    gs = float(np.abs(ref_grad).max())
    assert np.abs(r["grad_est"] - ref_grad).max() <= 2e-4 * gs
