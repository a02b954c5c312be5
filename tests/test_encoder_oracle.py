"""The d-vector oracle (oracle/encoder_oracle.py): encoder against golden vectors from the notebook's unmodified classes,
mel filterbank against an independent implementation of librosa's definition."""
import glob
import os

import numpy as np
import pytest

from oracle import encoder_oracle as eo
from voicesplit_b200 import synth

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "encoder_*.npz")))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_encoder_oracle_matches_reference(path):
    g = np.load(path)
    sd = synth.make_encoder_state_dict(int(g["wseed"]), str(g["flavour"]))
    mels = synth.encoder_mel_inputs(int(g["iseed"]), [int(t) for t in g["frames"]])
    for mel, want in zip(mels, g["dvec"]):
        got = eo.speaker_encoder(sd, mel)
        assert np.abs(got - want).max() <= 2e-6            # reference ran in fp32; d-vector entries are ~0.06


def test_mel_filterbank_matches_independent_implementation():
    import torchaudio
    fb = torchaudio.functional.melscale_fbanks(n_freqs=601, f_min=0.0, f_max=8000.0, n_mels=40, sample_rate=16000, norm="slaney",
                                               mel_scale="slaney").T.numpy()
    mine = eo.mel_filterbank(16000, 1200, 40)
    assert mine.shape == (40, 601)
    assert np.abs(mine - fb).max() <= 1e-5 * np.abs(fb).max()            # torchaudio computes in fp32
    # every triangle integrates to ~1 in Hz (slaney normalisation): sum * bin width (sr / n_fft) == 1
    assert np.allclose(mine.sum(1) * (16000 / 1200), 1.0, atol=0.05)


def test_get_mel_shape_and_floor():
    y = synth.make_reference_audio(1, 16000, 3)[0]
    m = eo.get_mel(y)
    assert m.shape == (40, 101) and np.isfinite(m).all() and m.min() >= -6.0
    assert eo.get_mel(np.zeros(4000)).max() == pytest.approx(-6.0)      # log10(0 + 1e-6)


def test_too_short_reference_raises():
    with pytest.raises(ValueError):
        eo.speaker_encoder(synth.make_encoder_state_dict(1), np.zeros((40, 79)))
