"""CPU: pins the oracle (oracle/convnext_oracle.py) against the reference, through the committed golden fixtures
(outputs of the UNMODIFIED reference, oracle/make_golden.py).
The reference ships no tests / golden vectors of its own for this path (SURVEY.md 8c).
"""
import os

import numpy as np
import pytest
import torch

from oracle import convnext_oracle as O
from oracle import weights


def _demo_wave(g):
    return torch.from_numpy(g["pcm"].astype(np.float32) / 32768.0)[None]


def test_oracle_matches_golden_demo_clip(golden_dir, parity_sd):
    g = np.load(os.path.join(golden_dir, "demo_clip.npz"))
    wave = _demo_wave(g)
    taps = {}
    out = O.forward(wave, parity_sd, taps=taps)
    assert np.abs(out["clipwise_logits"].numpy() - g["logits"]).max() < 2e-5
    assert np.abs(out["clipwise_output"].numpy() - g["probs"]).max() < 1e-5
    assert np.abs(taps["scene"].numpy() - g["scene"]).max() < 2e-5
    frame = O.forward_frame_embeddings(wave, parity_sd)
    assert frame.shape == (1, 768, 31, 7)                      # README.md:61
    assert np.abs(frame.numpy() - g["frame"]).max() < 5e-5
    lm = taps["logmel_bn"].numpy()[:, :: int(g["logmel_stride"])]
    assert np.abs(lm - g["logmel_bn"]).max() < 1e-4
    labels = np.where(out["clipwise_output"][0].numpy() > 0.25)[0]
    assert np.array_equal(labels, g["labels"])                 # thresholded label set, demo_convnext.py:87-88


@pytest.mark.parametrize("kind", ["noise", "tones"])
def test_oracle_matches_golden_synthetic(golden_dir, parity_sd, kind):
    g = np.load(os.path.join(golden_dir, f"synth_{kind}.npz"))
    wave = weights.make_waveforms(2, kind=kind, seed=0)
    cks = np.array([wave.double().sum().item(), wave.double().abs().sum().item()])
    assert np.allclose(cks, g["wave_cks"], rtol=1e-12)
    out = O.forward(wave, parity_sd)
    assert np.abs(out["clipwise_logits"].numpy() - g["logits"]).max() < 2e-5
    frame = O.forward_frame_embeddings(wave, parity_sd).numpy()
    assert np.abs(frame[:, :, :: int(g["frame_stride"])] - g["frame_t0"]).max() < 5e-5


def test_oracle_variable_length(golden_dir, parity_sd):
    g = np.load(os.path.join(golden_dir, "synth_short.npz"))
    wave = weights.make_waveforms(1, n_samples=int(g["n_samples"]), kind="noise", seed=3)
    frame = O.forward_frame_embeddings(wave, parity_sd).numpy()
    assert frame.shape == g["frame"].shape
    assert np.abs(frame - g["frame"]).max() < 5e-5
    assert np.abs(O.forward(wave, parity_sd)["clipwise_logits"].numpy() - g["logits"]).max() < 2e-5


def test_oracle_fp64_close_to_fp32(parity_sd):
    """The fp64 evaluation of the same formulas is the 'truth' used for error budgets."""
    wave = weights.make_waveforms(1, n_samples=32000, kind="tones", seed=5)
    a = O.forward(wave, parity_sd, torch.float32)["clipwise_logits"]
    b = O.forward(wave, parity_sd, torch.float64)["clipwise_logits"]
    assert (a.double() - b).abs().max() < 5e-4


# ---- the torchlibrosa / librosa restatement (the one piece the reference does not contain) pinned by independent code ----
def test_shim_mel_filterbank_equals_torchaudio_slaney():
    """librosa.filters.mel(32000, 1024, 224, 50, 14000) (htk=False, norm='slaney') restated in the shim ==
    torchaudio.functional.melscale_fbanks(513, 50, 14000, 224, 32000, 'slaney', 'slaney') -- an independent
    implementation of the same published definition.  This is `logmel_extractor.melW` (CX:190-200)."""
    TAF = pytest.importorskip("torchaudio.functional")
    from oracle.torchlibrosa_shim.torchlibrosa.stft import librosa_mel
    ours = torch.from_numpy(librosa_mel(32000, 1024, 224, 50, 14000).T.copy())             # (513, 224) like melW
    ref = TAF.melscale_fbanks(513, 50.0, 14000.0, 224, 32000, norm="slaney", mel_scale="slaney")
    assert ours.shape == ref.shape == (513, 224)
    assert (ours - ref).abs().max().item() < 1e-6
    _, _, melW = weights.frontend_constants()
    assert torch.equal(melW, ours)
    # structure the fused front end relies on: non-zero rows only inside [fmin, fmax], every filter non-empty
    nz = (ours.abs().sum(1) > 0).nonzero().flatten()
    assert nz.min().item() >= 1 and nz.max().item() <= 448 and (ours.sum(0) > 0).all()


def test_shim_stft_equals_torch_stft():
    """The shim's conv1d-DFT (periodic Hann, reflect pad 512, hop 320, W = omega^(x*y)) == torch.stft with the
    same parameters (an FFT, not a matrix product): pins conv_real / conv_imag (CX:179-187) and the framing."""
    from oracle.torchlibrosa_shim.torchlibrosa.stft import STFT, Spectrogram
    torch.manual_seed(0)
    wave = torch.cat([weights.make_waveforms(1, n_samples=48000, kind="tones", seed=2),
                      weights.make_waveforms(1, n_samples=48000, kind="noise", seed=2)])
    real, imag = STFT(n_fft=1024, hop_length=320, win_length=1024, window="hann", center=True, pad_mode="reflect")(wave)
    ref = torch.stft(wave.double(), 1024, hop_length=320, win_length=1024,
                     window=torch.hann_window(1024, periodic=True, dtype=torch.float64), center=True,
                     pad_mode="reflect", return_complex=True)                    # (B, 513, T)
    assert real.shape == (2, 1, 151, 513)
    scale = ref.abs().max().item()
    assert (real[:, 0].double() - ref.real.transpose(1, 2)).abs().max().item() < 2e-6 * scale
    assert (imag[:, 0].double() - ref.imag.transpose(1, 2)).abs().max().item() < 2e-6 * scale
    # and the oracle's functional form == the shim module (what the unmodified reference instantiates)
    sd = weights.make_state_dict("init", 0)
    p_mod = Spectrogram(n_fft=1024, hop_length=320, win_length=1024)(wave)[:, 0]
    assert torch.equal(O.spectrogram(wave, sd), p_mod)
    # fp64 power spectrum of the oracle against |torch.stft|^2 (the error budget's "truth")
    p64 = O.spectrogram(wave, sd, torch.float64)
    assert (p64 - (ref.abs() ** 2).transpose(1, 2)).abs().max().item() < 1e-6 * scale ** 2


def test_stock_head_fixture_matches_oracle(golden_dir):
    """parity_stock_head.npz (gamma ~ U(0.1,0.6), head std 0.02; outputs of the unmodified reference) vs the oracle."""
    g = np.load(os.path.join(golden_dir, "parity_stock_head.npz"))
    sd = weights.make_state_dict("parity_stock_head", int(g["parity_seed"]))
    for k in ("head_audioset.weight", "stages.3.2.gamma"):
        t = sd[k].double()
        assert np.allclose([t.sum().item(), t.abs().sum().item()], g["cks/" + k], rtol=1e-12, atol=1e-9)
    assert abs(sd["head_audioset.weight"].std().item() - 0.02) < 2e-4          # the reference's own init width
    wave = weights.make_waveforms(2, kind="tones", seed=0)
    out = O.forward(wave[:, :], sd)
    assert np.abs(out["clipwise_logits"].numpy() - g["tones/logits"]).max() < 2e-5
