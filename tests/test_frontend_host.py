"""Tacotron2's mel front end without a GPU: the fp64 oracle against torchaudio's filterbank and torch.stft, the module's
tables against the oracle, and the argument checks of TacotronSTFT, MelSpec(lengths=) and `cli vocode` / `cli score`."""
import numpy as np
import pytest
import torch
import torchaudio
from scipy.signal import get_window

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli
from constant_memory_waveglow_b200.condition import MelSpec, mel_lengths
from constant_memory_waveglow_b200.datasets import wav_write
from oracle import tacotron_stft as O

# (sr, n_fft, n_mels, fmin, fmax): the published Tacotron2 front end, and others
BANKS = [(22050, 1024, 80, 0.0, 8000.0), (16000, 256, 40, 50.0, None), (44100, 2048, 128, 0.0, 11025.0),
         (22050, 512, 80, 125.0, 7600.0)]


@pytest.mark.parametrize("sr,n_fft,n_mels,fmin,fmax", BANKS)
def test_oracle_mel_basis_matches_torchaudio(sr, n_fft, n_mels, fmin, fmax):
    want = torchaudio.functional.melscale_fbanks(n_fft // 2 + 1, fmin, fmax if fmax is not None else sr / 2, n_mels, sr,
                                                 norm="slaney", mel_scale="slaney").T.double()
    got = torch.from_numpy(O.mel_basis(sr, n_fft, n_mels, fmin, fmax))
    assert got.shape == want.shape
    # torchaudio computes in float32 and places the bins with linspace instead of rfftfreq
    assert (got - want).abs().max().item() < 1e-6


@pytest.mark.parametrize("sr,n_fft,n_mels,fmin,fmax", BANKS)
def test_module_mel_basis_is_the_oracle_rounded_once(sr, n_fft, n_mels, fmin, fmax):
    t = cm.TacotronSTFT(n_fft, n_fft // 4, n_fft, n_mels, sr, fmin, fmax)
    assert t.mel_basis.dtype == torch.float32 and t.mel_basis.shape == (n_mels, n_fft // 2 + 1)
    assert torch.equal(t.mel_basis, torch.from_numpy(O.mel_basis(sr, n_fft, n_mels, fmin, fmax)).float())
    assert list(t.state_dict()) == ["mel_basis"]


@pytest.mark.parametrize("n_fft,win", [(1024, 1024), (1024, 800), (256, 256), (2048, 2048)])
def test_window_is_scipy_periodic_hann(n_fft, win):
    t = cm.TacotronSTFT(n_fft, n_fft // 4, win)
    assert torch.allclose(t.window.double(), torch.from_numpy(get_window("hann", win, fftbins=True)), atol=1e-7, rtol=0)
    w = O.forward_basis(n_fft, win)[0, 0]                    # row 0 of the basis is the padded window itself
    left = (n_fft - win) // 2
    assert torch.equal(w[:left], torch.zeros(left, dtype=torch.float64))
    assert torch.allclose(w[left:left + win], torch.from_numpy(get_window("hann", win, fftbins=True)), atol=0, rtol=0)


@pytest.mark.parametrize("n_fft,hop,win,T", [(1024, 256, 1024, 7000), (256, 64, 256, 129), (2048, 512, 1600, 5000),
                                             (1024, 256, 1024, 513)])
def test_oracle_stft_matches_torch_stft(n_fft, hop, win, T):
    g = torch.Generator().manual_seed(T)
    y = torch.rand(2, T, generator=g, dtype=torch.float64) * 2 - 1
    mag = O.stft_magnitude(y, n_fft, hop, win)
    w = torch.from_numpy(get_window("hann", win, fftbins=True))
    S = torch.stft(y, n_fft, hop, win_length=win, window=w, center=True, pad_mode="reflect", onesided=True,
                   return_complex=True).abs()
    assert mag.shape == S.shape == (2, n_fft // 2 + 1, T // hop + 1)
    assert (mag - S).abs().max().item() <= 1e-12 * max(1.0, S.abs().max().item())


def test_oracle_mel_spectrogram_is_log_clamped_mel():
    y = torch.rand(1, 4000, generator=torch.Generator().manual_seed(0), dtype=torch.float64) * 2 - 1
    y[:, 1000:3000] = 0                                      # silent frames: the clamp at 1e-5 applies
    mel = O.mel_spectrogram(y)
    want = torch.log(torch.clamp(torch.from_numpy(O.mel_basis(22050, 1024, 80, 0.0, 8000.0)) @
                                 O.stft_magnitude(y, 1024, 256, 1024), min=1e-5))
    assert torch.equal(mel, want) and mel.shape == (1, 80, 4000 // 256 + 1)
    assert (mel == np.log(1e-5)).any()


def test_constructor_checks():
    with pytest.raises(NotImplementedError):
        cm.TacotronSTFT(filter_length=1000)
    with pytest.raises(ValueError):
        cm.TacotronSTFT(filter_length=1024, win_length=2048)
    with pytest.raises(ValueError):
        cm.TacotronSTFT(hop_length=0)


def test_lengths_checks():
    t = cm.TacotronSTFT()
    y = torch.zeros(3, 2000)
    for bad in ([2000, 2000], [2001, 600, 600], [512, 600, 600], [0, 600, 600], [600.0, 600, 600]):
        with pytest.raises((ValueError, TypeError)):
            t.mel_spectrogram(y, lengths=bad)
    with pytest.raises(ValueError, match="reflect padding"):
        t.mel_spectrogram(torch.zeros(1, 512))               # n_fft/2 = 512 samples: too short to reflect
    with pytest.raises(ValueError):
        t.mel_spectrogram(torch.zeros(2, 2, 600))
    assert mel_lengths(y, [513, 2000, 1024], 1024, 512, "t") == [513, 2000, 1024]
    # MelSpec pads (n_fft/2 - hop/2, n_fft/2 + hop/2): a length must exceed the larger pad
    m = MelSpec(22050, 1024, 256, n_mels=80)
    with pytest.raises(ValueError, match="reflect padding"):
        m(y, lengths=[640, 2000, 2000])
    assert mel_lengths(y, [641, 2000, 2000], 1024, 512 - 128, "MelSpec") == [641, 2000, 2000]


def test_cpu_tensors_raise():
    with pytest.raises(RuntimeError, match="CUDA"):
        cm.TacotronSTFT().mel_spectrogram(torch.zeros(2, 2000))
    with pytest.raises(RuntimeError, match="CUDA"):
        cm.TacotronSTFT().mel_spectrogram(torch.zeros(2, 2000), lengths=[2000, 1000])
    with pytest.raises(RuntimeError, match="CUDA"):
        MelSpec(22050, 1024, 256, n_mels=80)(torch.zeros(2, 2000), lengths=[2000, 1000])


def _nvidia_checkpoint(tmp_path):
    from oracle import nvidia_glow as NG
    cfg = dict(n_mel_channels=80, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
               WN_config=dict(n_layers=2, n_channels=32, kernel_size=3))
    path = tmp_path / "nv.pt"
    torch.save(NG.randomize(NG.WaveGlow(**cfg), seed=0).float().state_dict(), path)
    return str(path)


def _error(verb, argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main([verb] + argv)
    assert e.value.code == 2
    return capsys.readouterr().err


@pytest.mark.parametrize("verb", ["vocode", "score"])
def test_cli_refuses_a_wav_at_another_sampling_rate(verb, tmp_path, capsys):
    from tests.test_nvidia_host import TINY_WAVEGLOW, lightning_checkpoint
    wav = tmp_path / "a.wav"
    wav_write(str(wav), torch.zeros(1, 4000), 16000)
    out = [str(tmp_path / "out")] if verb == "vocode" else []
    err = _error(verb, [_nvidia_checkpoint(tmp_path)] + out + [str(wav)], capsys)
    assert "16000 Hz" in err and "22050 Hz" in err
    wav_write(str(wav), torch.zeros(1, 4000), 22050)        # the Lightning checkpoint's conditioner runs at 16 kHz
    err = _error(verb, [lightning_checkpoint(tmp_path, TINY_WAVEGLOW)] + out + [str(wav)], capsys)
    assert "22050 Hz" in err and "16000 Hz" in err


def test_cli_score_flags(tmp_path, capsys):
    wav = tmp_path / "a.wav"
    wav_write(str(wav), torch.zeros(1, 4000), 22050)
    assert "--max-batch" in _error("score", ["x.pt", str(wav), "--max-batch", "0"], capsys)
    assert "--sigma" in _error("score", ["x.pt", str(wav), "-s", "0"], capsys)
