"""Spectral distances without a GPU: the fp64 oracle against an independent restatement on torch.stft, its identities, the
DCT, the argument checks of SpectralDistance and of cmwg_spectral_distance, and the usage errors of `cli compare`."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from scipy.fft import dct

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import _lib, cli
from constant_memory_waveglow_b200.datasets import wav_write
from constant_memory_waveglow_b200.distance import dct_matrix
from oracle import distance_oracle as O
from oracle import tacotron_stft as TS

ERR_ARG, ERR_UNSUPPORTED = -1, -3


def _noise(n, seed):
    return np.random.default_rng(seed).uniform(-1, 1, n)


def _harmonic_with_silence(n, seed):
    """Three partials with exact-zero stretches: the silent frames hit both clamps (1e-10 on the power, 1e-5 on the mel)."""
    t = np.arange(n) / 22050.0
    x = 0.3 * np.sin(2 * np.pi * 220 * t) + 0.2 * np.sin(2 * np.pi * 660 * t) + 0.1 * np.sin(2 * np.pi * 1100 * t + seed)
    x[n // 4:n // 2] = 0.0
    x[-(n // 8):] = 0.0
    return x


def _torch_restatement(ref, est, n_fft=1024, hop=256, win=1024, sr=22050, n_mels=80, fmin=0.0, fmax=8000.0, n_cep=25):
    """The three distances from torch.stft(center=True, pad_mode='reflect') in float64, written apart from the oracle."""
    w = torch.hann_window(win, periodic=True, dtype=torch.float64)
    spec = [torch.stft(torch.from_numpy(np.asarray(s, dtype=np.float64)), n_fft, hop, win_length=win, window=w,
                       center=True, pad_mode="reflect", onesided=True, return_complex=True) for s in (ref, est)]
    P = [s.real ** 2 + s.imag ** 2 for s in spec]
    X = [torch.log10(torch.clamp(p, min=1e-10)) for p in P]
    lsd = torch.sqrt(((X[0] - X[1]) ** 2).mean(0)).mean()
    basis = torch.from_numpy(TS.mel_basis(sr, n_fft, n_mels, fmin, fmax))
    m = [torch.log(torch.clamp(basis @ s.abs(), min=1e-5)) for s in spec]
    mel_l1 = (m[0] - m[1]).abs().mean(0).mean()
    D = torch.from_numpy(dct(np.eye(n_mels), norm="ortho", axis=0)[1:n_cep])
    mcd = (10 / math.log(10) * torch.sqrt(2 * ((D @ (m[0] - m[1])) ** 2).sum(0))).mean()
    return float(lsd), float(mel_l1), float(mcd)


@pytest.mark.parametrize("n", [513, 4096, 5000])
@pytest.mark.parametrize("signal", ["noise", "harmonic"])
def test_oracle_matches_torch_stft_restatement(signal, n):
    make = _noise if signal == "noise" else _harmonic_with_silence
    ref = make(n, 1)
    est = make(n, 2) if signal == "noise" else 0.7 * ref + 0.05 * _noise(n, 3) * (ref != 0)
    got = O.distances(ref, est)
    want = _torch_restatement(ref, est)
    for g, w in zip(got, want):
        assert abs(g - w) <= 1e-10 * max(1.0, abs(w)), (got, want)
    if signal == "harmonic" and n > 513:
        # the silent stretches are at both clamps: those frames add 0 to every term
        S = TS.stft_magnitude(torch.from_numpy(ref[None]), 1024, 256, 1024)[0]
        assert bool((S.max(0).values == 0).any())


def test_oracle_identities():
    for x in (_noise(5000, 4), _harmonic_with_silence(6000, 5)):
        assert O.distances(x, x) == (0.0, 0.0, 0.0)
    x = _noise(5000, 6)                                   # noise: no bin, scaled or not, is at a clamp
    lsd, mel_l1, mcd = O.distances(x, 0.5 * x)
    assert abs(lsd - 2 * math.log10(2)) <= 1e-9
    assert abs(mel_l1 - math.log(2)) <= 1e-9
    assert abs(mcd) <= 1e-9


def test_dct_is_orthonormal_dct_ii():
    D = O.dct_matrix(80, 80)
    assert np.abs(D @ D.T - np.eye(80)).max() <= 1e-13
    assert np.abs(dct_matrix(25, 80).numpy() - O.dct_matrix(25, 80)).max() <= 1e-14
    sd = cm.SpectralDistance(n_mel_channels=40, n_cepstra=13)
    assert sd.dct.dtype == torch.float32 and sd.dct.shape == (13, 40)
    assert torch.equal(sd.dct, dct_matrix(13, 40).float())
    assert list(sd.state_dict()) == ["mel_basis"]
    assert torch.equal(sd.mel_basis, cm.TacotronSTFT(n_mel_channels=40).mel_basis)


class _CudaLooking(torch.Tensor):
    @property
    def is_cuda(self):
        return True


@pytest.mark.parametrize("lengths,exc", [([2000, 2001], ValueError), ([512, 2000], ValueError), ([0, 600], ValueError),
                                         ([600.0, 600], TypeError), ([600], ValueError),
                                         (torch.tensor([600, 600]).as_subclass(_CudaLooking), TypeError),
                                         (torch.tensor([600.0, 600.0]), TypeError)])
def test_length_checks_raise_before_the_device(lengths, exc):
    x = torch.zeros(2, 2000)
    with pytest.raises(exc):
        cm.SpectralDistance()(x, x, lengths=lengths)


def test_argument_checks_raise_before_the_device():
    sd = cm.SpectralDistance()
    with pytest.raises(ValueError, match="same shape"):
        sd(torch.zeros(2, 2000), torch.zeros(2, 1999))
    with pytest.raises(ValueError, match="reflect padding"):
        sd(torch.zeros(512), torch.zeros(512))
    with pytest.raises(ValueError):
        sd(torch.zeros(1, 2, 600), torch.zeros(1, 2, 600))
    with pytest.raises(RuntimeError, match="CUDA"):           # valid arguments reach the device check
        sd(torch.zeros(2, 2000), torch.zeros(2, 2000), lengths=[513, 2000])
    for n_cep in (1, 81, 2.0, True):
        with pytest.raises(ValueError, match="n_cepstra"):
            cm.SpectralDistance(n_cepstra=n_cep)
    with pytest.raises(NotImplementedError):
        cm.SpectralDistance(filter_length=1000)
    with pytest.raises(NotImplementedError):
        cm.SpectralDistance(filter_length=8192)
    assert cm.SpectralDistance(n_mel_channels=40, n_cepstra=40).n_cepstra == 40


def _err(lib):
    return lib.cmwg_last_error().decode()


def _sd_c(lib, B=2, T=4000, lengths=None, n_fft=1024, hop=256, n_mels=80, n_cep=25, lengths_dev=None):
    host = None if lengths is None else (C.c_int * len(lengths))(*lengths)
    dev = lengths_dev if lengths_dev is not None else (None if lengths is None else 8)   # never read on an argument error
    return lib.cmwg_spectral_distance(None, None, T, B, T, host, dev, None, None, None, None, None, n_fft, hop, n_mels,
                                      n_cep, None, None, None)


@pytest.mark.parametrize("kw,match", [(dict(lengths=[512, 4000]), "outside"), (dict(lengths=[4000, 4001]), "outside"),
                                      (dict(T=512), "outside"), (dict(lengths=[600, 700], lengths_dev=0), "both"),
                                      (dict(B=-1), "bad sizes"), (dict(hop=0), "bad sizes"), (dict(n_cep=1), "n_cepstra"),
                                      (dict(n_cep=81), "n_cepstra"), (dict(n_mels=0), "n_mels")])
def test_c_argument_errors(kw, match):
    lib = _lib.load()
    assert _sd_c(lib, **kw) == ERR_ARG
    assert match in _err(lib), _err(lib)


@pytest.mark.parametrize("n_fft", [64, 1000, 8192])
def test_c_refuses_unsupported_transform_sizes(n_fft):
    lib = _lib.load()
    assert _sd_c(lib, n_fft=n_fft) == ERR_UNSUPPORTED and "power of two" in _err(lib)


def test_c_valid_arguments_reach_the_pointer_check():
    lib = _lib.load()
    assert _sd_c(lib, lengths=[513, 4000]) == ERR_ARG and "NULL pointer" in _err(lib)
    assert _sd_c(lib, B=0) == 0                          # an empty batch is a no-op


def test_c_abi_symbols_and_workspace_bytes():
    lib = _lib.load()
    for name in ("cmwg_spectral_distance", "cmwg_spectral_distance_workspace_bytes"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    assert lib.cmwg_spectral_distance_workspace_bytes(3, 22050, 1024, 256) == 3 * 3 * (22050 // 256 + 1) * 4
    assert lib.cmwg_spectral_distance_workspace_bytes(0, 22050, 1024, 256) == 0


# ------------------------------------------------------------------------------------------------------------------
# cli compare
# ------------------------------------------------------------------------------------------------------------------
def _error(argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(["compare"] + argv)
    assert e.value.code == 2
    return capsys.readouterr().err


def test_cli_compare_usage_errors(tmp_path, capsys):
    synth = tmp_path / "synth"
    synth.mkdir()
    ref = tmp_path / "a.wav"
    wav_write(str(ref), torch.zeros(1, 4000), 22050)
    err = _error([str(synth), str(ref)], capsys)                       # no synth/a.wav
    assert str(synth / "a.wav") in err and str(ref) in err
    wav_write(str(synth / "a.wav"), torch.zeros(1, 4000), 16000)
    err = _error([str(synth), str(ref)], capsys)                       # rates differ, no --resample
    assert "16000 Hz" in err and "22050" in err and "--resample" in err
    wav_write(str(synth / "a.wav"), torch.zeros(1, 4257), 22050)
    err = _error([str(synth), str(ref)], capsys)                       # 257 samples apart: more than a hop
    assert str(ref) in err and str(synth / "a.wav") in err and "4000" in err and "4257" in err
    wav_write(str(synth / "a.wav"), torch.zeros(1, 4000), 22050)
    err = _error([str(synth), str(ref), "--sampling-rate", "16000"], capsys)
    assert "22050 Hz" in err and "16000" in err
    wav_write(str(ref), torch.zeros(1, 512), 22050)
    wav_write(str(synth / "a.wav"), torch.zeros(1, 512), 22050)
    assert "too few" in _error([str(synth), str(ref)], capsys)
    assert "--max-batch" in _error([str(synth), str(ref), "--max-batch", "0"], capsys)


def test_cli_lists_compare():
    with pytest.raises(SystemExit) as e:
        cli.main([])
    assert "compare" in str(e.value.code)
