"""Denoiser without a device: the fp64 oracle against torch.stft / torch.istft, and the argument checks of Denoiser, of
ops.denoise (which Denoiser.forward calls) and of the C entry points (cmwg_denoise, cmwg_stft_frame_magnitude)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from constant_memory_waveglow_b200 import Denoiser, _lib, ops
from oracle import denoise_oracle as O

ERR_ARG = -1


def _torch_window(n_fft, win_length):
    w = torch.hann_window(win_length, periodic=True, dtype=torch.float64)
    left = (n_fft - win_length) // 2
    return torch.nn.functional.pad(w, (left, n_fft - win_length - left))


@pytest.mark.parametrize("n_fft,win_length,hop,n", [(1024, 1024, 256, 5000), (1024, 1024, 256, 513), (512, 400, 128, 1901),
                                                    (256, 256, 64, 129), (2048, 2048, 512, 22050)])
def test_oracle_matches_torch_stft_istft(n_fft, win_length, hop, n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n)
    w = O.window(n_fft, win_length)
    tw = _torch_window(n_fft, win_length)
    assert np.abs(w - tw.numpy()).max() < 1e-15
    S = O.stft(x, n_fft, hop, w)
    St = torch.stft(torch.from_numpy(x), n_fft, hop, window=tw, center=True, pad_mode="reflect", onesided=True,
                    return_complex=True).numpy()
    assert S.shape == St.shape == (n_fft // 2 + 1, n // hop + 1)
    assert np.abs(S - St).max() <= 1e-12 * np.abs(St).max()
    M = S * rng.uniform(0, 1, S.shape)
    y = O.istft(M, n_fft, hop, w, n)
    yt = torch.istft(torch.from_numpy(M), n_fft, hop, window=tw, center=True, length=n).numpy()
    assert np.abs(y - yt).max() <= 1e-12 * np.abs(yt).max()
    # the denoise definition: magnitude max(|S| - s b, 0), phase of S
    bias = rng.uniform(0, 2, n_fft // 2 + 1)
    d = O.denoise(x, bias, 0.5, n_fft, hop, w)
    mag = np.abs(St)
    gain = np.maximum(mag - 0.5 * bias[:, None], 0) / mag
    dt = torch.istft(torch.from_numpy(St * gain), n_fft, hop, window=tw, center=True, length=n).numpy()
    assert np.abs(d - dt).max() <= 1e-12 * np.abs(dt).max()


@pytest.mark.parametrize("n_fft,hop,n", [(1024, 256, 513), (1024, 256, 220500), (128, 32, 1000)])
def test_oracle_strength_zero_reconstructs(n_fft, hop, n):
    x = np.random.default_rng(1).standard_normal(n)
    y = O.denoise(x, np.ones(n_fft // 2 + 1), 0.0, n_fft, hop, O.window(n_fft, n_fft))
    assert np.linalg.norm(y - x) / np.linalg.norm(x) < 1e-12


@pytest.mark.parametrize("kw,match", [(dict(filter_length=1000), "power of two"), (dict(filter_length=64), "power of two"),
                                      (dict(filter_length=8192), "power of two"), (dict(n_overlap=3), "n_overlap"),
                                      (dict(n_overlap=0), "n_overlap"), (dict(win_length=2048), "win_length"),
                                      (dict(win_length=256), "win_length"), (dict(mode="normal"), "mode")])
def test_denoiser_constructor_rejects(kw, match):
    # the arguments are checked before the model is touched
    with pytest.raises(ValueError, match=match):
        Denoiser(None, **kw)


def _cpu_args(B=2, T=4000):
    return torch.zeros(B, T), torch.ones(1024), torch.ones(513)


@pytest.mark.parametrize("strength", [-0.1, math.nan, math.inf, True, "0.1"])
def test_denoise_rejects_bad_strength(strength):
    x, w, b = _cpu_args()
    with pytest.raises(ValueError, match="strength"):
        ops.denoise(x, w, b, strength, 256)


@pytest.mark.parametrize("lengths,exc,match", [([512, 4000], ValueError, "outside"), ([4001, 4000], ValueError, "outside"),
                                               ([0, 4000], ValueError, "outside"), ([4000], ValueError, "2 lengths|1 lengths"),
                                               ([4000, 4000, 4000], ValueError, "lengths for a batch"),
                                               ([600.0, 4000], TypeError, "integers"),
                                               (torch.tensor([600.0, 4000.0]), TypeError, "integer")])
def test_denoise_rejects_bad_lengths(lengths, exc, match):
    x, w, b = _cpu_args()
    with pytest.raises(exc, match=match):
        ops.denoise(x, w, b, 0.1, 256, lengths=lengths)


def test_denoise_rejects_short_audio_and_cpu_tensors():
    _, w, b = _cpu_args()
    with pytest.raises(ValueError, match="outside"):
        ops.denoise(torch.zeros(512), w, b, 0.1, 256)
    with pytest.raises(ValueError, match=r"\(T,\) or \(B, T\)"):
        ops.denoise(torch.zeros(1, 1, 600), w, b, 0.1, 256)
    # valid arguments: no CPU implementation
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.denoise(torch.zeros(2, 4000), w, b, 0.1, 256, lengths=[513, 4000])


def _err(lib):
    return lib.cmwg_last_error().decode()


def _denoise_c(lib, B=2, T=4000, lengths=None, strength=0.1, n_fft=1024, hop=256, lengths_dev=None):
    host = None if lengths is None else (C.c_int * len(lengths))(*lengths)
    dev = lengths_dev if lengths_dev is not None else (None if lengths is None else 8)   # never read on an argument error
    return lib.cmwg_denoise(None, T, B, T, host, dev, None, None, strength, n_fft, hop, None, None, None)


@pytest.mark.parametrize("kw,match", [(dict(n_fft=1000), "power of two"), (dict(n_fft=8192), "power of two"),
                                      (dict(hop=0), "hop"), (dict(hop=513), "hop"), (dict(strength=-1.0), "strength"),
                                      (dict(strength=math.nan), "strength"), (dict(strength=math.inf), "strength"),
                                      (dict(lengths=[512, 4000]), "outside"), (dict(lengths=[4000, 4001]), "outside"),
                                      (dict(T=512), "outside"), (dict(lengths=[600, 700], lengths_dev=0), "both"),
                                      (dict(B=-1), "bad sizes")])
def test_c_denoise_argument_errors(kw, match):
    lib = _lib.load()
    assert _denoise_c(lib, **kw) == ERR_ARG
    assert match in _err(lib) or any(m in _err(lib) for m in match.split("|")), _err(lib)


def test_c_denoise_valid_arguments_reach_the_pointer_check():
    lib = _lib.load()
    assert _denoise_c(lib, lengths=[513, 4000]) == ERR_ARG and "NULL pointer" in _err(lib)
    assert _denoise_c(lib, B=0) == 0                     # an empty batch is a no-op


@pytest.mark.parametrize("T,n_fft,hop,frame,match", [(4000, 1000, 256, 0, "power of two"), (4000, 1024, 0, 0, "hop"),
                                                     (512, 1024, 256, 0, "reflect"), (4000, 1024, 256, -1, "frame"),
                                                     (4000, 1024, 256, 16, "frame")])
def test_c_stft_frame_magnitude_argument_errors(T, n_fft, hop, frame, match):
    lib = _lib.load()
    assert lib.cmwg_stft_frame_magnitude(None, T, None, n_fft, hop, frame, None, None) == ERR_ARG
    assert match in _err(lib), _err(lib)


def test_c_denoise_workspace_bytes():
    lib = _lib.load()
    assert lib.cmwg_denoise_workspace_bytes(3, 22050, 1024, 256) == 3 * (22050 // 256 + 1) * 1024 * 4
    assert lib.cmwg_denoise_workspace_bytes(0, 22050, 1024, 256) == 0
