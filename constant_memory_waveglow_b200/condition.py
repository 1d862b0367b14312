"""Conditioners: the step right before the flow in training and inference (reference ``model/condition.py``).

``MelSpec(sr, n_fft, hop_length, **kwargs)`` mirrors ``model/condition.py:7-19`` -- reflection padding by
``(n_fft/2 - hop/2, n_fft/2 + hop/2)``, torchaudio's ``MelSpectrogram(center=False)`` (periodic Hann window, power 2,
HTK mel scale, no normalisation unless asked for) and ``log(mel + 1e-7)`` -- as ONE fused CUDA kernel
(``cmwg_melspec_fwd``, csrc/melspec.cu): the padded signal, the complex STFT and the power spectrogram never reach
HBM.  torchaudio is not imported; the filterbank is rebuilt from its published definition
(``torchaudio.functional.melscale_fbanks``) and the buffers keep the reference's state-dict keys
(``mel.1.spectrogram.window``, ``mel.1.mel_scale.fb``, persistent buffers as in torchaudio, so a Lightning
checkpoint's ``conditioner.mel.1.*`` entries load here and vice versa).  ``MelSpec.forward(x, lengths=...)`` runs a
zero-padded batch of different-length items in one call (``cmwg_melspec_fwd_varlen``); each item gets its own call's bits.

``TacotronSTFT`` is the mel front end of Tacotron2 (``layers.TacotronSTFT.mel_spectrogram``), the input NVIDIA's WaveGlow
is trained on: reflect padding by ``n_fft/2``, ``|STFT|`` with a periodic Hann window, a Slaney-scale, Slaney-normalised
filterbank (librosa's ``filters.mel``) and ``log(clamp(x, min=1e-5))``, through the same kernel.
"""
from __future__ import annotations

import math
from typing import List, Optional

import numpy as np
import torch
from torch import Tensor, nn

from . import _lib as L
from . import ops
from .base import audio_lengths

__all__ = ["MelSpec", "TacotronSTFT", "mel_filterbank", "slaney_mel_basis"]


def _hz_to_mel(f: float, scale: str) -> float:
    if scale == "htk":
        return 2595.0 * math.log10(1.0 + f / 700.0)
    # slaney: linear below 1 kHz, logarithmic above
    f_sp = 200.0 / 3
    if f >= 1000.0:
        return 1000.0 / f_sp + math.log(f / 1000.0) / (math.log(6.4) / 27.0)
    return f / f_sp


def _mel_to_hz(m: Tensor, scale: str) -> Tensor:
    if scale == "htk":
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
    f_sp = 200.0 / 3
    hz = f_sp * m
    min_log_mel = 1000.0 / f_sp
    logstep = math.log(6.4) / 27.0
    above = m >= min_log_mel
    hz[above] = 1000.0 * torch.exp(logstep * (m[above] - min_log_mel))
    return hz


def mel_filterbank(n_freqs: int, f_min: float, f_max: float, n_mels: int, sample_rate: int, norm=None,
                   mel_scale: str = "htk") -> Tensor:
    """(n_freqs, n_mels) triangular filters, fp32 -- the definition of torchaudio.functional.melscale_fbanks:
    bin centres linspace(0, sr // 2, n_freqs); n_mels + 2 band edges equally spaced on the mel axis between
    f_min and f_max; band m rises from edge m to edge m+1 and falls to edge m+2."""
    if norm not in (None, "slaney"):
        raise ValueError('norm must be one of None or "slaney"')
    if mel_scale not in ("htk", "slaney"):
        raise ValueError('mel_scale should be one of "htk" or "slaney".')
    bins = torch.linspace(0, sample_rate // 2, n_freqs)
    edges_mel = torch.linspace(_hz_to_mel(f_min, mel_scale), _hz_to_mel(f_max, mel_scale), n_mels + 2)
    edges = _mel_to_hz(edges_mel, mel_scale)
    width = edges[1:] - edges[:-1]                              # (n_mels + 1)
    dist = edges.unsqueeze(0) - bins.unsqueeze(1)               # (n_freqs, n_mels + 2)
    falling = -dist[:, :-2] / width[:-1]
    rising = dist[:, 2:] / width[1:]
    fb = torch.clamp(torch.minimum(falling, rising), min=0.0)
    if norm == "slaney":
        fb = fb * (2.0 / (edges[2:n_mels + 2] - edges[:n_mels])).unsqueeze(0)
    return fb


def _kernel_tables(window: Tensor, fb: Tensor, n_fft: int, device):
    """(full-length window, fb (n_freqs, n_mels) transposed to (n_mels, n_freqs), lo, hi) on `device`, the tables of the
    mel kernels: band m is non-zero only on bins [lo[m], hi[m])."""
    w = window.detach().to(device=device, dtype=torch.float32)
    if w.numel() < n_fft:                                   # torch.stft centres a short window in the frame
        left = (n_fft - w.numel()) // 2
        w = torch.nn.functional.pad(w, (left, n_fft - w.numel() - left))
    f = fb.detach().to(device=device, dtype=torch.float32).contiguous()
    nz = f != 0
    any_nz = nz.any(0)
    lo = torch.where(any_nz, nz.float().argmax(0), torch.zeros_like(any_nz, dtype=torch.long))
    hi = torch.where(any_nz, f.shape[0] - nz.flip(0).float().argmax(0), torch.zeros_like(any_nz, dtype=torch.long))
    return w.contiguous(), f.t().contiguous(), lo.int().contiguous(), hi.int().contiguous()


def mel_lengths(x: Tensor, lengths, n_fft: int, pad_left: int, what: str) -> Optional[List[int]]:
    """audio_lengths for a mel transform that reflect-pads by pad_left and n_fft - pad_left: each length (T when `lengths`
    is None) must exceed the larger pad."""
    return audio_lengths(x, lengths, max(pad_left, n_fft - pad_left), what)


def _melspec_varlen(x: Tensor, lens: Optional[List[int]], tables, n_fft: int, hop: int, n_mels: int, pad_left: int,
                    power_is_one: int, log_mode: int, eps: float) -> Tensor:
    """cmwg_melspec_fwd_varlen of x (B, T) or (T,) on the GPU -> (B, n_mels, T // hop + 1) (or (n_mels, frames))."""
    x, squeeze = ops.audio_batch(x)
    B, T = x.shape
    window, fbt, lo, hi = tables
    out = torch.empty((B, n_mels, T // hop + 1), device=x.device, dtype=torch.float32)
    lens_host, lens_dev = ops.lengths_arg(lens, x.device)
    L.check(L.load().cmwg_melspec_fwd_varlen(x.data_ptr(), x.stride(0) if B > 1 else T, B, T, lens_host, L.ptr(lens_dev),
                                             window.data_ptr(), fbt.data_ptr(), lo.data_ptr(), hi.data_ptr(), n_fft, hop,
                                             n_mels, pad_left, power_is_one, log_mode, eps, out.data_ptr(),
                                             L.stream_ptr(x.device)), "melspec_fwd_varlen")
    return out[0] if squeeze else out


def _slaney_hz_to_mel(f: np.ndarray) -> np.ndarray:
    f_sp = 200.0 / 3
    mels = f / f_sp
    min_log_hz, min_log_mel, logstep = 1000.0, 1000.0 / f_sp, np.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, min_log_hz) / min_log_hz) / logstep, mels)


def _slaney_mel_to_hz(m: np.ndarray) -> np.ndarray:
    f_sp = 200.0 / 3
    freqs = f_sp * m
    min_log_hz, min_log_mel, logstep = 1000.0, 1000.0 / f_sp, np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), freqs)


def slaney_mel_basis(sr: float, n_fft: int, n_mels: int, fmin: float = 0.0, fmax: Optional[float] = None) -> Tensor:
    """(n_mels, n_fft // 2 + 1) float64 -- librosa's ``filters.mel(sr=sr, n_fft=n_fft, n_mels=n_mels, fmin=fmin,
    fmax=fmax)`` (Slaney mel scale, Slaney area normalisation), computed in float64 throughout; librosa itself rounds the
    triangles to float32 before the normalisation, so its float32 table can differ from this one rounded once in the last
    bit.  Bin centres are ``rfftfreq(n_fft, 1 / sr)``; band m rises from edge m to edge m+1 and falls to edge m+2 of
    n_mels + 2 edges equally spaced on the mel axis, and is scaled by 2 / (edge m+2 - edge m) in Hz."""
    fmax = float(sr) / 2 if fmax is None else float(fmax)
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    mel_f = _slaney_mel_to_hz(np.linspace(_slaney_hz_to_mel(np.float64(fmin)), _slaney_hz_to_mel(np.float64(fmax)),
                                          n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    lower = -ramps[:n_mels] / fdiff[:n_mels, None]
    upper = ramps[2:n_mels + 2] / fdiff[1:n_mels + 1, None]
    weights = np.maximum(0.0, np.minimum(lower, upper))
    weights = weights * (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]
    return torch.from_numpy(weights)


class _Buffers(nn.Module):
    """Holds one buffer under the attribute name torchaudio uses."""

    def __init__(self, name: str, value: Tensor):
        super().__init__()
        self.register_buffer(name, value)


class _MelSpectrogramState(nn.Module):
    """Parameter container laid out like torchaudio.transforms.MelSpectrogram (``spectrogram.window``,
    ``mel_scale.fb``) so module paths and state-dict keys match the reference's ``MelSpec.mel[1]``."""

    def __init__(self, window: Tensor, fb: Tensor):
        super().__init__()
        self.spectrogram = _Buffers("window", window)
        self.mel_scale = _Buffers("fb", fb)


class _ReflectionPadSpec(nn.Module):
    """Records the padding of ``nn.ReflectionPad1d`` (slot 0 of the reference's Sequential); the padding itself is
    index arithmetic inside the kernel."""

    def __init__(self, padding):
        super().__init__()
        self.padding = tuple(padding)

    def extra_repr(self) -> str:
        return f"{self.padding}"


class MelSpec(nn.Module):
    """Log-mel conditioner, x (B, T) or (T,) -> (B, n_mels, T // hop + 1)  (reference ``model/condition.py:7-19``).

    Keyword arguments are those of ``torchaudio.transforms.MelSpectrogram`` that the reference's configs use or
    that have a direct meaning here: ``f_min``, ``f_max``, ``n_mels``, ``win_length`` (<= n_fft, centred zero
    padding), ``power`` (1 or 2), ``norm``, ``mel_scale``, ``window_fn``.
    """

    def __init__(self, sr, n_fft, hop_length, f_min: float = 0.0, f_max=None, n_mels: int = 128, win_length=None,
                 power: float = 2.0, normalized: bool = False, norm=None, mel_scale: str = "htk",
                 window_fn=torch.hann_window, wkwargs=None, **unsupported) -> None:
        super().__init__()
        if unsupported:
            raise TypeError(f"MelSpec: unsupported MelSpectrogram arguments {sorted(unsupported)}")
        if normalized:
            raise NotImplementedError("MelSpec: normalized=True is not built")
        if power not in (1, 1.0, 2, 2.0):
            raise NotImplementedError("MelSpec: power must be 1 or 2")
        if n_fft & (n_fft - 1) or not 128 <= n_fft <= 4096:
            raise NotImplementedError("MelSpec: n_fft must be a power of two in [128, 4096]")
        self.sample_rate, self.n_fft, self.hop_length = int(sr), int(n_fft), int(hop_length)
        self.power = float(power)
        self.n_mels = int(n_mels)
        win_length = int(win_length) if win_length is not None else self.n_fft
        window = window_fn(win_length, **(wkwargs or {})).float()
        f_max = float(f_max) if f_max is not None else float(self.sample_rate // 2)
        fb = mel_filterbank(self.n_fft // 2 + 1, float(f_min), f_max, self.n_mels, self.sample_rate, norm, mel_scale)
        self.mel = nn.Sequential(
            _ReflectionPadSpec((self.n_fft // 2 - self.hop_length // 2, self.n_fft // 2 + self.hop_length // 2)),
            _MelSpectrogramState(window, fb))
        self._cache = None

    def _device_tables(self, device):
        """(full-length window, fb transposed to (n_mels, n_freqs), lo, hi) on `device`; rebuilt when the buffers change identity or version."""
        st = self.mel[1]
        window, fb = st.spectrogram.window, st.mel_scale.fb
        key = (window.data_ptr(), window._version, fb.data_ptr(), fb._version, str(device))
        if self._cache is not None and self._cache[0] == key:
            return self._cache[1]
        tables = _kernel_tables(window, fb, self.n_fft, device)
        self._cache = (key, tables)
        return tables

    def forward(self, x: Tensor, lengths=None) -> Tensor:
        """``lengths``: valid samples per item of a zero-padded batch x (B, T).  Item b then gets ``len_b // hop + 1`` frames
        equal, bit for bit, to ``self(x[b, :len_b])``, and zeros after them."""
        pad_left = self.n_fft // 2 - self.hop_length // 2
        if lengths is not None:
            lens = mel_lengths(x, lengths, self.n_fft, pad_left, "MelSpec")
            L.require_cuda(x, op="MelSpec")
            return _melspec_varlen(x, lens, self._device_tables(x.device), self.n_fft, self.hop_length, self.n_mels,
                                   pad_left, int(self.power == 1.0), 1, 1e-7)
        L.require_cuda(x, op="MelSpec")
        if x.dim() not in (1, 2):
            raise ValueError(f"MelSpec: expected audio (T,) or (B, T), got {tuple(x.shape)}")
        x, squeeze = ops.audio_batch(x)
        B, T = x.shape
        lib = L.load()
        frames = lib.cmwg_melspec_frames(T, self.n_fft, self.hop_length)
        window, fbt, lo, hi = self._device_tables(x.device)
        out = torch.empty((B, self.n_mels, frames), device=x.device, dtype=torch.float32)
        L.check(lib.cmwg_melspec_fwd(x.data_ptr(), x.stride(0) if B > 1 else T, B, T, window.data_ptr(), fbt.data_ptr(),
                                     lo.data_ptr(), hi.data_ptr(), self.n_fft, self.hop_length, self.n_mels,
                                     int(self.power == 1.0), 1e-7, 1, out.data_ptr(), L.stream_ptr(x.device)),
                "melspec_fwd")
        return out[0] if squeeze else out


class TacotronSTFT(nn.Module):
    """Tacotron2's mel front end (NVIDIA/tacotron2 ``layers.TacotronSTFT``), the conditioning NVIDIA's WaveGlow is trained
    on, with NVIDIA's constructor arguments.  ``mel_spectrogram(y, lengths=None)``: y (B, T) or (T,) on the GPU ->
    (B, n_mel_channels, T // hop_length + 1) (or (n_mel_channels, frames)) =
    ``log(clamp(mel_basis @ |STFT(y)|, min=1e-5))`` with the STFT of ``stft.STFT``: reflect padding by filter_length/2,
    frames every hop_length samples, a periodic Hann window of win_length samples centred in the frame by zero padding.

    ``lengths``: valid samples per item of a zero-padded batch y.  Item b then gets ``len_b // hop_length + 1`` frames equal,
    bit for bit, to ``mel_spectrogram(y[b, :len_b])``, followed by zeros.  Each length must exceed filter_length/2.

    Unlike NVIDIA's, ``mel_spectrogram`` does not assert that y lies in [-1, 1]; the transform is defined for any input,
    and a model trained on such mels expects audio in that range.  ``mel_basis`` (n_mel_channels, filter_length/2 + 1) is
    a buffer, librosa's ``filters.mel`` computed in float64 and rounded once to float32 (``slaney_mel_basis``); load
    librosa's own table with ``load_state_dict({"mel_basis": ...})`` for its exact bits."""

    def __init__(self, filter_length: int = 1024, hop_length: int = 256, win_length: int = 1024,
                 n_mel_channels: int = 80, sampling_rate: int = 22050, mel_fmin: float = 0.0, mel_fmax=8000.0) -> None:
        super().__init__()
        if filter_length & (filter_length - 1) or not 128 <= filter_length <= 4096:
            raise NotImplementedError("TacotronSTFT: filter_length must be a power of two in [128, 4096]")
        if not 1 <= win_length <= filter_length:
            raise ValueError(f"TacotronSTFT: win_length {win_length} outside [1, filter_length = {filter_length}]")
        if hop_length < 1 or n_mel_channels < 1:
            raise ValueError("TacotronSTFT: hop_length and n_mel_channels must be >= 1")
        self.filter_length, self.hop_length, self.win_length = int(filter_length), int(hop_length), int(win_length)
        self.n_mel_channels, self.sampling_rate = int(n_mel_channels), int(sampling_rate)
        self.mel_fmin, self.mel_fmax = float(mel_fmin), None if mel_fmax is None else float(mel_fmax)
        basis = slaney_mel_basis(self.sampling_rate, self.filter_length, self.n_mel_channels, self.mel_fmin, self.mel_fmax)
        self.register_buffer("mel_basis", basis.float())
        # scipy.signal.get_window("hann", win_length, fftbins=True): the periodic Hann window
        self.register_buffer("window", torch.hann_window(self.win_length, periodic=True, dtype=torch.float64).float(),
                             persistent=False)
        self._cache = None

    @property
    def n_mels(self) -> int:
        return self.n_mel_channels

    def _device_tables(self, device):
        """The kernel tables on `device`; rebuilt when a buffer changes identity or version (load_state_dict, to())."""
        key = (self.window.data_ptr(), self.window._version, self.mel_basis.data_ptr(), self.mel_basis._version, str(device))
        if self._cache is not None and self._cache[0] == key:
            return self._cache[1]
        tables = _kernel_tables(self.window, self.mel_basis.t(), self.filter_length, device)
        self._cache = (key, tables)
        return tables

    def mel_spectrogram(self, y: Tensor, lengths=None) -> Tensor:
        n_fft = self.filter_length
        lens = mel_lengths(y, lengths, n_fft, n_fft // 2, "TacotronSTFT")
        L.require_cuda(y, op="TacotronSTFT")
        return _melspec_varlen(y, lens, self._device_tables(y.device), n_fft, self.hop_length, self.n_mel_channels,
                               n_fft // 2, 1, 2, 1e-5)

    def forward(self, y: Tensor, lengths=None) -> Tensor:
        return self.mel_spectrogram(y, lengths)
