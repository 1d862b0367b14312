"""Spectral distances between audio pairs on the GPU, batched with per-item lengths: log-spectral distance (LSD), log-mel L1
and mel-cepstral distortion (MCD) on Tacotron2's STFT and mel, in one fused pass (``cmwg_spectral_distance``,
csrc/distance.cu).  ``oracle/distance_oracle.py`` restates the definitions in float64.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import torch
from torch import Tensor

from . import _lib as L
from . import ops
from .condition import TacotronSTFT, mel_lengths

__all__ = ["SpectralDistance", "Distances", "dct_matrix"]


class Distances(NamedTuple):
    lsd: Tensor
    mel_l1: Tensor
    mcd: Tensor


def dct_matrix(n_cepstra: int, n_mels: int) -> Tensor:
    """(n_cepstra, n_mels) float64, the first n_cepstra rows of the orthonormal DCT-II:
    D[d, j] = sqrt((1 if d == 0 else 2) / n_mels) cos(pi d (2 j + 1) / (2 n_mels))."""
    d = torch.arange(n_cepstra, dtype=torch.float64)[:, None]
    j = torch.arange(n_mels, dtype=torch.float64)[None, :]
    D = torch.cos(math.pi * d * (2 * j + 1) / (2 * n_mels)) * math.sqrt(2.0 / n_mels)
    D[0] = math.sqrt(1.0 / n_mels)
    return D


class SpectralDistance(TacotronSTFT):
    """``SpectralDistance(sampling_rate=22050, filter_length=1024, hop_length=256, win_length=1024, n_mel_channels=80,
    mel_fmin=0.0, mel_fmax=8000.0, n_cepstra=25)``: frame-level spectral distances between a reference and an estimate.

    ``forward(ref, est, lengths=None)``: ref, est (B, T) or (T,) CUDA tensors of the same shape -> ``Distances(lsd, mel_l1,
    mcd)``, (B,) float32 tensors (0-d for 1-D input).  Item b is compared over the first ``lengths[b]`` samples (T when
    ``lengths`` is None) of both signals, with n_fft/2 < len_b <= T; samples past it are never read.  With S, S^ the STFTs
    of ``TacotronSTFT`` (reflect padding by filter_length/2 at the item's end, periodic Hann window, len_b // hop + 1
    frames, filter_length/2 + 1 bins), each metric is the mean over frames of a per-frame term:

    - ``lsd``: sqrt(mean_k (log10 max(|S|^2, 1e-10) - log10 max(|S^|^2, 1e-10))^2), the 1e-10 being Tacotron2's 1e-5
      amplitude clamp squared;
    - ``mel_l1``: mean_j |m_j - m^_j| with m = ln max(mel_basis @ |S|, 1e-5), i.e. ``TacotronSTFT.mel_spectrogram``;
    - ``mcd``: (10 / ln 10) sqrt(2 sum_{d=1}^{n_cepstra-1} (c_d - c^_d)^2), c = D m with D the orthonormal DCT-II
      (``dct_matrix``); c0, the energy, is excluded.

    The MCD here is computed on mel-frequency cepstra of the Tacotron2 mel: no SPTK all-pass warped mel-cepstrum and no
    DTW, so its values are not comparable with papers that report SPTK ``mcep`` with DTW alignment.  The signals are not
    aligned in time either: the caller supplies aligned pairs.

    Batched items equal their solo calls bit for bit; the sums run in a fixed order (deterministic), identical inputs give
    exactly 0 and swapping ``ref`` and ``est`` gives identical results.  ``mel_basis`` is ``TacotronSTFT``'s buffer
    (load librosa's table with ``load_state_dict``); ``dct`` is a non-persistent buffer.  No autograd."""

    def __init__(self, sampling_rate: int = 22050, filter_length: int = 1024, hop_length: int = 256,
                 win_length: int = 1024, n_mel_channels: int = 80, mel_fmin: float = 0.0, mel_fmax=8000.0,
                 n_cepstra: int = 25) -> None:
        if isinstance(n_cepstra, bool) or not isinstance(n_cepstra, int) or not 2 <= n_cepstra <= n_mel_channels:
            raise ValueError(f"SpectralDistance: n_cepstra {n_cepstra!r} outside [2, n_mel_channels = {n_mel_channels}]")
        super().__init__(filter_length=filter_length, hop_length=hop_length, win_length=win_length,
                         n_mel_channels=n_mel_channels, sampling_rate=sampling_rate, mel_fmin=mel_fmin,
                         mel_fmax=mel_fmax)
        self.n_cepstra = int(n_cepstra)
        self.register_buffer("dct", dct_matrix(self.n_cepstra, self.n_mel_channels).float(), persistent=False)

    @torch.no_grad()
    def forward(self, ref: Tensor, est: Tensor, lengths=None) -> Distances:
        if ref.shape != est.shape:
            raise ValueError(f"SpectralDistance: ref and est must have the same shape, got {tuple(ref.shape)} and "
                             f"{tuple(est.shape)}")
        n_fft = self.filter_length
        lens = mel_lengths(ref, lengths, n_fft, n_fft // 2, "SpectralDistance")
        L.require_cuda(ref, est, op="SpectralDistance")
        if ref.device != est.device:
            raise ValueError(f"SpectralDistance: ref on {ref.device} and est on {est.device}")
        (x, squeeze), (y, _) = ops.audio_batch(ref), ops.audio_batch(est)
        x, y = x.contiguous(), y.contiguous()   # the kernel takes one batch stride, T, for both
        B, T = x.shape
        window, fbt, lo, hi = self._device_tables(x.device)
        dct = self.dct.to(x.device)
        lib = L.load()
        workspace = torch.empty((max(int(lib.cmwg_spectral_distance_workspace_bytes(B, T, n_fft, self.hop_length)), 4),),
                                device=x.device, dtype=torch.uint8)
        out = torch.empty((B, 3), device=x.device, dtype=torch.float32)
        lens_host, lens_dev = ops.lengths_arg(lens, x.device)
        L.check(lib.cmwg_spectral_distance(x.data_ptr(), y.data_ptr(), T, B, T, lens_host, L.ptr(lens_dev),
                                           window.data_ptr(), fbt.data_ptr(), lo.data_ptr(), hi.data_ptr(),
                                           dct.data_ptr(), n_fft, self.hop_length, self.n_mel_channels,
                                           self.n_cepstra, workspace.data_ptr(), out.data_ptr(),
                                           L.stream_ptr(x.device)), "spectral_distance")
        if squeeze:
            out = out[0]
        return Distances(*out.unbind(-1))

    def extra_repr(self) -> str:
        return (f"sampling_rate={self.sampling_rate}, filter_length={self.filter_length}, hop_length={self.hop_length}, "
                f"win_length={self.win_length}, n_mel_channels={self.n_mel_channels}, mel_fmin={self.mel_fmin}, "
                f"mel_fmax={self.mel_fmax}, n_cepstra={self.n_cepstra}")
