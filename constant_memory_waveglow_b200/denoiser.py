"""Denoiser of synthesised audio: removes the constant hiss ("bias") a flow vocoder leaves in its output by subtracting the
bias's magnitude spectrum, the ``Denoiser`` of NVIDIA's WaveGlow (its ``denoiser.py``, mode ``'zeros'``; the
``--denoiser_strength`` of its ``inference.py``) with the same constructor and call.

The bias is the model's output for an all-zero mel spectrogram (88 frames, sigma 0); its spectrum is the magnitude of the
first STFT frame.  ``denoiser(audio, strength)`` then computes, per item, S = STFT(audio), keeps the phase of S and sets the
magnitude to max(|S| - strength * bias, 0), and inverts the STFT (csrc/denoise.cu; the complex spectrogram never reaches
HBM).  A padded batch with per-item ``lengths`` (samples) gives each item exactly what a call on that item alone gives, and
zeros after its length.
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from . import ops

__all__ = ["Denoiser"]


class Denoiser(nn.Module):
    """``Denoiser(model, filter_length=1024, n_overlap=4, win_length=1024, mode="zeros")``; ``denoiser(audio, strength=0.1,
    lengths=None)``.

    ``model``: a flow model with ``infer`` and ``n_mels`` (WaveGlow, WaveFlow, ...), already on its CUDA device.  The STFT has
    ``n_fft = filter_length`` (a power of two in [128, 4096]), ``hop = filter_length / n_overlap`` and a periodic Hann window
    of ``win_length <= filter_length`` samples (``2 * hop <= win_length``), centred in the frame.  ``audio``: (T,) or (B, T)
    CUDA tensor; ``lengths``: per-item valid samples of a padded batch, each in (filter_length / 2, T].  No autograd.
    """

    def __init__(self, model: nn.Module, filter_length: int = 1024, n_overlap: int = 4, win_length: int = 1024,
                 mode: str = "zeros") -> None:
        super().__init__()
        n_fft, n_overlap, win_length = int(filter_length), int(n_overlap), int(win_length)
        if n_fft & (n_fft - 1) or not 128 <= n_fft <= 4096:
            raise ValueError(f"Denoiser: filter_length must be a power of two in [128, 4096], got {filter_length}")
        if n_overlap < 2 or n_fft % n_overlap:
            raise ValueError(f"Denoiser: n_overlap must divide filter_length and be >= 2, got {n_overlap}")
        hop = n_fft // n_overlap
        if not 2 * hop <= win_length <= n_fft:
            raise ValueError(f"Denoiser: win_length must be in [2 * hop, filter_length] = [{2 * hop}, {n_fft}], got "
                             f"{win_length}")
        if mode != "zeros":
            raise ValueError(f"Denoiser: mode {mode!r} is not supported (only 'zeros')")
        self.filter_length, self.n_overlap, self.win_length, self.hop_length = n_fft, n_overlap, win_length, hop
        device = next(model.parameters()).device
        window = torch.hann_window(win_length, periodic=True, dtype=torch.float32)
        left = (n_fft - win_length) // 2                        # torch.stft centres a short window in the frame
        window = nn.functional.pad(window, (left, n_fft - win_length - left)).to(device)
        with torch.no_grad():
            mel = torch.zeros((1, model.n_mels, 88), device=device)
            bias_audio = model.infer(mel, sigma=0.0)
            bias_spec = ops.stft_frame_magnitude(bias_audio, window, hop, 0)
        self.register_buffer("window", window)
        self.register_buffer("bias_spec", bias_spec)

    @torch.no_grad()
    def forward(self, audio: Tensor, strength: float = 0.1, lengths=None) -> Tensor:
        return ops.denoise(audio, self.window, self.bias_spec, strength, self.hop_length, lengths)

    def extra_repr(self) -> str:
        return f"filter_length={self.filter_length}, n_overlap={self.n_overlap}, win_length={self.win_length}"
