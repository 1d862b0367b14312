"""Band-limited resampling on the GPU: ``torchaudio.functional.resample`` per item of a padded batch, with per-item lengths.

``Resample(orig_freq, new_freq, resampling_method="sinc_interp_hann", lowpass_filter_width=6, rolloff=0.99, beta=None)``
takes the constructor of ``torchaudio.transforms.Resample``.  With g = gcd(orig, new), O = orig / g, N = new / g,
base = min(O, N) * rolloff and w = ceil(lpw * O / base), output sample n = k N + j of an item of len samples is

    y[n] = sum_i K[j][i] * x[k O + i - w],   i in [0, 2w + O),   x = 0 outside [0, len)

for n < ceil(N len / O), where K[j][i] is torchaudio's windowed sinc at t = ((i - w) / O - j / N) * base clamped to
[-lpw, lpw] (``_get_sinc_resample_kernel``, computed in float64 as it does for a float64 waveform).  A tap with
|t| >= lpw is zero in exact arithmetic (lpw is an integer, so sin(lpw pi) = 0); torchaudio's values there are rounding
residue below 1e-15.  The table keeps, per phase j, the taps from the first one with |t| < lpw, L of them (the longest
such span over all phases), padded with exact zeros, and is rounded once from float64 to float32.  csrc/resample.cu
evaluates only those L taps per output sample.  torchaudio is not imported.

When orig == new the output is a copy of the input (an identity table through the same kernel).
"""
from __future__ import annotations

import math
import numbers
from typing import List, Optional, Tuple

import torch
from torch import Tensor, nn

from . import ops

__all__ = ["Resample", "resample_table"]

KAISER_BETA = 14.769656459379492          # torchaudio's default beta for sinc_interp_kaiser
METHODS = ("sinc_interp_hann", "sinc_interp_kaiser")


def _check_freq(f, what: str) -> int:
    if isinstance(f, bool) or not isinstance(f, numbers.Real) or not math.isfinite(f):
        raise ValueError(f"Resample: {what} must be a number, got {f!r}")
    if f <= 0:
        # torchaudio.functional.resample's wording
        raise ValueError("Original frequency and desired frequecy should be positive")
    if int(f) != f:
        # torchaudio's wording (_get_sinc_resample_kernel)
        raise ValueError("Frequencies must be of integer type to ensure quality resampling computation. "
                         "To work around this, manually convert both frequencies to integer values "
                         "that maintain their resampling rate ratio before passing them into the function. "
                         "Example: To downsample a 44100 hz waveform by a factor of 8, use "
                         "`orig_freq=8` and `new_freq=1` instead of `orig_freq=44100` and `new_freq=5512.5`. "
                         "For more information, please refer to https://github.com/pytorch/audio/issues/1487.")
    return int(f)


def check_args(orig_freq, new_freq, resampling_method: str, lowpass_filter_width, rolloff: float,
               beta) -> Tuple[int, int, int, float, Optional[float]]:
    """(orig, new, lpw, rolloff, beta) after the checks; beta is None for the Hann window, which ignores it (as
    torchaudio does), and defaults to torchaudio's 14.769656459379492 for the Kaiser window."""
    orig, new = _check_freq(orig_freq, "orig_freq"), _check_freq(new_freq, "new_freq")
    if resampling_method not in METHODS:
        raise ValueError("Invalid resampling method: {}".format(resampling_method))
    if isinstance(lowpass_filter_width, bool) or not isinstance(lowpass_filter_width, numbers.Real) \
            or not math.isfinite(lowpass_filter_width):
        raise ValueError(f"Resample: lowpass_filter_width must be an integer, got {lowpass_filter_width!r}")
    if lowpass_filter_width <= 0:
        raise ValueError("Low pass filter width should be positive.")           # torchaudio's wording
    if int(lowpass_filter_width) != lowpass_filter_width:
        raise ValueError(f"Resample: lowpass_filter_width must be an integer, got {lowpass_filter_width!r}")
    if isinstance(rolloff, bool) or not isinstance(rolloff, numbers.Real) or not 0 < rolloff <= 1:
        raise ValueError(f"Resample: rolloff must be in (0, 1], got {rolloff!r}")
    if resampling_method == "sinc_interp_kaiser":
        beta = KAISER_BETA if beta is None else beta
        if isinstance(beta, bool) or not isinstance(beta, numbers.Real) or not math.isfinite(beta):
            raise ValueError(f"Resample: beta must be a finite number, got {beta!r}")
        beta = float(beta)
    else:
        beta = None
    return orig, new, int(lowpass_filter_width), float(rolloff), beta


def sinc_taps(O: int, N: int, lpw: int, rolloff: float, method: str, beta: Optional[float], i: Tensor) -> Tuple[Tensor, Tensor]:
    """(taps, t before the clamp), float64, of torchaudio's _get_sinc_resample_kernel for reduced rates O, N at tap indices
    i (N, C) int64 of phase j = row, with its operations in its order (elementwise, so any subset of the taps gets the bits
    the full kernel has there), in float64 as for a float64 waveform; beta is a float32 tensor there, so i0(beta) is a
    float32 value."""
    base = min(O, N) * rolloff
    w = math.ceil(lpw * O / base)
    idx = (i - w).to(torch.float64) / O
    t = torch.arange(0, -N, -1, dtype=torch.float64)[:, None] / N + idx
    t *= base
    raw = t.clone()
    t = t.clamp_(-lpw, lpw)
    if method == "sinc_interp_hann":
        window = torch.cos(t * math.pi / lpw / 2) ** 2
    else:
        beta_t = torch.tensor(float(beta))
        window = torch.i0(beta_t * torch.sqrt(1 - (t / lpw) ** 2)) / torch.i0(beta_t)
    t *= math.pi
    scale = base / O
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * scale
    return kernels, raw


def resample_table(orig_freq, new_freq, resampling_method: str = "sinc_interp_hann", lowpass_filter_width=6,
                   rolloff: float = 0.99, beta=None) -> Tuple[Tensor, Tensor, int, int, int]:
    """(table (L, N) float32, first (N,) int32, O, N, w) on the CPU, the operands of cmwg_resample: table[m][j] is tap
    first[j] + m of phase j of torchaudio's kernel (0 past the phase's span of taps with |t| < lpw), built in float64 and
    rounded once.  orig == new gives the identity: table [[1]], first [0], O = N = 1, w = 0.

    Only a window of candidate taps per phase is evaluated, not torchaudio's N x (2w + O) kernel, which for an odd ratio
    (44.1 -> 22.051 kHz: 22051 x 44126) would take gigabytes."""
    orig, new, lpw, rolloff, beta = check_args(orig_freq, new_freq, resampling_method, lowpass_filter_width, rolloff, beta)
    if orig == new:
        return torch.ones((1, 1)), torch.zeros((1,), dtype=torch.int32), 1, 1, 0
    g = math.gcd(orig, new)
    O, N = orig // g, new // g
    base = min(O, N) * rolloff
    w = math.ceil(lpw * O / base)
    K = 2 * w + O
    # |t| < lpw  <=>  i - w in (O j / N - lpw O / base, O j / N + lpw O / base): a span of < 2 lpw O / base + 1 taps
    j = torch.arange(N, dtype=torch.float64)
    lo = torch.floor(w + O * j / N - lpw * O / base).long() - 1
    C = min(math.ceil(2 * lpw * O / base) + 4, K)
    lo = lo.clamp(0, K - C)
    i = lo[:, None] + torch.arange(C)
    kernels, t = sinc_taps(O, N, lpw, rolloff, resampling_method, beta, i)
    kept = t.abs() < lpw
    # the window holds every kept tap (its ends are dropped or are the kernel's ends), and they are one run: t rises with i
    first = kept.to(torch.int8).argmax(1)
    span = kept.sum(1)
    c = torch.arange(C)
    if not (bool((~kept[:, 0] | (lo == 0)).all() and (~kept[:, -1] | (lo + C == K)).all() and (span > 0).all())
            and torch.equal(kept, (c >= first[:, None]) & (c < (first + span)[:, None]))):
        raise RuntimeError(f"Resample: the taps with |t| < lpw of {orig} -> {new} Hz do not form one run per phase "
                           "inside the candidate window")
    m = torch.arange(int(span.max()))
    taps = kernels.gather(1, (first[:, None] + m).clamp(max=C - 1))
    table = torch.where(m < span[:, None], taps, torch.zeros((), dtype=torch.float64)).t()
    return table.float().contiguous(), (lo + first).to(torch.int32).contiguous(), O, N, w


class Resample(nn.Module):
    """``Resample(orig_freq=16000, new_freq=16000, resampling_method="sinc_interp_hann", lowpass_filter_width=6,
    rolloff=0.99, beta=None)``, torchaudio's ``transforms.Resample`` on the GPU, batched with per-item lengths.

    ``forward(x, lengths=None)``: x (B, T) or (T,) CUDA tensor -> (B, ceil(N T / O)) or (ceil(N T / O),) float32.
    ``lengths``: valid samples per item of a zero-padded batch, each in [1, T]; item b then holds
    ``output_lengths(lengths)[b]`` samples equal, bit for bit, to ``self(x[b, :lengths[b]])``, and zeros after them.
    Samples past an item's length are never read (they may be NaN).

    Rejects non-integer or non-positive frequencies, a non-integer or non-positive lowpass_filter_width, rolloff outside
    (0, 1] and an unknown method (torchaudio's deprecated aliases included); beta is ignored with the Hann window.  The
    table is a non-persistent buffer built once in float64 and rounded to float32; it moves with ``.to(device)``.  Its
    values are those of torchaudio's float64 kernel; ``torchaudio.transforms.Resample`` caches a float32 kernel whose
    phase offsets j / N are divided in float32, so its bits differ from this table's by rounding.  No autograd."""

    def __init__(self, orig_freq=16000, new_freq=16000, resampling_method: str = "sinc_interp_hann",
                 lowpass_filter_width=6, rolloff: float = 0.99, beta=None) -> None:
        super().__init__()
        orig, new, lpw, rolloff, beta = check_args(orig_freq, new_freq, resampling_method, lowpass_filter_width,
                                                   rolloff, beta)
        self.orig_freq, self.new_freq = orig, new
        self.resampling_method, self.lowpass_filter_width, self.rolloff, self.beta = resampling_method, lpw, rolloff, beta
        table, first, self.O, self.N, self.width = resample_table(orig, new, resampling_method, lpw, rolloff, beta)
        self.register_buffer("table", table, persistent=False)
        self.register_buffer("first", first, persistent=False)

    def output_lengths(self, lengths) -> List[int]:
        """ceil(N * n / O) for each length n (samples), in exact integer arithmetic."""
        from .base import lengths_list
        lens = lengths_list(lengths, len(lengths), "Resample.output_lengths", "samples")
        for n in lens:
            if n < 0:
                raise ValueError(f"Resample.output_lengths: negative length {n}")
        return [(self.N * n + self.O - 1) // self.O for n in lens]

    @torch.no_grad()
    def forward(self, x: Tensor, lengths=None) -> Tensor:
        return ops.resample(x, self.table, self.first, self.O, self.N, self.width, lengths)

    def extra_repr(self) -> str:
        s = f"orig_freq={self.orig_freq}, new_freq={self.new_freq}, resampling_method={self.resampling_method!r}, " \
            f"lowpass_filter_width={self.lowpass_filter_width}, rolloff={self.rolloff}"
        return s + (f", beta={self.beta}" if self.beta is not None else "")
