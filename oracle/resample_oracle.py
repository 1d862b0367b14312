"""fp64 numpy reference of band-limited resampling (constant_memory_waveglow_b200.Resample, csrc/resample.cu), test-only.

torchaudio.functional.resample(x, orig, new, lpw, rolloff, method, beta) restated: with g = gcd(orig, new), O = orig / g,
N = new / g, base = min(O, N) * rolloff and w = ceil(lpw * O / base),

    y[k N + j] = sum_{i < 2w + O} K[j][i] * x[k O + i - w]      (x = 0 outside [0, len)),   n < ceil(N len / O)

K[j][i] = sinc(pi t) * window(t) * base / O at t = clamp(((i - w) / O - j / N) * base, -lpw, lpw), the window
cos(pi t / (2 lpw))^2 (sinc_interp_hann) or i0(beta sqrt(1 - (t / lpw)^2)) / i0(beta) (sinc_interp_kaiser).  torchaudio
holds beta in a float32 tensor, so beta and i0(beta) are float32 values there; so they are here.

The compact form keeps, per phase j, only the taps with |t| < lpw (the others are zero in exact arithmetic): `first[j]`,
the index of the first, and L = the longest such span; table (L, N) with zeros past each phase's span.
"""
import math

import numpy as np
import torch


def reduced(orig: int, new: int):
    g = math.gcd(orig, new)
    return orig // g, new // g


def output_length(n: int, orig: int, new: int) -> int:
    O, N = reduced(orig, new)
    return -(-N * n // O)


def kernel(orig: int, new: int, lpw: int = 6, rolloff: float = 0.99, method: str = "sinc_interp_hann", beta=None,
           phases=None):
    """(K (N, 2w + O), t (N, 2w + O) before the clamp, w), float64; only the rows `phases` (all when None)."""
    O, N = reduced(orig, new)
    base = min(O, N) * rolloff
    w = math.ceil(lpw * O / base)
    i = np.arange(-w, w + O, dtype=np.float64)
    j = np.arange(N, dtype=np.float64) if phases is None else np.asarray(phases, dtype=np.float64)
    t = (-j[:, None] / N + i[None, :] / O) * base
    tc = np.clip(t, -lpw, lpw)
    if method == "sinc_interp_hann":
        win = np.cos(tc * math.pi / lpw / 2) ** 2
    elif method == "sinc_interp_kaiser":
        b32 = torch.tensor(float(14.769656459379492 if beta is None else beta))          # float32, as torchaudio holds it
        win = np.i0(float(b32) * np.sqrt(1 - (tc / lpw) ** 2)) / float(torch.i0(b32))
    else:
        raise ValueError(method)
    x = tc * math.pi
    with np.errstate(invalid="ignore", divide="ignore"):
        s = np.where(x == 0, 1.0, np.sin(x) / x)
    return s * (win * (base / O)), t, w


def compact_table(orig: int, new: int, lpw: int = 6, rolloff: float = 0.99, method: str = "sinc_interp_hann", beta=None):
    """(table (L, N) float64, first (N,) int64, w): the taps with |t| < lpw of each phase, from its first one on."""
    K, t, w = kernel(orig, new, lpw, rolloff, method, beta)
    N = K.shape[0]
    first = np.zeros(N, dtype=np.int64)
    spans = []
    for j in range(N):
        keep = np.nonzero(np.abs(t[j]) < lpw)[0]
        first[j] = keep[0]
        spans.append(keep)
    L = max(len(s) for s in spans)
    table = np.zeros((L, N))
    for j, keep in enumerate(spans):
        table[:len(keep), j] = K[j, keep]
    return table, first, w


def resample_full(x, orig: int, new: int, lpw: int = 6, rolloff: float = 0.99, method: str = "sinc_interp_hann",
                  beta=None) -> np.ndarray:
    """torchaudio's full kernel over one signal x (len,), float64; orig == new returns x."""
    x = np.asarray(x, dtype=np.float64)
    if orig == new:
        return x.copy()
    O, N = reduced(orig, new)
    K, _, w = kernel(orig, new, lpw, rolloff, method, beta)
    n = x.shape[0]
    xp = np.pad(x, (w, w + O))
    k = np.arange(n // O + 1)
    X = xp[k[:, None] * O + np.arange(2 * w + O)[None, :]]
    return (X @ K.T).reshape(-1)[:output_length(n, orig, new)]


def resample_compact(x, table: np.ndarray, first: np.ndarray, w: int, orig: int, new: int) -> np.ndarray:
    """The compact form over one signal x (len,): y[kN + j] = sum_m table[m, j] x[kO + first[j] + m - w]."""
    x = np.asarray(x, dtype=np.float64)
    if orig == new:
        return x.copy()
    O, N = reduced(orig, new)
    L = table.shape[0]
    n = x.shape[0]
    n_out = output_length(n, orig, new)
    nn = np.arange(n_out)
    k, j = nn // N, nn % N
    idx = (k * O + first[j] - w)[:, None] + np.arange(L)[None, :]
    ok = (idx >= 0) & (idx < n)
    X = np.where(ok, x[np.clip(idx, 0, max(n - 1, 0))], 0.0)
    return (X * table[:, j].T).sum(1)
