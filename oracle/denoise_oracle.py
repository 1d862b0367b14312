"""fp64 numpy reference of the denoiser (constant_memory_waveglow_b200.Denoiser, csrc/denoise.cu), test-only.

STFT(x) = torch.stft(x, n_fft, hop, window=w, center=True, pad_mode="reflect", onesided=True); ISTFT = torch.istft(...,
center=True, length=n); denoise(x) = ISTFT(max(|S| - strength * bias, 0) * S / |S|) with 0 where |S| = 0.
"""
import numpy as np


def window(n_fft: int, win_length: int) -> np.ndarray:
    """Periodic Hann window of win_length samples, zero-padded to n_fft and centred (torch.stft's placement)."""
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(win_length) / win_length)
    left = (n_fft - win_length) // 2
    return np.pad(w, (left, n_fft - win_length - left))


def stft(x: np.ndarray, n_fft: int, hop: int, w: np.ndarray) -> np.ndarray:
    """(n_fft // 2 + 1, len(x) // hop + 1) complex128."""
    x = np.asarray(x, dtype=np.float64)
    if not n_fft // 2 < x.shape[-1]:
        raise ValueError("reflect padding needs more than n_fft // 2 samples")
    xp = np.pad(x, (n_fft // 2, n_fft // 2), mode="reflect")
    frames = x.shape[-1] // hop + 1
    idx = np.arange(frames)[:, None] * hop + np.arange(n_fft)[None, :]
    return np.fft.rfft(xp[idx] * w[None, :], axis=1).T


def istft(S: np.ndarray, n_fft: int, hop: int, w: np.ndarray, length: int) -> np.ndarray:
    """Windowed overlap-add of the inverse frames, divided by the overlap-add of w^2, trimmed by n_fft // 2."""
    frames = S.shape[1]
    y = np.fft.irfft(S.T, n=n_fft, axis=1) * w[None, :]
    total = n_fft + hop * (frames - 1)
    num, env = np.zeros(total), np.zeros(total)
    for f in range(frames):
        num[f * hop:f * hop + n_fft] += y[f]
        env[f * hop:f * hop + n_fft] += w * w
    sl = slice(n_fft // 2, n_fft // 2 + length)
    if np.abs(env[sl]).min() < 1e-11:
        raise ValueError("window overlap-add vanishes")
    return num[sl] / env[sl]


def denoise(x: np.ndarray, bias: np.ndarray, strength: float, n_fft: int, hop: int, w: np.ndarray) -> np.ndarray:
    S = stft(x, n_fft, hop, w)
    mag = np.abs(S)
    m = np.maximum(mag - strength * np.asarray(bias, dtype=np.float64)[:, None], 0.0)
    with np.errstate(invalid="ignore", divide="ignore"):
        gain = np.where(mag > 0, m / mag, 0.0)
    return istft(S * gain, n_fft, hop, w, x.shape[-1])


def bias_spectrum(bias_audio: np.ndarray, n_fft: int, hop: int, w: np.ndarray) -> np.ndarray:
    """|STFT(bias_audio)| of frame 0 (NVIDIA's mode 'zeros')."""
    return np.abs(stft(bias_audio, n_fft, hop, w)[:, 0])
