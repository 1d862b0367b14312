"""fp64 reference of the spectral distances (constant_memory_waveglow_b200.SpectralDistance), test-only.

Per pair of 1-D signals, on the STFT and mel of oracle/tacotron_stft.py (Tacotron2's ``stft.STFT`` and
``TacotronSTFT.mel_spectrogram``): with S, S^ the magnitudes (n_fft/2 + 1 bins, len // hop + 1 frames), per frame

    LSD     sqrt(mean_k (X - X^)^2),                                X = log10(max(S^2, 1e-10))
    mel L1  mean_j |m_j - m^_j|,                                    m = ln(max(mel_basis @ S, 1e-5))
    MCD     (10 / ln 10) sqrt(2 sum_{d=1}^{n_cep-1} (c_d - c^_d)^2),  c = D m, D the orthonormal DCT-II (n_cep x n_mels)

and each metric is the mean of its frame terms.  D is scipy's ``dct(type=2, norm="ortho")`` of the identity.
"""
import numpy as np
import torch
from scipy.fft import dct

from . import tacotron_stft as TS


def dct_matrix(n_cep, n_mels):
    """(n_cep, n_mels) float64: rows 0 .. n_cep-1 of the orthonormal DCT-II, c = D @ m."""
    return dct(np.eye(n_mels), type=2, norm="ortho", axis=0)[:n_cep]


def frame_terms(ref, est, sampling_rate=22050, filter_length=1024, hop_length=256, win_length=1024, n_mel_channels=80,
                mel_fmin=0.0, mel_fmax=8000.0, n_cepstra=25, basis=None):
    """(lsd, mel_l1, mcd) per frame, three float64 arrays of len // hop + 1, for 1-D signals ref and est of one length.
    `basis` overrides the filterbank (for instance with the float32 table a module holds)."""
    ref, est = np.asarray(ref, dtype=np.float64), np.asarray(est, dtype=np.float64)
    assert ref.shape == est.shape and ref.ndim == 1
    if basis is None:
        basis = TS.mel_basis(sampling_rate, filter_length, n_mel_channels, mel_fmin, mel_fmax)
    basis = np.asarray(torch.as_tensor(basis).double())
    S = TS.stft_magnitude(torch.from_numpy(np.stack([ref, est])), filter_length, hop_length, win_length).numpy()
    X = np.log10(np.maximum(S ** 2, 1e-10))
    lsd = np.sqrt(np.mean((X[0] - X[1]) ** 2, axis=0))
    m = np.log(np.maximum(basis @ S, 1e-5))                  # (2, n_mels, frames)
    mel_l1 = np.mean(np.abs(m[0] - m[1]), axis=0)
    c = dct_matrix(n_cepstra, n_mel_channels) @ m
    mcd = 10.0 / np.log(10.0) * np.sqrt(2.0 * np.sum((c[0, 1:] - c[1, 1:]) ** 2, axis=0))
    return lsd, mel_l1, mcd


def distances(ref, est, **kw):
    """(lsd, mel_l1, mcd) of one pair: the means of frame_terms over the frames."""
    return tuple(float(np.mean(t)) for t in frame_terms(ref, est, **kw))
