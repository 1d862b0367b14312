"""fp64 reference of Tacotron2's mel front end (constant_memory_waveglow_b200.TacotronSTFT), test-only.

A literal restatement of NVIDIA/tacotron2 ``stft.STFT.transform`` and ``layers.TacotronSTFT.mel_spectrogram``:
the Fourier basis is ``np.fft.fft(np.eye(n_fft))`` cut to n_fft/2 + 1 rows (real parts, then imaginary parts) times the
window; the input is reflect-padded by n_fft/2 on both sides and convolved with that basis at stride hop; the magnitude
is ``sqrt(re^2 + im^2)``; the mel is ``mel_basis @ magnitude`` and the output ``log(clamp(mel, min=1e-5))``.  The
filterbank restates librosa's ``filters.mel`` (Slaney mel scale, Slaney normalisation) in float64 numpy.
"""
import numpy as np
import torch
import torch.nn.functional as F
from scipy.signal import get_window


def hz_to_mel(frequencies):
    """librosa.hz_to_mel(htk=False)."""
    frequencies = np.asanyarray(frequencies, dtype=np.float64)
    f_min, f_sp = 0.0, 200.0 / 3
    mels = (frequencies - f_min) / f_sp
    min_log_hz = 1000.0
    min_log_mel = (min_log_hz - f_min) / f_sp
    logstep = np.log(6.4) / 27.0
    if frequencies.ndim:
        log_t = frequencies >= min_log_hz
        mels[log_t] = min_log_mel + np.log(frequencies[log_t] / min_log_hz) / logstep
    elif frequencies >= min_log_hz:
        mels = min_log_mel + np.log(frequencies / min_log_hz) / logstep
    return mels


def mel_to_hz(mels):
    """librosa.mel_to_hz(htk=False)."""
    mels = np.asanyarray(mels, dtype=np.float64)
    f_min, f_sp = 0.0, 200.0 / 3
    freqs = f_min + f_sp * mels
    min_log_hz = 1000.0
    min_log_mel = (min_log_hz - f_min) / f_sp
    logstep = np.log(6.4) / 27.0
    log_t = mels >= min_log_mel
    freqs[log_t] = min_log_hz * np.exp(logstep * (mels[log_t] - min_log_mel))
    return freqs


def mel_basis(sr, n_fft, n_mels, fmin=0.0, fmax=None):
    """librosa.filters.mel(sr=sr, n_fft=n_fft, n_mels=n_mels, fmin=fmin, fmax=fmax, htk=False, norm='slaney') in float64
    (librosa stores the weights as float32 before normalising; here nothing is rounded)."""
    if fmax is None:
        fmax = float(sr) / 2
    weights = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float64)
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    mel_f = mel_to_hz(np.linspace(hz_to_mel(fmin), hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, np.newaxis]
    return weights


def forward_basis(filter_length, win_length):
    """stft.STFT.__init__: (2 (n_fft/2 + 1), 1, n_fft) float64, the windowed real and imaginary Fourier rows."""
    fourier_basis = np.fft.fft(np.eye(filter_length))
    cutoff = int(filter_length / 2 + 1)
    fourier_basis = np.vstack([np.real(fourier_basis[:cutoff, :]), np.imag(fourier_basis[:cutoff, :])])
    basis = torch.from_numpy(fourier_basis[:, None, :])
    fft_window = get_window("hann", win_length, fftbins=True)
    lpad = (filter_length - win_length) // 2                 # librosa.util.pad_center
    fft_window = np.pad(fft_window, (lpad, filter_length - win_length - lpad))
    return basis * torch.from_numpy(fft_window).double()


def stft_magnitude(y, filter_length, hop_length, win_length):
    """stft.STFT.transform: y (B, T) -> |STFT| (B, n_fft/2 + 1, T // hop + 1), float64."""
    y = torch.as_tensor(y).double()
    num_batches, num_samples = y.shape
    x = y.view(num_batches, 1, num_samples)
    x = F.pad(x.unsqueeze(1), (filter_length // 2, filter_length // 2, 0, 0), mode="reflect").squeeze(1)
    ft = F.conv1d(x, forward_basis(filter_length, win_length).to(x.device), stride=hop_length, padding=0)
    cutoff = filter_length // 2 + 1
    real, imag = ft[:, :cutoff, :], ft[:, cutoff:, :]
    return torch.sqrt(real ** 2 + imag ** 2)


def mel_spectrogram(y, filter_length=1024, hop_length=256, win_length=1024, n_mel_channels=80, sampling_rate=22050,
                    mel_fmin=0.0, mel_fmax=8000.0, basis=None):
    """layers.TacotronSTFT.mel_spectrogram: y (B, T) -> (B, n_mels, T // hop + 1), float64.  `basis` overrides the
    filterbank (for instance with the float32 table a module holds)."""
    mag = stft_magnitude(y, filter_length, hop_length, win_length)
    if basis is None:
        basis = mel_basis(sampling_rate, filter_length, n_mel_channels, mel_fmin, mel_fmax)
    mel = torch.matmul(torch.as_tensor(basis).double().to(mag.device), mag)
    return torch.log(torch.clamp(mel, min=1e-5))
