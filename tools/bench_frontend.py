"""Mel front-end throughput: TacotronSTFT.mel_spectrogram (csrc/melspec.cu, cmwg_melspec_fwd_varlen) per utterance and on
length-sorted batches with per-item lengths, against NVIDIA's conv-basis STFT restated in PyTorch (fp32), and as a share of
the synthesis of the same batches.

Workload (that of tools/bench_varlen.py): 64 utterances of 1-8 s (seeded) at 22.05 kHz, audio uniform in [-0.5, 0.5];
TacotronSTFT defaults (filter_length 1024, hop 256, 80 mels, fmax 8 kHz).  Modes, alternated in one run:
  solo          one mel_spectrogram call per utterance;
  batch_N       length-sorted batches of N (16, 64) in one call each, with lengths;
  torch_solo    NVIDIA's stft.STFT.transform + mel_basis matmul + log(clamp) in fp32 PyTorch (conv1d with the windowed
                Fourier basis), one utterance per call, on the same GPU;
  synth_N       NvidiaWaveGlow.infer(h, lengths=frames) of the same batches (published configuration, random weights):
                the synthesis the front end precedes in copy synthesis.
Rates are VALID samples per second (MHz), from CUDA events around each pass over all utterances (synchronised, warm-up
excluded, L2 flushed by a 256 MB write before every pass); the minimum over --reps passes.  Prints one JSON line.

  python tools/bench_frontend.py [--reps 5]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402
from tools.bench_varlen import HOP, SIGMA, SR, gpu_info  # noqa: E402

PUBLISHED = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
                 WN_config=dict(n_layers=8, n_channels=256, kernel_size=3))


def torch_frontend(t: cm.TacotronSTFT, dev):
    """NVIDIA's TacotronSTFT.mel_spectrogram (stft.py / layers.py) in fp32 PyTorch on `dev`."""
    n_fft = t.filter_length
    fb = np.fft.fft(np.eye(n_fft))
    cut = n_fft // 2 + 1
    basis = torch.from_numpy(np.vstack([np.real(fb[:cut]), np.imag(fb[:cut])])[:, None, :]).float()
    w = torch.hann_window(t.win_length, periodic=True, dtype=torch.float64).float()
    left = (n_fft - t.win_length) // 2
    basis = (basis * F.pad(w, (left, n_fft - t.win_length - left))).to(dev)
    mel_basis = t.mel_basis.to(dev)

    def run(y):
        # true fp32 convolution; the flag is scoped because the package's precision policy reads it too
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            x = F.pad(y.view(1, 1, 1, -1), (n_fft // 2, n_fft // 2, 0, 0), mode="reflect").squeeze(1)
            ft = F.conv1d(x, basis, stride=t.hop_length)
            mag = torch.sqrt(ft[:, :cut] ** 2 + ft[:, cut:] ** 2)
            return torch.log(torch.clamp(torch.matmul(mel_basis, mag), min=1e-5))
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_frontend: needs a CUDA device")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    m = cm.NvidiaWaveGlow(**PUBLISHED)
    with torch.no_grad():
        for p in m.parameters():
            p.normal_(0, 0.02)
    m = m.to(dev).eval()
    t = cm.TacotronSTFT().to(dev)
    g = torch.Generator().manual_seed(1234)
    secs = torch.rand(args.utterances, generator=g) * 7 + 1
    samples = [int(s * SR) for s in secs.tolist()]
    audio = [((torch.rand(n, generator=g) - 0.5)).to(dev) for n in samples]
    order = sorted(range(len(samples)), key=lambda i: samples[i])
    valid = sum(samples)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ref = torch_frontend(t, dev)

    batches = {n: [pad_batch([audio[i] for i in order[s:s + n]]) for s in range(0, len(order), n)] for n in (16, 64)}
    synth = {}
    with torch.no_grad():
        for n in (16, 64):
            synth[n] = []
            for x, lens in batches[n]:
                mel = t.mel_spectrogram(x, lengths=lens)
                frames = [k // HOP + 1 for k in lens]
                synth[n].append((mel, frames, torch.randn(len(lens), mel.shape[-1] * HOP, device=dev) * SIGMA))

    def run(name):
        with torch.no_grad():
            if name == "solo":
                for i in order:
                    t.mel_spectrogram(audio[i])
            elif name == "torch_solo":
                for i in order:
                    ref(audio[i])
            elif name.startswith("batch_"):
                for x, lens in batches[int(name[6:])]:
                    t.mel_spectrogram(x, lengths=lens)
            else:
                for h, fl, z in synth[int(name[6:])]:
                    m.infer(h, SIGMA, z=z, lengths=fl)

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    names = ["solo", "batch_16", "batch_64", "torch_solo", "synth_16", "synth_64"]
    for name in names:   # warm-up: every shape once
        run(name)
    times = {name: [] for name in names}
    for _ in range(args.reps):
        for name in names:
            times[name].append(timed(lambda: run(name)))
    best = {k: min(v) for k, v in times.items()}
    mhz = {k: valid / v / 1e6 for k, v in best.items()}

    # agreement with the PyTorch restatement (fp32 both sides), over every utterance's valid frames
    with torch.no_grad():
        worst = 0.0
        for x, lens in batches[16]:
            mel = t.mel_spectrogram(x, lengths=lens)
            for j, n in enumerate(lens):
                worst = max(worst, (mel[j, :, :n // HOP + 1] - ref(x[j, :n])[0]).abs().max().item())
    name, power = gpu_info()
    print(json.dumps({
        "gpu": name, "power_limit": power, "utterances": len(samples), "valid_samples": valid,
        "seconds_of_audio": round(valid / SR, 2), "filter_length": t.filter_length, "hop": t.hop_length,
        "mhz": {k: round(v, 1) for k, v in mhz.items()},
        "pass_ms_min": {k: round(v * 1e3, 3) for k, v in best.items()},
        "share_of_synthesis": {f"batch_{n}": round(best[f"batch_{n}"] / best[f"synth_{n}"], 5) for n in (16, 64)},
        "speedup_over_torch_solo": {k: round(best["torch_solo"] / best[k], 2) for k in ("solo", "batch_16", "batch_64")},
        "max_abs_log_mel_vs_torch": worst,
    }))


if __name__ == "__main__":
    main()
