"""Denoiser throughput: the CUDA denoiser (csrc/denoise.cu) per utterance and on length-sorted batches with per-item lengths,
against torch.stft / torch.istft per utterance, and as a share of the synthesis of the same batches.

Workload (that of tools/bench_varlen.py): the LJ-configuration WaveGlow (12 flows, n_group 8, 256-channel WN of depth 8,
random weights), 64 utterances of 1-8 s (seeded) at 22.05 kHz synthesised with sigma 0.6; Denoiser(model) defaults
(filter_length 1024, hop 256), strength 0.1.  Modes, alternated in one run:
  solo          one Denoiser call per utterance;
  batch_N       length-sorted batches of N (16, 64) in one call each, with lengths;
  torch_solo    torch.stft -> magnitude subtraction -> torch.istft per utterance on the same GPU;
  synth_N       infer(h, lengths=frames) of the same batches (the synthesis the denoiser follows in `cli synth-batch`).
Rates are VALID samples per second (MHz), from CUDA events around each pass over all 64 utterances (synchronised, warm-up
excluded, L2 flushed by a 256 MB write before every pass); the minimum over --reps passes.  Bytes per pass are counted from
shapes: the audio read once, the (frames x n_fft) fp32 workspace written and read once, the padded output written.
Prints one JSON line.

  python tools/bench_denoise.py [--reps 5]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402
from tools.bench_varlen import HOP, N_GROUP, SIGMA, SR, gpu_info  # noqa: E402

STRENGTH = 0.1
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_denoise: needs a CUDA device")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    m = cm.WaveGlow(12, N_GROUP, 4, 2, HOP, 80, True, zero_init=False)
    m.apply(cm.remove_weight_norms)
    m = m.to(dev).eval()
    g = torch.Generator().manual_seed(1234)
    secs = torch.rand(args.utterances, generator=g) * 7 + 1
    frames = [max(1, int(s * SR) // HOP) for s in secs.tolist()]
    mels = [torch.randn(80, f, generator=g).to(dev) for f in frames]
    noise = [torch.randn(f * HOP, generator=g).to(dev) * SIGMA for f in frames]
    order = sorted(range(len(frames)), key=lambda i: frames[i])
    valid = sum(frames) * HOP
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    d = cm.Denoiser(m)
    n_fft, hop = d.filter_length, d.hop_length

    synth, audio = {}, [None] * len(frames)
    for n in (16, 64):
        synth[n] = []
        for s in range(0, len(order), n):
            idx = order[s:s + n]
            h, fl = pad_batch([mels[i] for i in idx])
            z, _ = pad_batch([noise[i] for i in idx])
            synth[n].append((h, fl, z))
            with torch.no_grad():
                x = m.infer(h, SIGMA, z=z, lengths=fl)
            for j, i in enumerate(idx):
                audio[i] = x[j, :fl[j] * HOP].clone()
    batches = {n: [pad_batch([audio[i] for i in order[s:s + n]]) for s in range(0, len(order), n)] for n in (16, 64)}

    def torch_denoise(x):
        S = torch.stft(x, n_fft, hop, window=d.window, center=True, pad_mode="reflect", onesided=True, return_complex=True)
        mag = S.abs()
        gain = torch.where(mag > 0, torch.clamp(mag - STRENGTH * d.bias_spec[:, None], min=0) / mag, torch.zeros_like(mag))
        return torch.istft(S * gain, n_fft, hop, window=d.window, center=True, length=x.shape[-1])

    def run(name):
        with torch.no_grad():
            if name == "solo":
                for i in order:
                    d(audio[i], STRENGTH)
            elif name == "torch_solo":
                for i in order:
                    torch_denoise(audio[i])
            elif name.startswith("batch_"):
                for x, lens in batches[int(name[6:])]:
                    d(x, STRENGTH, lengths=lens)
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
    mhz = {k: valid / t / 1e6 for k, t in best.items()}

    def pass_bytes(items):
        """(T_padded, lengths) per call -> bytes the two kernels need: audio in, workspace out and in, output out."""
        total = 0
        for T, lens in items:
            total += 4 * (sum(lens) + 2 * sum((n // hop + 1) * n_fft for n in lens) + len(lens) * T)
        return total

    nbytes = {"solo": pass_bytes([(len(audio[i]), [len(audio[i])]) for i in order])}
    for n in (16, 64):
        nbytes[f"batch_{n}"] = pass_bytes([(x.shape[1], lens) for x, lens in batches[n]])
    hbm = {k: {"gbytes": round(v / 1e9, 4), "tbytes_per_s": round(v / best[k] / 1e12, 3),
               "share_of_hbm_peak": round(v / best[k] / HBM_BYTES_PER_S, 4)} for k, v in nbytes.items()}

    # agreement with the torch path on one batch (fp32 both sides)
    x, lens = batches[16][-1]
    with torch.no_grad():
        ours = d(x, STRENGTH, lengths=lens)
        worst = max(((ours[j, :n] - torch_denoise(x[j, :n])).norm() / torch_denoise(x[j, :n]).norm()).item()
                    for j, n in enumerate(lens))
    name, power = gpu_info()
    print(json.dumps({
        "gpu": name, "power_limit": power, "utterances": len(frames), "valid_samples": valid,
        "seconds_of_audio": round(valid / SR, 2), "n_fft": n_fft, "hop": hop, "strength": STRENGTH,
        "mhz": {k: round(v, 1) for k, v in mhz.items()},
        "pass_ms_min": {k: round(v * 1e3, 3) for k, v in best.items()},
        "share_of_synthesis": {f"batch_{n}": round(best[f"batch_{n}"] / best[f"synth_{n}"], 5) for n in (16, 64)},
        "speedup_over_torch_solo": {k: round(best["torch_solo"] / best[k], 2) for k in ("solo", "batch_16", "batch_64")},
        "kernel_bytes": hbm, "max_rel_l2_vs_torch": worst,
    }))


if __name__ == "__main__":
    main()
