"""Spectral-distance throughput: the fused CUDA pass (csrc/distance.cu) per pair and on length-sorted batches with per-item
lengths, against a per-utterance torch path on the same GPU.

Workload: the 64 utterance durations of tools/bench_varlen.py (1-8 s at 22.05 kHz, seeded), as pairs of independent uniform
noise in [-1, 1], with SpectralDistance's defaults (n_fft 1024, hop 256, 80 mels, 25 cepstra).  Modes, alternated in one run:
  solo       one SpectralDistance call per pair;
  batch_N    length-sorted batches of N (16, 64) in one call each, with lengths;
  torch      per pair: torch.stft(center=True, pad_mode="reflect") of both signals, then the same definitions with torch
             ops in fp32 (the module's mel basis and DCT), TF32 off.
Rates are VALID samples (of one signal of each pair) per second, from CUDA events around each pass over all 64 pairs
(synchronised, warm-up excluded, L2 flushed by a 256 MB write before every pass); the minimum over --reps passes.  Bytes
per pass are counted from shapes: both signals' valid samples read once, the per-frame terms written and read once (3 floats
per frame and item of the padded batch's workspace rows that are computed), the (B, 3) result written.  Frames overlap by
3/4, so each sample is fetched by four CTAs; the count assumes the repeats hit in cache.  Prints one JSON line.

  python tools/bench_distance.py [--reps 5]
"""
import argparse
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402
from tools.bench_varlen import gpu_info  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def torch_distances(sd, window, ref, est):
    """The three distances of one pair with torch ops (fp32), the definitions of SpectralDistance."""
    spec = torch.stft(torch.stack([ref, est]), sd.filter_length, sd.hop_length, window=window, center=True,
                      pad_mode="reflect", onesided=True, return_complex=True)
    P = spec.real ** 2 + spec.imag ** 2
    X = torch.log10(torch.clamp(P, min=1e-10))
    lsd = torch.sqrt(((X[0] - X[1]) ** 2).mean(0)).mean()
    m = torch.log(torch.clamp(sd.mel_basis @ spec.abs(), min=1e-5))
    dm = m[0] - m[1]
    mel_l1 = dm.abs().mean(0).mean()
    c = sd.dct[1:] @ dm
    mcd = (10 / math.log(10) * torch.sqrt(2 * (c ** 2).sum(0))).mean()
    return torch.stack([lsd, mel_l1, mcd])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_distance: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(1234)
    secs = (torch.rand(args.utterances, generator=g) * 7 + 1).tolist()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sd = cm.SpectralDistance().to(dev)
    window = torch.hann_window(sd.win_length, periodic=True, dtype=torch.float64).float().to(dev)
    gs = torch.Generator(device=dev).manual_seed(7)
    pairs = [(torch.rand(int(s * 22050), generator=gs, device=dev) * 2 - 1,
              torch.rand(int(s * 22050), generator=gs, device=dev) * 2 - 1) for s in secs]
    order = sorted(range(len(pairs)), key=lambda i: pairs[i][0].numel())
    lens_all = [r.numel() for r, _ in pairs]
    batches = {}
    for n in (16, 64):
        batches[n] = []
        for s in range(0, len(order), n):
            idx = order[s:s + n]
            x, lens = pad_batch([pairs[i][0] for i in idx])
            y, _ = pad_batch([pairs[i][1] for i in idx])
            batches[n].append((idx, x, y, lens))

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    def run(name):
        with torch.no_grad():
            if name == "solo":
                for i in order:
                    sd(*pairs[i])
            elif name == "torch":
                for i in order:
                    torch_distances(sd, window, *pairs[i])
            else:
                for _, x, y, lens in batches[int(name[6:])]:
                    sd(x, y, lengths=lens)

    names = ["solo", "batch_16", "batch_64", "torch"]
    for name in names:   # warm-up: every shape once
        run(name)
    times = {name: [] for name in names}
    for _ in range(args.reps):
        for name in names:
            times[name].append(timed(lambda: run(name)))
    best = {k: min(v) for k, v in times.items()}
    valid = sum(lens_all)
    hop = sd.hop_length

    def pass_bytes(items):
        # items: (padded T, lengths) per call
        return sum(2 * 4 * sum(lens) + 2 * 3 * 4 * sum(n // hop + 1 for n in lens) + 3 * 4 * len(lens) for _, lens in items)

    nbytes = {"solo": pass_bytes([(n, [n]) for n in lens_all])}
    for n in (16, 64):
        nbytes[f"batch_{n}"] = pass_bytes([(x.shape[1], lens) for _, x, _, lens in batches[n]])
    # agreement with the torch path, every pair, from the batches of 16
    worst = [0.0, 0.0, 0.0]
    with torch.no_grad():
        for idx, x, y, lens in batches[16]:
            ours = torch.stack(sd(x, y, lengths=lens), 1)
            for j, i in enumerate(idx):
                ref = torch_distances(sd, window, *pairs[i])
                for k in range(3):
                    worst[k] = max(worst[k], abs(ours[j, k].item() - ref[k].item()) / abs(ref[k].item()))
    name, power = gpu_info()
    print(json.dumps({
        "gpu": name, "power_limit": power, "utterances": len(secs), "seconds_of_audio": round(valid / 22050, 1),
        "l2_flushed": True, "valid_samples": valid,
        "msamples_per_s": {k: round(valid / t / 1e6, 1) for k, t in best.items()},
        "pass_ms_min": {k: round(t * 1e3, 3) for k, t in best.items()},
        "speedup_over_torch": {k: round(best["torch"] / best[k], 1) for k in ("solo", "batch_16", "batch_64")},
        "bytes": {k: {"mbytes": round(v / 1e6, 2), "tbytes_per_s": round(v / best[k] / 1e12, 3),
                      "share_of_hbm_peak": round(v / best[k] / HBM_BYTES_PER_S, 4)} for k, v in nbytes.items()},
        "max_rel_diff_vs_torch": {"lsd": worst[0], "mel_l1": worst[1], "mcd": worst[2]},
        "tf32": False,
    }))


if __name__ == "__main__":
    main()
