"""Resampling throughput: the CUDA resampler (csrc/resample.cu) per utterance and on length-sorted batches with per-item
lengths, against torchaudio.functional.resample per utterance on the same GPU.

Workload: the 64 utterance durations of tools/bench_varlen.py (1-8 s, seeded), as uniform noise in [-1, 1] at the source
rate, for three rate pairs: 48 kHz -> 22.05 kHz, 16 kHz -> 22.05 kHz and 22.05 kHz -> 48 kHz (Hann window, lpw 6,
rolloff 0.99).  Modes, alternated in one run:
  solo           one Resample call per utterance;
  batch_N        length-sorted batches of N (16, 64) in one call each, with lengths;
  torchaudio     torchaudio.functional.resample per utterance (fp32, on the GPU).
Rates are VALID output samples per second (MHz), from CUDA events around each pass over all 64 utterances (synchronised,
warm-up excluded, L2 flushed by a 256 MB write before every pass); the minimum over --reps passes.  A pass of the batched
modes is one kernel launch per batch, so its time is kernel time plus the launch gaps.  Bytes per pass are counted from
shapes: the valid input samples read once, the padded output written once (the table is a few KB and stays in cache).
Prints one JSON line.

  python tools/bench_resample.py [--reps 5]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402
from tools.bench_varlen import gpu_info  # noqa: E402

PAIRS = [(48000, 22050), (16000, 22050), (22050, 48000)]
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resample: needs a CUDA device")
    import torchaudio
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(1234)
    secs = (torch.rand(args.utterances, generator=g) * 7 + 1).tolist()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    results = {}
    for orig, new in PAIRS:
        r = cm.Resample(orig, new).to(dev)
        gs = torch.Generator(device=dev).manual_seed(orig + new)
        sig = [torch.rand(int(s * orig), generator=gs, device=dev) * 2 - 1 for s in secs]
        order = sorted(range(len(sig)), key=lambda i: sig[i].numel())
        lens_all = [sig[i].numel() for i in range(len(sig))]
        valid = sum(r.output_lengths(lens_all))
        batches = {n: [pad_batch([sig[i] for i in order[s:s + n]]) for s in range(0, len(order), n)] for n in (16, 64)}

        def run(name):
            with torch.no_grad():
                if name == "solo":
                    for i in order:
                        r(sig[i])
                elif name == "torchaudio":
                    for i in order:
                        torchaudio.functional.resample(sig[i], orig, new)
                else:
                    for x, lens in batches[int(name[6:])]:
                        r(x, lengths=lens)

        names = ["solo", "batch_16", "batch_64", "torchaudio"]
        for name in names:   # warm-up: every shape once
            run(name)
        times = {name: [] for name in names}
        for _ in range(args.reps):
            for name in names:
                times[name].append(timed(lambda: run(name)))
        best = {k: min(v) for k, v in times.items()}

        def pass_bytes(items):
            return sum(4 * (sum(lens) + len(lens) * ((r.N * T + r.O - 1) // r.O)) for T, lens in items)

        nbytes = {"solo": pass_bytes([(n, [n]) for n in lens_all])}
        for n in (16, 64):
            nbytes[f"batch_{n}"] = pass_bytes([(x.shape[1], lens) for x, lens in batches[n]])
        # agreement with torchaudio on one batch, fp32 both sides (torchaudio builds its kernel in fp32 for an fp32
        # input); its conv1d runs in TF32 under torch's default cuDNN settings, so it is compared with TF32 off as well
        x, lens = batches[16][-1]
        worst = {}
        with torch.no_grad():
            y = r(x, lengths=lens)
            for key, tf32 in (("default_tf32", torch.backends.cudnn.allow_tf32), ("tf32_off", False)):
                worst[key] = 0.0
                with torch.backends.cudnn.flags(enabled=torch.backends.cudnn.enabled, allow_tf32=tf32):
                    for j, (n, m) in enumerate(zip(lens, r.output_lengths(lens))):
                        ref = torchaudio.functional.resample(x[j, :n], orig, new)
                        worst[key] = max(worst[key], ((y[j, :m] - ref).norm() / ref.norm()).item())
        results[f"{orig}->{new}"] = {
            "O": r.O, "N": r.N, "taps_per_phase": r.table.shape[0], "valid_output_samples": valid,
            "mhz": {k: round(valid / t / 1e6, 1) for k, t in best.items()},
            "pass_ms_min": {k: round(t * 1e3, 3) for k, t in best.items()},
            "speedup_over_torchaudio": {k: round(best["torchaudio"] / best[k], 1) for k in ("solo", "batch_16", "batch_64")},
            "bytes": {k: {"mbytes": round(v / 1e6, 2), "tbytes_per_s": round(v / best[k] / 1e12, 3),
                          "share_of_hbm_peak": round(v / best[k] / HBM_BYTES_PER_S, 4)} for k, v in nbytes.items()},
            "max_rel_l2_vs_torchaudio": worst,
            "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
        }
    name, power = gpu_info()
    print(json.dumps({"gpu": name, "power_limit": power, "utterances": len(secs),
                      "seconds_of_audio": round(sum(int(s * 22050) for s in secs) / 22050, 1), "l2_flushed": True,
                      "pairs": results}))


if __name__ == "__main__":
    main()
