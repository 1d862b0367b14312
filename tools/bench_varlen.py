"""Batched synthesis of utterances of different lengths: per-item lengths against one call per utterance and against padding.

Workload: the LJ configuration (12 flows, n_group 8, 256-channel WN of depth 8), random weights (zero_init=False, weight
norm removed), 64 utterances with lengths drawn from a seeded uniform 1-8 s at 22.05 kHz, sigma 0.6, default precision.
Modes, alternated in one run:
  solo        one utterance per infer() call;
  varlen_N    length-sorted batches of N (4, 16, 64) through infer(h, lengths=frames);
  padded_N    the same batches padded to their longest item without lengths (wrong output for the shorter items: it shows
              what the padding costs).
Regression leg: 4 x 10 s, all lengths equal, the per-item-lengths path against the ordinary one.
Rates are VALID audio samples per second (kHz), from CUDA events around each pass (synchronised, warm-up excluded, L2 flushed
by a 256 MB write before every pass).  Prints one JSON line.

  python tools/bench_varlen.py [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402

SR, HOP, N_GROUP, SIGMA = 22050, 256, 8, 0.6


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return name, power
    except Exception as e:  # pragma: no cover
        return torch.cuda.get_device_name(), f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--utterances", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_varlen: needs a CUDA device")
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

    def batches(n):
        out = []
        for s in range(0, len(order), n):
            idx = order[s:s + n]
            h, fl = pad_batch([mels[i] for i in idx])
            z, _ = pad_batch([noise[i] for i in idx])
            out.append((h, fl, z))
        return out

    plans = {"solo": [(mels[i][None], [frames[i]], noise[i][None]) for i in order]}
    for n in (4, 16, 64):
        plans[f"varlen_{n}"] = batches(n)
        plans[f"padded_{n}"] = plans[f"varlen_{n}"]

    def run(name):
        with torch.no_grad():
            for h, fl, z in plans[name]:
                if name.startswith("varlen"):
                    m.infer(h, SIGMA, z=z, lengths=fl)
                else:
                    m.infer(h, SIGMA, z=z)

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    for name in plans:   # warm-up: every shape once (descriptor encodes, workspace growth)
        run(name)
    times = {name: [] for name in plans}
    for _ in range(args.reps):
        for name in plans:
            times[name].append(timed(lambda: run(name)))
    khz = {name: valid / min(ts) / 1e3 for name, ts in times.items()}

    tiles = lambda n: -(-(n * HOP // N_GROUP) // 256)  # noqa: E731  (row tiles of one WN call per item)
    row_tiles = {}
    for n in (4, 16, 64):
        ex = sum(tiles(frames[i]) for i in order)
        padded = sum(len(idx) * tiles(max(frames[i] for i in idx))
                     for idx in (order[s:s + n] for s in range(0, len(order), n)))
        row_tiles[f"batch_{n}"] = {"executed": ex, "padded": padded}

    # regression leg: 4 x 10 s, all lengths equal -- the per-item-lengths path (called directly: the public entry routes
    # all-equal lengths to the ordinary path) against the ordinary one
    f10 = 10 * SR // HOP
    h10 = torch.randn(4, 80, f10, generator=g).to(dev)
    z10 = torch.randn(4, f10 * HOP, generator=g).to(dev) * SIGMA
    lens10 = [f10 * HOP] * 4
    with torch.no_grad():
        reg = {"ordinary": lambda: m.reverse(z10, h10),
               "varlen": lambda: m._direct_reverse(*m._varlen_prepare(z10, h10, lens10))}
        for fn in reg.values():
            fn()
        rt = {k: [] for k in reg}
        for _ in range(args.reps * 2):
            for k, fn in reg.items():
                rt[k].append(timed(fn))
        same = torch.equal(m.reverse(z10, h10)[0], reg["varlen"]()[0])
    name, power = gpu_info()
    print(json.dumps({
        "gpu": name, "power_limit": power, "utterances": len(frames), "valid_samples": valid,
        "seconds_of_audio": valid / SR, "khz": {k: round(v, 1) for k, v in khz.items()},
        "pass_seconds_min": {k: round(min(v), 5) for k, v in times.items()},
        "row_tiles_per_wn_call": row_tiles,
        "regression_4x10s": {"ordinary_ms": [round(t * 1e3, 3) for t in rt["ordinary"]],
                             "varlen_ms": [round(t * 1e3, 3) for t in rt["varlen"]], "same_audio": same},
    }))


if __name__ == "__main__":
    main()
