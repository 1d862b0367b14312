"""Exact fp32 outputs of this library's MelSpec kernel (cmwg_melspec_fwd) on fixed inputs, for the bit-identity check of
tests/test_gpu_denoise.py: the radix-2 FFT now lives in csrc/fft.cuh, shared with the denoiser, and MelSpec must give the
same bits it gave before that move.  Written on a B200 from the commit before the move:

    python tests/golden/make_golden_melspec_bits.py OUT.pt
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

# every transform size the kernel is instantiated for, both powers, a short centred window, odd lengths
CASES = [
    dict(sr=22050, n_fft=1024, hop_length=256, f_max=8000, n_mels=80),
    dict(sr=22050, n_fft=1024, hop_length=256, f_max=8000, n_mels=80, power=1),
    dict(sr=16000, n_fft=128, hop_length=32, n_mels=20),
    dict(sr=16000, n_fft=256, hop_length=64, n_mels=40, win_length=200),
    dict(sr=22050, n_fft=512, hop_length=128, n_mels=64),
    dict(sr=22050, n_fft=2048, hop_length=256, n_mels=128, win_length=1600, power=1),
    dict(sr=44100, n_fft=4096, hop_length=512, n_mels=160),
]
B, T, SEED = 2, 6001, 7


def inputs():
    g = torch.Generator().manual_seed(SEED)
    x = torch.rand(B, T, generator=g) * 2 - 1
    x[0, : T // 4] *= 1e-3
    return x


def compute(x):
    from constant_memory_waveglow_b200.condition import MelSpec
    with torch.no_grad():
        return [MelSpec(**c).cuda()(x.cuda()).cpu() for c in CASES]


def main():
    from constant_memory_waveglow_b200 import build
    build.build()
    x = inputs()
    torch.save({"cases": CASES, "x": x, "out": compute(x)}, sys.argv[1])


if __name__ == "__main__":
    main()
