"""Compare this package's NvidiaWaveGlow with NVIDIA's own code and checkpoint: for a user who has NVIDIA/waveglow (its
glow.py) and a published checkpoint.

    python tools/compare_nvidia_waveglow.py --glow-dir PATH/TO/waveglow CKPT [--frames 200] [--sigma 0.6] [--seed 0]

Builds NVIDIA's glow.WaveGlow from the dimensions found in CKPT and loads the checkpoint's weights into it (the file itself
is read by load_nvidia_waveglow's reader, which runs no code from it), replays the noise NVIDIA's infer() draws into this
package's infer(z=...), and prints the relative L2 difference of the two syntheses on random mels as one JSON line.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200 import nvidia  # noqa: E402


def nvidia_keyed(sd, n_layers):
    """NVIDIA-keyed weights for the current glow.py, which has one cond_layer per WN."""
    out = dict(sd)
    k = 0
    while f"WN.{k}.cond_layers.0.bias" in out:
        for n in ("weight_g", "weight_v", "weight", "bias"):
            parts = [out.pop(f"WN.{k}.cond_layers.{i}.{n}") for i in range(n_layers) if f"WN.{k}.cond_layers.{i}.{n}" in out]
            if parts:
                out[f"WN.{k}.cond_layer.{n}"] = torch.cat(parts, 0)
        k += 1
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("ckpt")
    ap.add_argument("--glow-dir", default=None, help="a checkout of NVIDIA/waveglow (the directory holding glow.py)")
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--sigma", type=float, default=0.6)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not args.glow_dir:
        raise SystemExit("compare_nvidia_waveglow: pass --glow-dir DIR, a checkout of NVIDIA/waveglow: this check runs "
                         "NVIDIA's own glow.py against this package")
    sys.path.insert(0, os.path.abspath(args.glow_dir))
    import glow  # noqa: E402  (NVIDIA's module)

    sd = nvidia.nvidia_state_dict(nvidia._read_checkpoint(args.ckpt))
    cfg, _ = nvidia.convert_state_dict(sd)
    theirs = glow.WaveGlow(cfg["n_mel_channels"], cfg["n_flows"], cfg["n_group"], cfg["n_early_every"],
                           cfg["n_early_size"], cfg["WN_config"])
    if not any(k.endswith("weight_g") for k in sd):
        theirs = glow.WaveGlow.remove_weightnorm(theirs)
    theirs.load_state_dict(nvidia_keyed(sd, cfg["WN_config"]["n_layers"]))
    theirs = theirs.cuda().eval()
    ours = cm.load_nvidia_waveglow(args.ckpt)

    g = torch.Generator().manual_seed(args.seed)
    mel = (torch.randn(args.batch, cfg["n_mel_channels"], args.frames, generator=g) - 5.0).cuda()
    with torch.no_grad():
        torch.cuda.manual_seed(args.seed)
        audio_theirs = theirs.infer(mel, sigma=args.sigma).float()
        # the same draws in the same order: (B, n_remaining, T') first, then (B, n_early_size, T') per early output
        torch.cuda.manual_seed(args.seed)
        Tq = args.frames * 256 // cfg["n_group"]
        rem = cfg["n_group"] - cfg["n_early_size"] * ((cfg["n_flows"] - 1) // cfg["n_early_every"])
        parts = [torch.cuda.FloatTensor(args.batch, rem, Tq).normal_()]
        for k in reversed(range(cfg["n_flows"])):
            if k % cfg["n_early_every"] == 0 and k > 0:
                parts.insert(0, torch.cuda.FloatTensor(args.batch, cfg["n_early_size"], Tq).normal_())
        zs = args.sigma * torch.cat(parts, 1)                       # squeezed (B, n_group, T')
        z = zs.permute(0, 2, 1).reshape(args.batch, -1)
        audio_ours = ours.infer(mel, args.sigma, z=z)
    d = audio_ours.double() - audio_theirs.double()
    print(json.dumps({"checkpoint": os.path.basename(args.ckpt), "precision": cm.get_precision(), "samples": z.shape[1],
                      "rel_l2": (d.norm() / audio_theirs.double().norm()).item(), "max_abs": d.abs().max().item()}))


if __name__ == "__main__":
    main()
