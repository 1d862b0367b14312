"""Command line of the harness: ``python -m constant_memory_waveglow_b200.cli {train,synth,synth-batch} ...``.

The reference's own ``train.py`` runs unchanged on the ``pytorch_lightning`` / ``model`` / ``datasets`` shims at the
repository root; its ``inference.py`` cannot in this image (``torchaudio.load`` / ``save`` need the absent TorchCodec),
so the two entry points exist here with the reference's flags (``train.py:81-93``, ``inference.py:62-70``) on top of the
RIFF reader/writer of ``datasets.py``.  Multi-GPU: launch ``train`` under ``torchrun --nproc-per-node N``.  ``synth-batch``
re-synthesises many files, batching utterances of different lengths into one call each (``WaveGlow.infer(lengths=...)``).
``-d/--denoiser-strength`` on ``synth`` and ``synth-batch`` runs the bias-spectrum ``Denoiser`` on the output (one call per
batch, with the per-item lengths); at 0, the default, it is skipped.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch

from . import trainer as TR
from .datasets import wav_read, wav_write
from .utils import remove_weight_norms


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return out, a.elapsed_time(b) / 1e3


def train(argv) -> None:
    p = argparse.ArgumentParser(prog="cli train", description="constant-memory WaveGlow training (train.py flags)")
    p = TR.Trainer.add_argparse_args(TR.LightModel.add_model_specific_args(p))
    p.add_argument("--config", type=str)
    p.add_argument("--ckpt-path", type=str)
    p.add_argument("--seed", type=int, default=None)
    p.add_argument("--lr", type=float, default=None, help="force learning rate")
    p.add_argument("--no-tf32", action="store_true", help="fp32 operands on the exact engine (train.py:92-97)")
    args = p.parse_args(argv)
    if args.no_tf32:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    config = json.load(open(args.config)) if args.config else None
    TR.seed_everything(args.seed)
    world = max(1, int(__import__("os").environ.get("WORLD_SIZE", "1")))
    if config is not None:
        config["data_loader"]["batch_size"] //= world          # train.py:51-53: the configured batch is global
    if args.ckpt_path:
        lit = TR.LightModel.load_from_checkpoint(args.ckpt_path, **({"config": config} if config is not None else {}))
    else:
        if config is None:
            p.error("--config or --ckpt-path is required")
        lit = TR.LightModel(config)

    class _ForceLR(TR.Callback):
        def on_train_start(self, trainer, pl_module):
            for o in trainer.optimizers:
                for g in o.param_groups:
                    g["lr"] = args.lr

    cbs = [TR.ModelSummary(max_depth=2), TR.LearningRateMonitor("epoch")] + ([_ForceLR()] if args.lr else [])
    if args.max_epochs is None and args.max_steps in (-1, None):
        args.max_epochs = 100                                   # train.py:76
    tr = TR.Trainer.from_argparse_args(args, callbacks=cbs, detect_anomaly=True)
    tr.fit(lit, ckpt_path=args.ckpt_path)


def synth(argv) -> None:
    p = argparse.ArgumentParser(prog="cli synth", description="analysis + synthesis of one file (inference.py flags)")
    p.add_argument("ckpt", type=str)
    p.add_argument("infile", type=str)
    p.add_argument("outfile", type=str)
    p.add_argument("-s", "--sigma", type=float, default=0.6)
    p.add_argument("-n", "--n-group", type=int, default=None)
    _add_denoiser_arg(p)
    args = p.parse_args(argv)
    _check_denoiser_arg(p, args)
    lit = TR.LightModel.load_from_checkpoint(args.ckpt, map_location="cpu")
    model, conditioner = lit.model, lit.conditioner
    model.apply(remove_weight_norms)
    dev = torch.device("cuda")
    model, conditioner = model.to(dev).eval(), conditioner.to(dev)
    from .datasets import wav_info
    sr = wav_info(args.infile).sample_rate
    y = wav_read(args.infile).mean(0, keepdim=True).to(dev)
    if args.n_group and y.shape[1] % args.n_group:
        y = y[:, :-(y.shape[1] % args.n_group)]
    cond = conditioner(y)
    with torch.no_grad():
        (z, logdet), cost = _timed(lambda: model(y.clone(), cond))
        z = z.squeeze()
        print(z.mean().item(), z.std().item())
        print("Forward LL:", logdet.mean().item() / z.size(0) - 0.5 * (
            z.pow(2).mean().item() / args.sigma ** 2 + math.log(2 * math.pi) + 2 * math.log(args.sigma)))
        print("Time cost: {:.4f}, Speed: {:.4f} kHz".format(cost, z.numel() / cost / 1000))
        x, cost = _timed(lambda: model.infer(cond, args.sigma))
    print("Time cost: {:.4f}, Speed: {:.4f} kHz".format(cost, x.numel() / cost / 1000))
    if args.denoiser_strength > 0:
        x = _denoiser(model, x.numel(), p)(x, args.denoiser_strength)
    print(x.max().item(), x.min().item())
    wav_write(args.outfile, x.reshape(1, -1), sr)


def _add_denoiser_arg(p: argparse.ArgumentParser) -> None:
    p.add_argument("-d", "--denoiser-strength", type=float, default=0.0,
                   help="subtract this multiple of the model's bias spectrum from the output (Denoiser); 0 = off")


def _check_denoiser_arg(p: argparse.ArgumentParser, args) -> None:
    if not 0 <= args.denoiser_strength < math.inf:
        p.error("--denoiser-strength must be a finite number >= 0")


def _denoiser(model, shortest: int, p: argparse.ArgumentParser):
    """The Denoiser of `model` for outputs of at least `shortest` samples (its STFT needs more than filter_length / 2)."""
    from .denoiser import Denoiser
    d = Denoiser(model)
    if shortest <= d.filter_length // 2:
        p.error(f"--denoiser-strength: an output of {shortest} samples is too short to denoise "
                f"(more than {d.filter_length // 2} needed)")
    return d


def _load_for_synthesis(ckpt: str):
    lit = TR.LightModel.load_from_checkpoint(ckpt, map_location="cpu")
    model, conditioner = lit.model, lit.conditioner
    model.apply(remove_weight_norms)
    dev = torch.device("cuda")
    return model.to(dev).eval(), conditioner.to(dev), dev


def item_noise(seed: int, index: int, n: int, sigma: float) -> torch.Tensor:
    """The noise of file `index` (command-line order) of a synth-batch run: N(0, sigma^2), n samples, from a CPU generator
    seeded by (seed, index) alone -- a rerun reproduces every file whatever the batching."""
    g = torch.Generator().manual_seed(int(seed) * 1_000_003 + int(index))
    return torch.randn(n, generator=g) * sigma


def synth_batch(argv) -> None:
    p = argparse.ArgumentParser(prog="cli synth-batch",
                                description="analysis + synthesis of many files, batched by length (one output per input)")
    p.add_argument("ckpt", type=str)
    p.add_argument("outdir", type=str)
    p.add_argument("infiles", type=str, nargs="+")
    p.add_argument("-s", "--sigma", type=float, default=0.6)
    p.add_argument("--max-batch", type=int, default=16, help="utterances per synthesis call")
    p.add_argument("--seed", type=int, default=0, help="noise seed; file i draws from a generator seeded by (seed, i)")
    _add_denoiser_arg(p)
    args = p.parse_args(argv)
    _check_denoiser_arg(p, args)
    if args.max_batch < 1:
        p.error("--max-batch must be >= 1")
    stems = [os.path.splitext(os.path.basename(f))[0] for f in args.infiles]
    if len(set(stems)) != len(stems):
        p.error("input files must have distinct names: outputs are written as OUTDIR/<name>.wav")
    model, conditioner, dev = _load_for_synthesis(args.ckpt)
    from .base import pad_batch
    from .datasets import wav_info
    os.makedirs(args.outdir, exist_ok=True)
    hop = model._hop_length
    conds, rates = [], []
    with torch.no_grad():
        for f in args.infiles:
            rates.append(wav_info(f).sample_rate)
            conds.append(conditioner(wav_read(f).mean(0, keepdim=True).to(dev))[0])
        order = sorted(range(len(conds)), key=lambda i: conds[i].shape[-1])
        denoiser = None
        if args.denoiser_strength > 0:
            denoiser = _denoiser(model, conds[order[0]].shape[-1] * hop, p)
        total, cost = 0, 0.0
        for s0 in range(0, len(order), args.max_batch):
            idx = order[s0:s0 + args.max_batch]
            h, frames = pad_batch([conds[i] for i in idx])
            z = torch.zeros((len(idx), h.shape[-1] * hop))
            for j, i in enumerate(idx):
                z[j, :frames[j] * hop] = item_noise(args.seed, i, frames[j] * hop, args.sigma)
            z = z.to(dev)
            x, dt = _timed(lambda: model.infer(h, args.sigma, z=z, lengths=frames))
            cost += dt
            if denoiser is not None:
                x = denoiser(x, args.denoiser_strength, lengths=[f * hop for f in frames])
            for j, i in enumerate(idx):
                n = frames[j] * hop
                total += n
                wav_write(os.path.join(args.outdir, stems[i] + ".wav"), x[j, :n].reshape(1, -1).cpu(), rates[i])
    print("{} files, {} samples, synthesis {:.4f} s, {:.4f} kHz".format(len(conds), total, cost, total / max(cost, 1e-9) / 1e3))


def main(argv=None) -> None:
    argv = list(sys.argv[1:] if argv is None else argv)
    verbs = {"train": train, "synth": synth, "synth-batch": synth_batch}
    if not argv or argv[0] not in verbs:
        raise SystemExit("usage: python -m constant_memory_waveglow_b200.cli {train,synth,synth-batch} [flags]  "
                         "(-h after the verb)")
    verbs[argv[0]](argv[1:])


if __name__ == "__main__":
    main()
