"""Command line of the harness: ``python -m constant_memory_waveglow_b200.cli {train,synth,synth-batch,vocode,score} ...``.

The reference's own ``train.py`` runs unchanged on the ``pytorch_lightning`` / ``model`` / ``datasets`` shims at the
repository root; its ``inference.py`` cannot in this image (``torchaudio.load`` / ``save`` need the absent TorchCodec),
so the two entry points exist here with the reference's flags (``train.py:81-93``, ``inference.py:62-70``) on top of the
RIFF reader/writer of ``datasets.py``.  Multi-GPU: launch ``train`` under ``torchrun --nproc-per-node N``.  ``synth-batch``
re-synthesises many files, batching utterances of different lengths into one call each (``WaveGlow.infer(lengths=...)``).
``-d/--denoiser-strength`` on ``synth`` and ``synth-batch`` runs the bias-spectrum ``Denoiser`` on the output (one call per
batch, with the per-item lengths); at 0, the default, it is skipped.  ``vocode`` synthesises mel spectrogram files (.pt /
.npy, as NVIDIA's ``inference.py`` reads them) with an NVIDIA WaveGlow checkpoint or this package's, batched the same way;
given ``.wav`` files it computes their mels first (Tacotron2's ``TacotronSTFT`` for NVIDIA checkpoints, the checkpoint's
conditioner otherwise): copy synthesis.  ``score`` prints the per-file negative log-likelihood of WAV files under a
checkpoint, in the convention of the training loss (``WaveGlowLoss``).
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


def _read_mel(path: str, n_mels: int, p: argparse.ArgumentParser) -> torch.Tensor:
    """A mel spectrogram file as NVIDIA's inference.py reads them: .pt (a tensor) or .npy, (n_mels, frames) or
    (1, n_mels, frames)."""
    if path.endswith(".npy"):
        import numpy as np
        m = torch.from_numpy(np.load(path, allow_pickle=False))
    elif path.endswith(".pt"):
        m = torch.load(path, map_location="cpu", weights_only=True)
    else:
        p.error(f"{path}: mel files must be .pt or .npy")
    if not isinstance(m, torch.Tensor) or m.dim() not in (2, 3) or (m.dim() == 3 and m.shape[0] != 1) \
            or not m.is_floating_point():
        p.error(f"{path}: expected a floating-point mel of shape (n_mels, frames) or (1, n_mels, frames), got "
                f"{tuple(m.shape) if isinstance(m, torch.Tensor) else type(m).__name__}")
    m = m.reshape(m.shape[-2], m.shape[-1])
    if m.shape[0] != n_mels or m.shape[1] < 1:
        p.error(f"{path}: mel of shape {tuple(m.shape)} does not fit the model ({n_mels} mel channels, >= 1 frame)")
    return m.float()


def _load_vocoder(ckpt: str, p: argparse.ArgumentParser):
    """(model on the CPU, default sampling rate) of an NVIDIA WaveGlow checkpoint or of this package's Lightning
    checkpoint, told apart by their contents (read with weights_only=True first either way)."""
    model, sr, _ = _load_vocoder_frontend(ckpt, p)
    return model, sr


def _load_vocoder_frontend(ckpt: str, p: argparse.ArgumentParser):
    """(model, default sampling rate, mel front end), on the CPU.  The front end maps audio to the model's mels:
    Tacotron2's TacotronSTFT for an NVIDIA checkpoint, the checkpoint's conditioner for this package's."""
    from . import nvidia
    from .condition import TacotronSTFT
    try:
        obj = nvidia._read_checkpoint(ckpt)
    except Exception as e:
        p.error(f"{ckpt}: not a checkpoint this command reads ({e})")
    if isinstance(obj, dict) and "hyper_parameters" in obj and isinstance(obj.get("state_dict"), dict) \
            and any(k.startswith("model.") for k in obj["state_dict"]):
        lit = TR.LightModel.load_from_checkpoint(ckpt, map_location="cpu")
        lit.model.apply(remove_weight_norms)
        return lit.model, int(lit.conditioner.sample_rate), lit.conditioner
    model = nvidia.load_nvidia_waveglow(obj, device="cpu")
    return model, 22050, TacotronSTFT(n_mel_channels=model.n_mels, sampling_rate=22050)


def _frontend_rate(frontend) -> int:
    return int(getattr(frontend, "sampling_rate", None) or frontend.sample_rate)


def _read_wav_mono(path: str, rate: int, p: argparse.ArgumentParser) -> torch.Tensor:
    """A WAV file as one channel (the mean of its channels); its sampling rate must be `rate` (there is no resampler)."""
    from .datasets import wav_info
    sr = wav_info(path).sample_rate
    if sr != rate:
        p.error(f"{path}: sampled at {sr} Hz; the model's mel front end expects {rate} Hz (resample it first)")
    return wav_read(path).mean(0)


def _frontend_mels(frontend, signals, names, max_batch: int, dev, p: argparse.ArgumentParser):
    """Mels of 1-D signals (on the CPU), one front-end call per length-sorted group of `max_batch` with per-item
    lengths; item i gets signals[i].numel() // hop + 1 frames.  Returns CPU tensors (n_mels, frames) in input order."""
    from .base import pad_batch
    from .condition import MelSpec, TacotronSTFT
    batched = isinstance(frontend, (MelSpec, TacotronSTFT))
    step = max_batch if batched else 1
    order = sorted(range(len(signals)), key=lambda i: signals[i].numel())
    hop = frontend.hop_length
    out = [None] * len(signals)
    for s0 in range(0, len(order), step):
        idx = order[s0:s0 + step]
        x, lens = pad_batch([signals[i] for i in idx])
        try:
            m = frontend(x.to(dev), lengths=lens) if batched else frontend(x.to(dev))
        except ValueError as e:
            p.error(f"{', '.join(names[i] for i in idx)}: {e}")
        for j, i in enumerate(idx):
            out[i] = m[j, :, :lens[j] // hop + 1].cpu()
    return out


def vocode(argv) -> None:
    p = argparse.ArgumentParser(prog="cli vocode", description="synthesis from mel spectrograms (.pt / .npy) or from the "
                                "mels of WAV files (copy synthesis), batched by length; NVIDIA WaveGlow or this package's "
                                "checkpoints")
    p.add_argument("ckpt", type=str)
    p.add_argument("outdir", type=str)
    p.add_argument("mels", type=str, nargs="+", help=".pt / .npy mel spectrograms or .wav files (at the front end's rate)")
    p.add_argument("-s", "--sigma", type=float, default=0.6)
    p.add_argument("--max-batch", type=int, default=16, help="utterances per synthesis call")
    p.add_argument("--seed", type=int, default=0, help="noise seed; file i draws from a generator seeded by (seed, i)")
    p.add_argument("--sampling-rate", type=int, default=None,
                   help="of the written WAVs (default: 22050 for NVIDIA checkpoints, else the conditioner's)")
    _add_denoiser_arg(p)
    args = p.parse_args(argv)
    _check_denoiser_arg(p, args)
    if args.max_batch < 1:
        p.error("--max-batch must be >= 1")
    if args.sampling_rate is not None and args.sampling_rate < 1:
        p.error("--sampling-rate must be >= 1")
    stems = [os.path.splitext(os.path.basename(f))[0] for f in args.mels]
    if len(set(stems)) != len(stems):
        p.error("mel files must have distinct names: outputs are written as OUTDIR/<name>.wav")
    model, sr, frontend = _load_vocoder_frontend(args.ckpt, p)
    sr = args.sampling_rate or sr
    is_wav = [f.lower().endswith(".wav") for f in args.mels]
    mels = [None if w else _read_mel(f, model.n_mels, p) for f, w in zip(args.mels, is_wav)]
    wav_idx = [i for i, w in enumerate(is_wav) if w]
    signals = [_read_wav_mono(args.mels[i], _frontend_rate(frontend), p) for i in wav_idx]
    from .base import pad_batch
    dev = torch.device("cuda")
    model = model.to(dev).eval()
    hop = model._hop_length
    # WAV inputs: mels from the front end, one call per batch with the per-item lengths; the output keeps each file's
    # sample count (the model gives frames * hop >= samples + 1)
    n_out = {}
    if wav_idx:
        with torch.no_grad():
            wav_mels = _frontend_mels(frontend.to(dev), signals, [args.mels[i] for i in wav_idx], args.max_batch, dev, p)
        for i, m, x in zip(wav_idx, wav_mels, signals):
            mels[i], n_out[i] = m, x.numel()
    os.makedirs(args.outdir, exist_ok=True)
    order = sorted(range(len(mels)), key=lambda i: mels[i].shape[-1])
    # families without per-item lengths (WaveFlow, WSRGlow, ...) synthesise one utterance per call
    max_batch = args.max_batch if model._supports_lengths else 1
    with torch.no_grad():
        denoiser = _denoiser(model, mels[order[0]].shape[-1] * hop, p) if args.denoiser_strength > 0 else None
        total, cost = 0, 0.0
        for s0 in range(0, len(order), max_batch):
            idx = order[s0:s0 + max_batch]
            h, frames = pad_batch([mels[i] for i in idx])
            z = torch.zeros((len(idx), h.shape[-1] * hop))
            for j, i in enumerate(idx):
                z[j, :frames[j] * hop] = item_noise(args.seed, i, frames[j] * hop, args.sigma)
            h, z = h.to(dev), z.to(dev)
            lengths = frames if model._supports_lengths else None
            x, dt = _timed(lambda: model.infer(h, args.sigma, z=z, lengths=lengths).reshape(len(idx), -1))
            cost += dt
            if denoiser is not None:
                x = denoiser(x, args.denoiser_strength, lengths=[f * hop for f in frames] if lengths else None)
            for j, i in enumerate(idx):
                n = n_out.get(i, frames[j] * hop)
                total += n
                wav_write(os.path.join(args.outdir, stems[i] + ".wav"), x[j, :n].reshape(1, -1).cpu(), sr)
    print("{} files, {} samples, synthesis {:.4f} s, {:.4f} kHz".format(len(mels), total, cost, total / max(cost, 1e-9) / 1e3))


def score(argv) -> None:
    p = argparse.ArgumentParser(prog="cli score", description="per-file negative log-likelihood of WAV files under an NVIDIA "
                                "WaveGlow or a package checkpoint, per sample as the training loss (WaveGlowLoss) gives it")
    p.add_argument("ckpt", type=str)
    p.add_argument("wavs", type=str, nargs="+")
    p.add_argument("-s", "--sigma", type=float, default=1.0, help="of the loss (NVIDIA trains with 1.0)")
    p.add_argument("--max-batch", type=int, default=16, help="files per forward call")
    args = p.parse_args(argv)
    if args.max_batch < 1:
        p.error("--max-batch must be >= 1")
    if not 0 < args.sigma < math.inf:
        p.error("--sigma must be a finite number > 0")
    for path, n, nll in score_files(args.ckpt, args.wavs, args.sigma, args.max_batch, p):
        print(f"{path}\t{n}\t{nll:.6f}")


def score_files(ckpt: str, paths, sigma: float, max_batch: int, p: argparse.ArgumentParser):
    """[(path, samples, NLL)] in input order.  Each file, cut to a multiple of n_group, gets WaveGlowLoss(sigma) of its own
    forward call: 0.5 sum z^2 / sigma^2 - log-det, over its samples.  Files run in length-sorted batches through
    forward(x, mel, lengths=...), which gives every item its own call's z and log-det bit for bit; families without
    per-item lengths run one file per call."""
    from .base import pad_batch
    from .loss import WaveGlowLoss
    from .nvidia import NvidiaWaveGlow
    model, _, frontend = _load_vocoder_frontend(ckpt, p)
    g, hop = getattr(model, "n_group", 1), model._hop_length
    signals = []
    for f in paths:
        x = _read_wav_mono(f, _frontend_rate(frontend), p)
        signals.append(x[:x.numel() - x.numel() % g])
    dev = torch.device("cuda")
    model, frontend = model.to(dev).eval(), frontend.to(dev)
    with torch.no_grad():
        mels = _frontend_mels(frontend, signals, list(paths), max_batch, dev, p)
    # The batched path conditions item b on its first ceil(n_b / hop) mel frames (the frames infer() synthesises from).
    # The front end gives n / hop + 1 frames, one more when hop divides n, and this package's upsampler reaches back from
    # that frame into the item's last samples; such files run alone.  NVIDIA's upsampler only reaches forward.
    alone = [not model._supports_lengths or (x.numel() % hop == 0 and not isinstance(model, NvidiaWaveGlow)) for x in signals]
    order = sorted((i for i in range(len(paths)) if not alone[i]), key=lambda i: signals[i].numel())
    groups = [order[s0:s0 + max_batch] for s0 in range(0, len(order), max_batch)] + [[i] for i in range(len(paths)) if alone[i]]
    loss = WaveGlowLoss(sigma)
    nll = [None] * len(paths)
    with torch.no_grad():
        for idx in groups:
            x, lens = pad_batch([signals[i] for i in idx])
            h, _ = pad_batch([mels[i] for i in idx])
            x, h = x.to(dev), h.to(dev)
            if len(idx) == 1:
                z, logdet = model(x, h)
            else:
                z, logdet = model(x, h, lengths=lens)
            z = z.reshape(len(idx), -1)
            logdet = logdet.reshape(len(idx))
            for j, i in enumerate(idx):
                nll[i] = float(loss(z[j:j + 1, :lens[j]].clone(), logdet[j:j + 1].clone()))
    return [(f, signals[i].numel(), nll[i]) for i, f in enumerate(paths)]


def main(argv=None) -> None:
    argv = list(sys.argv[1:] if argv is None else argv)
    verbs = {"train": train, "synth": synth, "synth-batch": synth_batch, "vocode": vocode, "score": score}
    if not argv or argv[0] not in verbs:
        raise SystemExit("usage: python -m constant_memory_waveglow_b200.cli {train,synth,synth-batch,vocode,score} [flags]  "
                         "(-h after the verb)")
    verbs[argv[0]](argv[1:])


if __name__ == "__main__":
    main()
