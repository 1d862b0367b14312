"""Data path (SURVEY §8 f3) and Lightning-free harness (f2): CPU tests of the host logic; one GPU test that trains."""
import argparse
import json
import os
import struct
import wave

import numpy as np
import pytest
import torch

from tests._util import load_golden

from constant_memory_waveglow_b200 import datasets as D
from constant_memory_waveglow_b200 import trainer as TR


def _write_fixture_files(root, fx):
    for (name, frames, ch), data in zip(fx["files"], fx["pcm"]):
        path = os.path.join(root, name)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with wave.open(path, "wb") as w:
            w.setnchannels(ch); w.setsampwidth(2); w.setframerate(22050)
            w.writeframes(data.numpy().astype("<i2").tobytes())


def test_random_wav_dataset_matches_reference_fixture(tmp_path):
    """File choice, frame offset and returned segment of every index equal what the reference class produced
    (tests/golden/make_golden_data.py), bit for bit."""
    fx = load_golden("random_wav.pt")
    _write_fixture_files(str(tmp_path), fx)
    for size, case in fx["cases"].items():
        ds = D.RandomWAVDataset(str(tmp_path), size, fx["segment"])
        assert len(ds) == size and ds.sr == case["sr"]
        assert np.array_equal(ds.boundaries, case["boundaries"].numpy())
        for i in range(size):
            k, off = ds.locate(i / size)
            assert os.path.relpath(str(ds.files[k]), str(tmp_path)) == case["files"][i]
            assert off == case["offsets"][i]
        if case["segments_x65536"] is not None:
            got = torch.stack([ds[i] for i in range(size)])
            assert got.shape == (size, fx["segment"]) and got.dtype == torch.float32
            assert torch.equal((got.double() * 65536).round().int(), case["segments_x65536"])


@pytest.mark.parametrize("bits,fmt", [(8, 1), (16, 1), (24, 1), (32, 1), (32, 3), (64, 3)])
def test_wav_reader_encodings(tmp_path, bits, fmt):
    """Every sample encoding of the container decodes to the value it encodes; extensible headers and odd chunks too."""
    rng = np.random.default_rng(bits + fmt)
    n, ch = 257, 2
    x = rng.uniform(-0.9, 0.9, size=(n, ch))
    if fmt == 3:
        arr = x.astype("<f4" if bits == 32 else "<f8"); want = arr.astype(np.float32); raw = arr.tobytes()
    elif bits == 8:
        q = np.round(x * 128 + 128).clip(0, 255).astype(np.uint8); want = (q.astype(np.float32) - 128) / 128; raw = q.tobytes()
    elif bits == 16:
        q = np.round(x * 32768).astype("<i2"); want = q.astype(np.float32) / 32768; raw = q.tobytes()
    elif bits == 24:
        q = np.round(x * 8388608).astype(np.int32); want = q.astype(np.float32) / 8388608
        raw = b"".join(struct.pack("<i", int(v))[:3] for v in q.reshape(-1))
    else:
        q = np.round(x * 2147483648).astype(np.int64).clip(-2 ** 31, 2 ** 31 - 1).astype("<i4")
        want = (q.astype(np.float64) / 2147483648).astype(np.float32); raw = q.tobytes()
    # WAVE_FORMAT_EXTENSIBLE header with a LIST chunk of odd length in front of the data
    ext = struct.pack("<HHIIHH", 0xFFFE, ch, 16000, 16000 * ch * bits // 8, ch * bits // 8, bits) + \
        struct.pack("<HHI", 22, bits, 3) + struct.pack("<H", fmt) + b"\x00" * 14
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(ext)) + ext + b"LIST" + struct.pack("<I", 5) + b"abcde\x00" + \
        b"data" + struct.pack("<I", len(raw)) + raw
    path = tmp_path / "x.wav"
    path.write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)
    info = D.wav_info(path)
    assert (info.sample_rate, info.num_frames, info.num_channels, info.bits_per_sample, info.fmt) == (16000, n, ch, bits, fmt)
    assert np.array_equal(D.wav_read(path).numpy(), want.T)
    assert np.array_equal(D.wav_read(path, 100, 50).numpy(), want.T[:, 100:150])
    assert D.wav_read(path, 250, 50).shape == (ch, 7)       # clipped at the end of the file
    assert D.wav_read(path, 999, 50).shape == (ch, 0)


def test_wav_write_round_trip_and_errors(tmp_path):
    x = torch.linspace(-1, 1, 1001)
    D.wav_write(tmp_path / "o.wav", x, 22050)
    y = D.wav_read(tmp_path / "o.wav")
    assert y.shape == (1, 1001) and (y[0] - x).abs().max() <= 1 / 32768
    (tmp_path / "bad.wav").write_bytes(b"not a wave file at all")
    with pytest.raises(ValueError):
        D.wav_info(tmp_path / "bad.wav")
    with pytest.raises(FileNotFoundError):
        D.RandomWAVDataset(str(tmp_path / "empty"), 4, 100)


def test_prefetcher_preserves_order_on_cpu():
    batches = [torch.full((3, 5), float(i)) for i in range(7)]
    out = list(D.DevicePrefetcher(batches, torch.device("cpu")))
    assert len(out) == 7 and all(torch.equal(a, b) for a, b in zip(out, batches))
    assert list(D.DevicePrefetcher([], torch.device("cpu"))) == []


TINY = {
    "name": "tiny",
    "arch": {"type": "WaveGlow", "args": dict(flows=4, n_group=8, n_early_every=2, n_early_size=2, hop_size=256, n_mels=80,
                                              memory_efficient=True, reverse_mode=False, dilation_channels=64,
                                              residual_channels=64, skip_channels=64, depth=2, radix=3, bias=False)},
    "dataset": {"type": "RandomWAVDataset", "args": {"data_dir": None, "size": 16, "segment": 4096}},
    "data_loader": {"batch_size": 4, "shuffle": True, "num_workers": 0, "pin_memory": False},
    "optimizer": {"type": "Adam", "args": {"lr": 1e-3, "weight_decay": 0}},
    "loss": {"type": "WaveGlowLoss", "args": {"sigma": 0.7, "elementwise_mean": True}},
    "conditioner": {"type": "MelSpec", "args": {"sr": 22050, "n_fft": 1024, "hop_length": 256, "f_max": 8000, "n_mels": 80}},
}


def _tiny_config(tmp_path):
    cfg = json.loads(json.dumps(TINY))
    root = tmp_path / "wavs"
    root.mkdir()
    g = torch.Generator().manual_seed(3)
    for i in range(3):
        t = torch.arange(20000) / 22050.0
        x = 0.3 * torch.sin(2 * np.pi * (220.0 * (i + 1)) * t) + 0.05 * torch.randn(20000, generator=g)
        D.wav_write(root / f"f{i}.wav", x, 22050)
    cfg["dataset"]["args"]["data_dir"] = str(root)
    return cfg


def test_lightmodel_surface_and_checkpoint_layout(tmp_path):
    """Reference model/lightning.py:16-68: hparams, reflection-built members, Lightning's checkpoint dictionary."""
    cfg = _tiny_config(tmp_path)
    lm = TR.LightModel(cfg)
    assert lm.hparams.arch["type"] == "WaveGlow" and set(lm.hparams) >= {"arch", "dataset", "data_loader", "optimizer", "loss", "conditioner"}
    assert type(lm.model).__name__ == "WaveGlow" and type(lm.conditioner).__name__ == "MelSpec" and type(lm.criterion).__name__ == "WaveGlowLoss"
    opt = lm.configure_optimizers()
    assert isinstance(opt, torch.optim.Adam) and opt.param_groups[0]["lr"] == 1e-3
    assert len(lm.train_dataloader().dataset) == 16
    path = tmp_path / "m.ckpt"
    torch.save(lm.checkpoint(epoch=2, global_step=9, optimizers=[opt]), path)
    ck = torch.load(path, weights_only=False)
    assert set(ck) >= {"state_dict", "hyper_parameters", "optimizer_states", "epoch", "global_step"}
    assert any(k.startswith("model.WNs.0.F.layers.0.W.weight_g") for k in ck["state_dict"])
    assert any(k.startswith("model.invconv1x1.0.weight") for k in ck["state_dict"])
    lm2 = TR.LightModel.load_from_checkpoint(path, map_location="cpu")          # inference.py:15
    assert all(torch.equal(a, b) for a, b in zip(lm.state_dict().values(), lm2.state_dict().values()))
    lm3 = TR.LightModel.load_from_checkpoint(path, config=cfg)                   # train.py:66-69
    assert lm3.hparams.loss["args"]["sigma"] == 0.7


def test_shim_import_names():
    """The import lines of train.py:8-10,14, inference.py:10 and model/lightning.py:5-13 resolve."""
    import pytorch_lightning as pl
    from pytorch_lightning.callbacks import DeviceStatsMonitor, LearningRateMonitor, ModelSummary  # noqa: F401
    from pytorch_lightning.plugins import DDPPlugin
    import datasets as module_data
    from model import LightModel, condition  # noqa: F401
    import model.loss as module_loss
    assert issubclass(LightModel, pl.LightningModule) and hasattr(pl, "seed_everything") and hasattr(pl, "Callback")
    assert hasattr(module_data, "RandomWAVDataset") and hasattr(module_loss, "WaveGlowLoss") and hasattr(condition, "MelSpec")
    DDPPlugin(find_unused_parameters=False)
    p = pl.Trainer.add_argparse_args(LightModel.add_model_specific_args(argparse.ArgumentParser()))
    a = p.parse_args(["--max_steps", "3", "--default_root_dir", "/tmp/x"])
    assert a.max_steps == 3 and a.default_root_dir == "/tmp/x"
    assert pl.seed_everything(5) == 5 and torch.initial_seed() == 5


@pytest.mark.gpu
def test_trainer_fits_and_checkpoint_synthesises(tmp_path):
    """End to end on the device: wave files -> RandomWAVDataset -> prefetcher -> MelSpec -> constant-memory
    WaveGlow step -> Adam, loss goes down; the checkpoint reloads and synthesises finite audio (inference.py:14-52)."""
    cfg = _tiny_config(tmp_path)
    TR.seed_everything(0)
    lm = TR.LightModel(cfg)
    with torch.no_grad():                       # the shipped init zeroes `end` (waveglow.py:93-96); give F something to learn from
        for wn in lm.model.WNs:
            wn.F.end.weight.normal_(0, 0.01)
    tr = TR.Trainer(max_epochs=6, default_root_dir=str(tmp_path / "run"), log_every_n_steps=1, detect_anomaly=True,
                    callbacks=[TR.ModelSummary(max_depth=2), TR.LearningRateMonitor("epoch")])
    tr.fit(lm)
    assert tr.global_step == 24 and tr.current_epoch == 6
    import csv
    rows = list(csv.DictReader(open(os.path.join(tr.logger.log_dir, "metrics.csv"))))
    losses = [float(r["loss"]) for r in rows]
    assert len(losses) == 24 and all(np.isfinite(losses))
    assert np.mean(losses[-4:]) < np.mean(losses[:4])
    assert tr.last_checkpoint and os.path.exists(tr.last_checkpoint)

    from constant_memory_waveglow_b200.utils import remove_weight_norms
    lm2 = TR.LightModel.load_from_checkpoint(tr.last_checkpoint, map_location="cpu")
    model = lm2.model
    model.apply(remove_weight_norms)
    model, cond_fn = model.cuda().eval(), lm2.conditioner.cuda()
    y = D.wav_read(os.path.join(cfg["dataset"]["args"]["data_dir"], "f0.wav")).mean(0, keepdim=True).cuda()
    y = y[:, :y.shape[1] - y.shape[1] % 8]
    cond = cond_fn(y)
    with torch.no_grad():
        z, logdet = model(y.clone(), cond)
        x = model.infer(cond, 0.6)
    assert torch.isfinite(z).all() and torch.isfinite(logdet).all() and torch.isfinite(x).all()
    assert x.numel() == cond.shape[-1] * 256

    # resuming continues the step count and the optimizer state
    tr2 = TR.Trainer(max_steps=tr.global_step + 2, default_root_dir=str(tmp_path / "run"), log_every_n_steps=1)
    lm3 = TR.LightModel(cfg)
    tr2.fit(lm3, ckpt_path=tr.last_checkpoint)
    assert tr2.global_step == tr.global_step + 2


@pytest.mark.gpu
def test_cli_train_then_synth(tmp_path, capsys):
    """The two entry points with the reference's flags: train two steps from a config, synthesise from the checkpoint."""
    from constant_memory_waveglow_b200 import cli
    cfg = _tiny_config(tmp_path)
    (tmp_path / "cfg.json").write_text(json.dumps(cfg))
    cli.main(["train", "--config", str(tmp_path / "cfg.json"), "--max_epochs", "1", "--seed", "3", "--lr", "5e-4",
              "--log_every_n_steps", "1", "--default_root_dir", str(tmp_path / "run")])
    ckpts = sorted((tmp_path / "run" / "lightning_logs" / "version_0" / "checkpoints").glob("*.ckpt"))
    assert len(ckpts) == 1
    ck = torch.load(ckpts[0], weights_only=False)
    assert ck["global_step"] == 4 and ck["optimizer_states"][0]["param_groups"][0]["lr"] == 5e-4
    cli.main(["synth", str(ckpts[0]), os.path.join(cfg["dataset"]["args"]["data_dir"], "f1.wav"), str(tmp_path / "out.wav"),
              "-n", "8", "-s", "0.6"])
    out = capsys.readouterr().out
    assert out.count("kHz") == 2 and "Forward LL:" in out
    info = D.wav_info(tmp_path / "out.wav")
    assert info.sample_rate == 22050 and info.num_frames % 256 == 0 and abs(info.num_frames - 20000) <= 256


def test_cli_usage_errors():
    from constant_memory_waveglow_b200 import cli
    with pytest.raises(SystemExit):
        cli.main([])
    with pytest.raises(SystemExit):
        cli.main(["train"])          # neither --config nor --ckpt-path
