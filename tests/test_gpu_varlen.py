"""Variable-length batched inference: every item of a padded batch with per-item lengths against the same item run alone.

Contract (WaveGlow.forward / reverse / infer with `lengths`, cmwg_wn_forward_varlen): on its valid samples an item gets
bit for bit what the call on that item alone gives (fp32 and fp16 operands), exact zeros after them, and a log-det over its
valid samples.  The log-det is bit-identical too: cmwg_logdet_accumulate_varlen sums an item's valid block in the order the
item-alone reduction uses.  bf16 is checked bitwise at the WN level (its model level is the same code path as fp16)."""
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import precision
from constant_memory_waveglow_b200.base import pad_batch
from tests._util import TOL, rel_l2

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(autouse=True)
def _restore_precision():
    old = precision.get_precision()
    yield
    precision.set_precision(old)
    os.environ.pop("CMWG_MEGA", None)


def _wn(bias, seed=0):
    torch.manual_seed(seed)
    wn = cm.WN(4, 80, 256, 256, 256, depth=8, radix=3, bias=bias, zero_init=False).cuda()
    if bias:
        with torch.no_grad():
            for m in wn.modules():
                if isinstance(m, torch.nn.Conv1d) and m.bias is not None:
                    m.bias.normal_(std=0.1)
    return wn


# rows of the WN (squeezed time steps): len == T, an item ending on a full tile (512 = 2 x 256), an item shorter than
# one tile, an item of one row (n_group samples), an item ending inside its third tile
KERNEL_T = 1300
KERNEL_LENS = [1300, 512, 100, 1, 700]


@pytest.mark.parametrize("prec,mega,bias", [("fp32", "1", False), ("fp32", "1", True), ("fp16", "1", False),
                                            ("fp16", "0", False), ("fp16", "1", True), ("bf16", "1", False),
                                            ("bf16", "0", True)])
def test_wn_forward_varlen_matches_each_item_alone(prec, mega, bias):
    os.environ["CMWG_MEGA"] = mega
    wn = _wn(bias)
    B, T = len(KERNEL_LENS), KERNEL_T
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, 8, T, generator=g).cuda()
    y = torch.randn(B, 80, T, generator=g).cuda()
    with torch.no_grad():
        # an ordinary full-length call first: the per-stream scratch slabs then hold non-zero data from it
        full, _ = wn._cmwg_forward(torch.randn(B, 8, T, generator=g).cuda(), y, save=False, prec=prec)
        assert full.abs().sum() > 0
        lens_dev = torch.tensor(KERNEL_LENS, dtype=torch.int32).cuda()
        lst = wn._cmwg_forward_varlen(x, y, (C.c_int * B)(*KERNEL_LENS), lens_dev, prec)
        for b, n in enumerate(KERNEL_LENS):
            solo, _ = wn._cmwg_forward(x[b:b + 1, :, :n].contiguous(), y[b:b + 1, :, :n].contiguous(), save=False, prec=prec)
            assert torch.equal(lst[b, :, :n], solo[0]), (prec, mega, bias, b, n, (lst[b, :, :n] - solo[0]).abs().max().item())


def test_wn_forward_varlen_rejects_bad_lengths():
    wn = _wn(False)
    x, y = torch.zeros(2, 8, 300).cuda(), torch.zeros(2, 80, 300).cuda()
    for bad in ([0, 300], [301, 10]):
        with pytest.raises(RuntimeError, match="outside"):
            wn._cmwg_forward_varlen(x, y, (C.c_int * 2)(*bad), torch.tensor(bad, dtype=torch.int32).cuda(), "fp16")


def _model(cfg, efficient=True, reverse_mode=False, seed=0):
    torch.manual_seed(seed)
    if cfg == "lj":
        m = cm.WaveGlow(12, 8, 4, 2, 256, 80, efficient, reverse_mode=reverse_mode, zero_init=False)
    else:
        m = cm.WaveGlow(12, 8, 4, 2, 256, 80, efficient, reverse_mode=reverse_mode, zero_init=False,
                        dilation_channels=128, residual_channels=128, skip_channels=128)
    m.apply(cm.remove_weight_norms)
    return m.cuda().eval()


# samples: len == T, a full-tile item (4096 = 512 rows), a one-tile item, one n_group, an item ending mid-frame
SAMPLES_T = 5120
SAMPLE_LENS = [5120, 4096, 800, 8, 2056]


def _inputs(seed=1):
    g = torch.Generator().manual_seed(seed)
    B, T = len(SAMPLE_LENS), SAMPLES_T
    x = (torch.rand(B, T, generator=g) * 2 - 1).cuda() * 0.5
    h = torch.randn(B, 80, T // 256, generator=g).cuda()
    return x, h


def _check_item(out, solo, n, prec, what):
    assert torch.equal(out[:n], solo), (what, prec, n, (out[:n] - solo).abs().max().item())
    assert (out[n:] == 0).all(), (what, "tail not zero")


def _check_logdet(ld, solo_ld, prec, what):
    assert torch.equal(ld, solo_ld), (what, prec, ld.item(), solo_ld.item())


@pytest.mark.parametrize("prec", ["fp32", "fp16"])
@pytest.mark.parametrize("cfg,efficient,reverse_mode", [("lj", True, False), ("lj", False, False), ("small", True, False),
                                                        ("small", False, True)])
def test_model_varlen_matches_solo_calls(prec, cfg, efficient, reverse_mode):
    precision.set_precision(prec)
    m = _model(cfg, efficient, reverse_mode)
    x, h = _inputs()
    lens = SAMPLE_LENS
    with torch.no_grad():
        z, ld = m.forward(x, h, lengths=lens)
        xr, ldr = m.reverse(z, h, lengths=torch.tensor(lens))
        for b, n in enumerate(lens):
            f = -(-n // 256)
            zs, lds = m.forward(x[b:b + 1, :n].clone(), h[b:b + 1, :, :f].clone())
            _check_item(z[b], zs[0], n, prec, "forward z")
            _check_logdet(ld[b], lds[0], prec, "forward logdet")
            xs, ldrs = m.reverse(z[b:b + 1, :n].clone(), h[b:b + 1, :, :f].clone())
            _check_item(xr[b], xs[0], n, prec, "reverse x")
            _check_logdet(ldr[b], ldrs[0], prec, "reverse logdet")
            assert rel_l2(xr[b, :n], x[b, :n]) < max(TOL[prec]["roundtrip"], 5e-6), ("round trip", b)


@pytest.mark.parametrize("prec", ["fp32", "fp16"])
def test_infer_varlen_matches_solo_infer(prec):
    precision.set_precision(prec)
    m = _model("lj")
    frames = [20, 16, 1, 7]
    g = torch.Generator().manual_seed(2)
    hs = [torch.randn(80, f, generator=g).cuda() for f in frames]
    h, fl = pad_batch(hs)
    assert fl == frames and h.shape == (4, 80, 20)
    z = torch.randn(4, 20 * 256, generator=g).cuda() * 0.6
    audio = m.infer(h, 0.6, z=z, lengths=frames)
    assert audio.shape == (4, 20 * 256)
    for b, f in enumerate(frames):
        solo = m.infer(hs[b][None], 0.6, z=z[b:b + 1, :f * 256].clone())
        _check_item(audio[b], solo.reshape(-1), f * 256, prec, "infer")


@pytest.mark.parametrize("prec", ["fp32", "fp16"])
def test_all_lengths_equal_T_change_nothing(prec):
    precision.set_precision(prec)
    m = _model("lj")
    x, h = _inputs(3)
    full = [SAMPLES_T] * x.shape[0]
    with torch.no_grad():
        z0, ld0 = m(x, h)
        z1, ld1 = m(x, h, lengths=full)
        x0, _ = m.reverse(z0, h)
        x1, _ = m.reverse(z0, h, lengths=full)
    assert torch.equal(z0, z1) and torch.equal(ld0, ld1) and torch.equal(x0, x1)


def test_lengths_need_no_grad():
    m = _model("small")
    x, h = _inputs()
    with pytest.raises(NotImplementedError, match="inference only"):
        m(x, h, lengths=SAMPLE_LENS)


def _tiny_checkpoint(tmp_path):
    from constant_memory_waveglow_b200 import datasets as D, trainer as TR
    cfg = {
        "name": "tiny",
        "arch": {"type": "WaveGlow", "args": dict(flows=4, n_group=8, n_early_every=2, n_early_size=2, hop_size=256,
                                                  n_mels=80, memory_efficient=True, reverse_mode=False,
                                                  dilation_channels=64, residual_channels=64, skip_channels=64, depth=2,
                                                  radix=3, bias=False)},
        "dataset": {"type": "RandomWAVDataset", "args": {"data_dir": str(tmp_path), "size": 4, "segment": 4096}},
        "data_loader": {"batch_size": 2, "shuffle": False, "num_workers": 0, "pin_memory": False},
        "optimizer": {"type": "Adam", "args": {"lr": 1e-3, "weight_decay": 0}},
        "loss": {"type": "WaveGlowLoss", "args": {"sigma": 0.7, "elementwise_mean": True}},
        "conditioner": {"type": "MelSpec", "args": {"sr": 22050, "n_fft": 1024, "hop_length": 256, "f_max": 8000,
                                                    "n_mels": 80}},
    }
    torch.manual_seed(4)
    wavs = []
    for i, n in enumerate([9000, 3000, 20000]):
        t = torch.arange(n) / 22050.0
        p = tmp_path / f"in{i}.wav"
        D.wav_write(p, 0.3 * torch.sin(2 * torch.pi * 200.0 * (i + 1) * t), 22050)
        wavs.append(str(p))
    lm = TR.LightModel(cfg)
    with torch.no_grad():
        for wn in lm.model.WNs:
            wn.F.end.weight.normal_(std=0.02)   # zero-initialised `end` convs would make every flow the identity
    path = tmp_path / "tiny.ckpt"
    torch.save(lm.checkpoint(epoch=0, global_step=0, optimizers=[lm.configure_optimizers()]), path)
    return str(path), wavs


def test_cli_synth_batch_matches_solo_inference(tmp_path):
    from constant_memory_waveglow_b200 import cli, datasets as D
    ckpt, wavs = _tiny_checkpoint(tmp_path)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, "-m", "constant_memory_waveglow_b200.cli", "synth-batch", ckpt, str(out), *wavs,
                        "-s", "0", "--max-batch", "2"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    model, conditioner, dev = cli._load_for_synthesis(ckpt)
    for f in wavs:
        cond = conditioner(D.wav_read(f).mean(0, keepdim=True).to(dev))
        want = model.infer(cond, 0.0).reshape(1, -1)
        info = D.wav_info(out / os.path.basename(f))
        assert info.sample_rate == 22050 and info.num_frames == cond.shape[-1] * 256
        got = D.wav_read(out / os.path.basename(f))
        # both through the 16-bit PCM writer: same samples
        ref_path = tmp_path / "ref.wav"
        D.wav_write(ref_path, want.cpu(), 22050)
        assert torch.equal(got, D.wav_read(ref_path)), f
