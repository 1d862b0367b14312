"""Denoiser on the device (csrc/denoise.cu) against the fp64 oracle (oracle/denoise_oracle.py), batched items against solo
calls, determinism, the CLI's -d flag, and MelSpec's output after its FFT moved into csrc/fft.cuh."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import _lib, ops
from constant_memory_waveglow_b200.condition import MelSpec
from oracle import denoise_oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
SR = 22050


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _window(n_fft):
    return torch.hann_window(n_fft, periodic=True, dtype=torch.float32)


def _signal(n, seed, noise=0.02):
    """Three sinusoids over white noise: at strength 1 the noise bins clamp and the tones survive."""
    g = np.random.default_rng(seed)
    t = np.arange(n) / SR
    x = sum(0.2 * np.sin(2 * np.pi * f * t + g.uniform(0, 6)) for f in g.uniform(100, 5000, 3))
    return torch.from_numpy((x + noise * g.standard_normal(n)).astype(np.float32))


def _bias(n_fft, seed, noise=0.02):
    """A bias spectrum 1-3 x the expected magnitude of the noise of _signal."""
    g = np.random.default_rng(seed)
    level = noise * np.sqrt(3 * n_fft / 8)                 # sqrt(sum w^2) of the periodic Hann window
    return torch.from_numpy((level * g.uniform(1, 3, n_fft // 2 + 1)).astype(np.float32))


def _padded(lens, T, seed):
    """(B, T) batch: item b's signal on [0, lens[b]), unrelated noise after it (the kernels must not read it)."""
    x = torch.randn(len(lens), T, generator=torch.Generator().manual_seed(seed))
    for b, n in enumerate(lens):
        x[b, :n] = _signal(n, seed + b)
    return x


@pytest.mark.parametrize("n_fft", [512, 1024, 2048])
@pytest.mark.parametrize("strength", [0.0, 0.01, 0.1, 1.0])
def test_denoise_matches_oracle(n_fft, strength):
    hop = n_fft // 4
    lens = [n_fft // 2 + 1, 3 * n_fft + 77, 10 * SR]
    T = max(lens)
    x, w, bias = _padded(lens, T, 11), _window(n_fft), _bias(n_fft, 3)
    out = ops.denoise(x.cuda(), w.cuda(), bias.cuda(), strength, hop, lengths=lens).cpu()
    for b, n in enumerate(lens):
        xi = x[b, :n].double().numpy()
        ref = O.denoise(xi, bias.double().numpy(), strength, n_fft, hop, w.double().numpy())
        assert _rel(out[b, :n], ref) <= 1e-5, (n_fft, strength, n, _rel(out[b, :n], ref))
        assert (out[b, n:] == 0).all()
        if strength == 1.0 and n == 10 * SR:
            mag = np.abs(O.stft(xi, n_fft, hop, w.double().numpy()))
            assert (mag <= bias.double().numpy()[:, None]).mean() > 0.5      # most bins clamp


def test_strength_zero_reconstructs_on_device():
    x = _signal(5 * SR, 2)
    out = ops.denoise(x.cuda(), _window(1024).cuda(), _bias(1024, 1).cuda(), 0.0, 256).cpu()
    assert _rel(out, x) < 1e-6


def test_batch_items_equal_solo_calls():
    n_fft, hop, strength = 1024, 256, 0.1
    lens = [10 * SR, n_fft // 2 + 1, 1000, 77777, 3 * n_fft + 77, 10 * SR - 1]
    T = max(lens)
    w, bias = _window(n_fft).cuda(), _bias(n_fft, 5).cuda()
    x = _padded(lens, T, 21).cuda()
    need = _lib.load().cmwg_denoise_workspace_bytes(len(lens), T, n_fft, hop)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    # a full-length call on other data first: every frame of the workspace then holds stale values
    other = ops.denoise(torch.randn(len(lens), T).cuda(), w, bias, strength, hop, workspace=ws)
    assert other.abs().sum() > 0
    out = ops.denoise(x, w, bias, strength, hop, lengths=lens, workspace=ws)
    for b, n in enumerate(lens):
        solo = ops.denoise(x[b, :n].clone(), w, bias, strength, hop)
        assert torch.equal(out[b, :n], solo), (b, n, (out[b, :n] - solo).abs().max().item())
        assert (out[b, n:] == 0).all(), (b, "tail not zero")


def test_two_calls_are_bitwise_equal():
    lens = [4 * SR, 2 * SR + 3]
    x = _padded(lens, max(lens), 8).cuda()
    w, bias = _window(1024).cuda(), _bias(1024, 6).cuda()
    a = ops.denoise(x, w, bias, 0.1, 256, lengths=lens)
    b = ops.denoise(x, w, bias, 0.1, 256, lengths=lens)
    assert torch.equal(a, b)


def _waveglow(n_mels=80):
    torch.manual_seed(0)
    m = cm.WaveGlow(4, 8, 2, 2, 256, n_mels, True, zero_init=False, dilation_channels=64, residual_channels=64,
                    skip_channels=64, depth=2)
    m.apply(cm.remove_weight_norms)
    return m.cuda().eval()


def _waveflow():
    torch.manual_seed(1)
    m = cm.WaveFlow(2, 32, 8, False, False, dilation_channels=64, residual_channels=64, skip_channels=64, bias=False,
                    zero_init=False)
    m.apply(cm.remove_weight_norms)
    return m.cuda().eval()


@pytest.mark.parametrize("kind", ["waveglow", "waveflow"])
def test_bias_spectrum_matches_oracle(kind):
    m = _waveglow() if kind == "waveglow" else _waveflow()
    d = cm.Denoiser(m)
    assert d.bias_spec.shape == (513,) and d.bias_spec.is_cuda
    with torch.no_grad():
        bias_audio = m.infer(torch.zeros(1, m.n_mels, 88, device="cuda"), sigma=0.0)
    ref = O.bias_spectrum(bias_audio.double().cpu().numpy().reshape(-1), 1024, 256, O.window(1024, 1024))
    assert np.linalg.norm(ref) > 0
    assert _rel(d.bias_spec.cpu(), ref) <= 1e-5
    # the module applies that bias: its output is ops.denoise with it, for 1-D and batched input
    x = _signal(SR, 4).cuda()
    want = ops.denoise(x, d.window, d.bias_spec, 0.3, 256)
    assert torch.equal(d(x, 0.3), want)
    assert torch.equal(d(x[None], 0.3, lengths=[SR])[0], want)


def test_denoiser_short_window():
    m = _waveglow()
    d = cm.Denoiser(m, filter_length=1024, n_overlap=4, win_length=800)
    w = O.window(1024, 800)
    assert np.abs(d.window.cpu().numpy() - w).max() < 1e-6          # fp32 rounding of torch.hann_window
    x = _signal(2 * SR, 9)
    ref = O.denoise(x.double().numpy(), d.bias_spec.double().cpu().numpy(), 0.5, 1024, 256, d.window.double().cpu().numpy())
    assert _rel(d(x.cuda(), 0.5).cpu(), ref) <= 1e-5


def test_melspec_bits_unchanged_by_fft_move():
    g = torch.load(os.path.join(GOLDEN, "melspec_bits.pt"))
    with torch.no_grad():
        for case, want in zip(g["cases"], g["out"]):
            got = MelSpec(**case).cuda()(g["x"].cuda()).cpu()
            assert torch.equal(got, want), (case, (got - want).abs().max().item())


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


def test_cli_synth_batch_denoised_matches_solo(tmp_path):
    from constant_memory_waveglow_b200 import cli, datasets as D
    ckpt, wavs = _tiny_checkpoint(tmp_path)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, "-m", "constant_memory_waveglow_b200.cli", "synth-batch", ckpt, str(out), *wavs,
                        "-s", "0", "--max-batch", "2", "-d", "0.1"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    model, conditioner, dev = cli._load_for_synthesis(ckpt)
    denoiser = cm.Denoiser(model)
    changed = False
    for f in wavs:
        cond = conditioner(D.wav_read(f).mean(0, keepdim=True).to(dev))
        plain = model.infer(cond, 0.0)
        want = denoiser(plain, 0.1).reshape(1, -1)
        changed |= not torch.equal(want, plain.reshape(1, -1))
        got = D.wav_read(out / os.path.basename(f))
        # both through the 16-bit PCM writer: same samples
        ref_path = tmp_path / "ref.wav"
        D.wav_write(ref_path, want.cpu(), 22050)
        assert torch.equal(got, D.wav_read(ref_path)), f
    assert changed
