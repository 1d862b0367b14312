"""NvidiaWaveGlow on the GPU: the upsampler GEMM's conditioning slab, synthesis and analysis against the fp64 restatement
of NVIDIA's model (oracle/nvidia_glow.py), ragged batches bit for bit against solo calls, the denoiser, checkpoints and
`cli vocode`."""
import copy

import numpy as np
import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli, nvidia
from constant_memory_waveglow_b200.datasets import wav_read
from oracle import nvidia_glow as NG

pytestmark = pytest.mark.gpu

SMALL = dict(n_mel_channels=80, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
             WN_config=dict(n_layers=3, n_channels=64, kernel_size=3))
PUBLISHED = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
                 WN_config=dict(n_layers=8, n_channels=256, kernel_size=3))
CONFIGS = {"small": SMALL, "published": PUBLISHED}
TOL = {"fp32": 1e-4, "fp16": 1e-2, "bf16": 4e-2}       # relative L2 error against the fp64 oracle
SLAB_TOL = {"fp16": 1e-3, "bf16": 8e-3}


@pytest.fixture
def prec_mode():
    old = cm.get_precision()
    yield cm.set_precision
    cm.set_precision(old)


_MODELS = {}


def models(name):
    """(fp64 oracle on the GPU, NvidiaWaveGlow with its weights)."""
    if name not in _MODELS:
        torch.manual_seed(0)
        ref = NG.randomize(NG.WaveGlow(**CONFIGS[name]).double(), seed=0).cuda().eval()
        _MODELS[name] = (ref, nvidia.load_nvidia_waveglow({k: v.float() for k, v in ref.state_dict().items()}))
    return _MODELS[name]


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


def mel(B, frames, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 80, frames, generator=g) * 0.5 - 1.0).cuda()


@pytest.mark.parametrize("prec", ["fp16", "bf16", "fp32"])
@pytest.mark.parametrize("T", [40 * 256, 40 * 256 - 8 * 13, 3 * 256 + 768])
def test_slab_against_oracle(prec, T):
    ref, model = models("small")
    h = mel(3, 40 if T >= 40 * 256 - 200 else 3, seed=T)
    Tq = T // 8
    with torch.no_grad():
        want = ref.conditioning(h.double(), T)                          # (B, 640, Tq)
        got = model._conditioning(h, Tq, prec)
    if prec == "fp32":
        assert rel(got, want) < 1e-6
        return
    dt = torch.float16 if prec == "fp16" else torch.bfloat16
    slab = got.data.view(dt).view(3, Tq, 640).permute(0, 2, 1)
    err = rel(slab, want)
    assert err < SLAB_TOL[prec], err
    # the bias and the boundary frames: the first and last squeezed steps of every item
    torch.testing.assert_close(slab[..., [0, Tq - 1]].double(), want[..., [0, Tq - 1]], rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("name", ["small", "published"])
@pytest.mark.parametrize("prec", ["fp32", "fp16", "bf16"])
def test_against_oracle(name, prec, prec_mode):
    prec_mode(prec)
    ref, model = models(name)
    h = mel(2, 24, seed=3)
    g = torch.Generator().manual_seed(5)
    z = (torch.randn(2, 24 * 256, generator=g) * 0.6).cuda()
    with torch.no_grad():
        x_ref = ref.infer(h.double(), z.double())
        x = model.infer(h, 0.6, z=z)
        assert rel(x, x_ref) < TOL[prec], rel(x, x_ref)
        T = 24 * 256 - 8 * 5
        xa = x_ref[:, :T].float()
        z_ref, ld_ref = ref(h.double(), xa.double())
        zz, ld = model(xa, h)
        assert rel(zz, z_ref) < TOL[prec], rel(zz, z_ref)
        assert rel(ld, ld_ref) < TOL[prec], (ld, ld_ref)
        xb, ldb = model.reverse(zz, h)
        assert rel(xb, xa) < TOL[prec], rel(xb, xa)
        assert rel(ldb, -ld) < TOL[prec]


@pytest.mark.parametrize("name", ["small", "published"])
@pytest.mark.parametrize("prec", ["fp32", "fp16"])
def test_ragged_batch_matches_solo(name, prec, prec_mode):
    prec_mode(prec)
    _, model = models(name)
    frames = [30, 1, 17, 9]                      # full length, one frame, mid-tile ends
    Fm = max(frames)
    h = mel(len(frames), Fm, seed=11)
    g = torch.Generator().manual_seed(12)
    z = (torch.randn(len(frames), Fm * 256, generator=g) * 0.6).cuda()
    hp, zp = h.clone(), z.clone()
    for b, f in enumerate(frames):               # garbage past each item's frames
        hp[b, :, f:] = 1e3
        zp[b, f * 256:] = 1e3
    with torch.no_grad():
        x = model.infer(hp, 0.6, z=zp, lengths=frames)
        lens = [f * 256 for f in frames]
        zz, ld = model(x, hp, lengths=lens)
        for b, f in enumerate(frames):
            n = f * 256
            solo = model.infer(h[b:b + 1, :, :f], 0.6, z=z[b:b + 1, :n])
            assert torch.equal(x[b, :n], solo.reshape(-1)), (b, f)
            assert torch.equal(x[b, n:], torch.zeros_like(x[b, n:]))
            zs, lds = model(x[b:b + 1, :n], h[b:b + 1, :, :f])
            assert torch.equal(zz[b, :n], zs.reshape(-1)), (b, f)
            assert torch.equal(zz[b, n:], torch.zeros_like(zz[b, n:]))
            assert torch.equal(ld[b:b + 1], lds), (b, f)


def test_autograd_is_refused():
    _, model = models("small")
    h = mel(1, 4)
    with pytest.raises(NotImplementedError):
        model(torch.zeros(1, 4 * 256, device="cuda"), h)
    with pytest.raises(NotImplementedError):
        model.reverse(torch.zeros(1, 4 * 256, device="cuda"), h)


def test_denoiser_runs():
    _, model = models("small")
    d = cm.Denoiser(model)
    with torch.no_grad():
        x = model.infer(mel(2, 20), 0.6)
        y = d(x, 0.1)
    assert y.shape == x.shape and torch.isfinite(y).all()


def test_pickled_checkpoint_synthesises_same_bits(tmp_path, monkeypatch):
    import sys
    import types
    ref, model = models("small")
    mod = types.ModuleType("glow")
    for n in ("WaveGlow", "WN", "Invertible1x1Conv"):
        monkeypatch.setattr(getattr(NG, n), "__module__", "glow")
        setattr(mod, n, getattr(NG, n))
    monkeypatch.setitem(sys.modules, "glow", mod)
    torch.save({"model": copy.deepcopy(ref).float().cpu()}, tmp_path / "wg.pt", _use_new_zipfile_serialization=False)
    loaded = nvidia.load_nvidia_waveglow(str(tmp_path / "wg.pt"))
    h = mel(2, 12)
    z = torch.randn(2, 12 * 256, device="cuda") * 0.6
    with torch.no_grad():
        assert torch.equal(loaded.infer(h, 0.6, z=z), model.infer(h, 0.6, z=z))


def test_vocode_matches_solo_infer(tmp_path):
    ref, model = models("small")
    ck = tmp_path / "nv.pt"
    torch.save({k: v.float().cpu() for k, v in ref.state_dict().items()}, ck)
    mels = [mel(1, f, seed=f)[0].cpu() for f in (7, 13, 4)]
    torch.save(mels[0], tmp_path / "a.pt")
    np.save(tmp_path / "b.npy", mels[1].unsqueeze(0).numpy())
    torch.save(mels[2].unsqueeze(0), tmp_path / "c.pt")
    files = [str(tmp_path / n) for n in ("a.pt", "b.npy", "c.pt")]
    out = tmp_path / "out"
    cli.main(["vocode", str(ck), str(out), *files, "--max-batch", "2", "--seed", "3", "-s", "0.6"])
    for i, (f, m) in enumerate(zip(("a", "b", "c"), mels)):
        n = m.shape[1] * 256
        z = cli.item_noise(3, i, n, 0.6).cuda()
        with torch.no_grad():
            want = model.infer(m.cuda().unsqueeze(0), 0.6, z=z.unsqueeze(0)).reshape(-1).cpu()
        got = wav_read(str(out / f"{f}.wav")).reshape(-1)
        assert got.shape[0] == n
        # 16-bit PCM: the written samples are exactly the solo call's, quantised as wav_write quantises
        assert torch.equal((got * 32768.0).round(), (want.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round())


TINY_WAVEFLOW = {"type": "WaveFlow", "args": dict(flows=2, n_group=16, n_mels=80, use_conv1x1=False,
                                                  memory_efficient=False, dilation_channels=64, residual_channels=64,
                                                  skip_channels=64)}


@pytest.mark.parametrize("family", ["WaveGlow", "WaveFlow"])
def test_vocode_lightning_checkpoint_matches_solo_infer(family, tmp_path):
    import argparse
    from tests.test_nvidia_host import TINY_WAVEGLOW, lightning_checkpoint
    ck = lightning_checkpoint(tmp_path, TINY_WAVEGLOW if family == "WaveGlow" else TINY_WAVEFLOW)
    mels = [mel(1, f, seed=f)[0].cpu() for f in (9, 5, 14)]
    files = []
    for i, m in enumerate(mels):
        torch.save(m, tmp_path / f"m{i}.pt")
        files.append(str(tmp_path / f"m{i}.pt"))
    out = tmp_path / "out"
    cli.main(["vocode", ck, str(out), *files, "--max-batch", "3", "--seed", "5", "-s", "0.6"])
    model, sr = cli._load_vocoder(ck, argparse.ArgumentParser())
    model = model.cuda().eval()
    assert type(model).__name__ == family and sr == 16000
    for i, m in enumerate(mels):
        n = m.shape[1] * 256
        z = cli.item_noise(5, i, n, 0.6).cuda()
        with torch.no_grad():
            want = model.infer(m.cuda().unsqueeze(0), 0.6, z=z.unsqueeze(0)).reshape(-1).cpu()
        got = wav_read(str(out / f"m{i}.wav")).reshape(-1)
        assert got.shape[0] == n
        assert torch.equal((got * 32768.0).round(), (want.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round()), i
