"""NVIDIA WaveGlow support without a GPU: the upsampler's GEMM formulation, the key mapping onto the package's modules
(checked in fp64 against oracle/nvidia_glow.py), the checkpoint reader and the `vocode` argument checks."""
import io
import os
import pickle
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from constant_memory_waveglow_b200 import cli, nvidia
from oracle import flow_oracle as FO
from oracle import nvidia_glow as NG

SMALL = dict(n_mel_channels=80, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
             WN_config=dict(n_layers=3, n_channels=32, kernel_size=3))


def gemm_conditioning(w: torch.Tensor, bias: torch.Tensor, mel: torch.Tensor, T: int, n_group: int = 8) -> torch.Tensor:
    """What cmwg_nvidia_upsample_slab computes, in the GEMM's terms: rows = frames q, K = 4 taps x C (k = j C + i),
    columns n = (r // n_group) * C n_group + o * n_group + r % n_group; returns the (B, C n_group, T / n_group) tensor."""
    C, _, L = w.shape
    hop, taps = 256, L // 256
    B, _, Fr = mel.shape
    Tq = T // n_group
    Fq = -(-Tq // (hop // n_group))
    a = torch.zeros((B, Fq, taps * C), dtype=mel.dtype)
    for j in range(taps):
        for q in range(Fq):
            if 0 <= q - j < Fr:
                a[:, q, j * C:(j + 1) * C] = mel[:, :, q - j]
    n = torch.arange(hop * C)
    r = (n // (C * n_group)) * n_group + n % n_group
    o = (n % (C * n_group)) // n_group
    wp = torch.stack([w[:, o, r + hop * j] for j in range(taps)], 0)          # (taps, C_in, N)
    wp = wp.reshape(taps * C, hop * C)
    out = a @ wp + bias[o]                                                    # (B, Fq, N)
    slab = out.reshape(B, Fq * hop // n_group, C * n_group)[:, :Tq]           # rows = squeezed steps
    return slab.permute(0, 2, 1)


@pytest.mark.parametrize("frames,T", [(5, 5 * 256), (5, 5 * 256 - 8 * 7), (3, 3 * 256 + 768), (1, 8)])
def test_gemm_formulation_matches_conv_transpose(frames, T):
    g = torch.Generator().manual_seed(frames * 1000 + T)
    w = torch.randn(80, 80, 1024, generator=g, dtype=torch.float64)
    b = torch.randn(80, generator=g, dtype=torch.float64)
    mel = torch.randn(2, 80, frames, generator=g, dtype=torch.float64)
    ref = NG.WaveGlow(**SMALL).double()
    ref.upsample.weight.data.copy_(w)
    ref.upsample.bias.data.copy_(b)
    with torch.no_grad():
        want = ref.conditioning(mel, T)
    torch.testing.assert_close(gemm_conditioning(w, b, mel, T), want, rtol=1e-12, atol=1e-10)


def test_gemm_formulation_matches_infer_trim():
    g = torch.Generator().manual_seed(7)
    w = torch.randn(80, 80, 1024, generator=g, dtype=torch.float64)
    b = torch.randn(80, generator=g, dtype=torch.float64)
    mel = torch.randn(1, 80, 6, generator=g, dtype=torch.float64)
    up = F.conv_transpose1d(mel, w, b, stride=256)[..., :-768]                 # NVIDIA's infer
    want = up.unfold(2, 8, 8).permute(0, 2, 1, 3).reshape(1, up.shape[2] // 8, 640).permute(0, 2, 1)
    torch.testing.assert_close(gemm_conditioning(w, b, mel, up.shape[2]), want, rtol=1e-12, atol=1e-10)


def _oracle(cond_layers=False, seed=0):
    torch.manual_seed(seed)
    return NG.randomize(NG.WaveGlow(**SMALL, cond_layers=cond_layers).double(), seed=seed)


def _package_flow(sd, cfg, x, mel, inverse):
    """The package's flow with the converted weights, in fp64 through oracle/flow_oracle.py (WN, coupling, 1x1 conv) and
    the restated upsampler."""
    n_group, every, esize = cfg["n_group"], cfg["n_early_every"], cfg["n_early_size"]
    T = x.shape[1]
    up = F.conv_transpose1d(mel, sd["upsample.weight"], sd["upsample.bias"], stride=256)[..., :T]
    y = up.reshape(up.shape[0], up.shape[1], T // n_group, n_group).permute(0, 1, 3, 2).reshape(up.shape[0], -1, T // n_group)
    xs = FO.squeeze(x, n_group)
    logdet = 0
    if not inverse:
        outs = []
        for k in range(cfg["n_flows"]):
            if k % every == 0 and k:
                outs.append(xs[:, :esize])
                xs = xs[:, esize:]
            xs, ldw = FO.conv1x1_forward(sd[f"invconv1x1.{k}.weight"], xs)
            xs, log_s = FO.coupling_forward(sd, f"WNs.{k}.F.", xs, y)
            logdet = logdet + ldw + log_s.sum((1, 2))
        outs.append(xs)
        return FO.unsqueeze(torch.cat(outs, 1)), logdet
    sizes = [esize] * ((cfg["n_flows"] - 1) // every) + [n_group - esize * ((cfg["n_flows"] - 1) // every)]
    *parts, z = xs.split(sizes, 1)
    for k in range(cfg["n_flows"] - 1, -1, -1):
        z, log_s = FO.coupling_reverse(sd, f"WNs.{k}.F.", z, y)
        z, ldw = FO.conv1x1_reverse(sd[f"invconv1x1.{k}.weight"], z)
        logdet = logdet + ldw + log_s.sum((1, 2))
        if k % every == 0 and k:
            z = torch.cat((parts.pop(), z), 1)
    return FO.unsqueeze(z), logdet


@pytest.mark.parametrize("cond_layers", [False, True])
def test_key_mapping_matches_oracle(cond_layers):
    ref = _oracle(cond_layers)
    cfg, sd = nvidia.convert_state_dict(nvidia.nvidia_state_dict(ref.state_dict()))
    assert cfg == {**SMALL, "WN_config": dict(SMALL["WN_config"])}
    g = torch.Generator().manual_seed(1)
    mel = torch.randn(2, 80, 4, generator=g, dtype=torch.float64)
    x = torch.randn(2, 4 * 256 - 64, generator=g, dtype=torch.float64) * 0.3
    with torch.no_grad():
        z_ref, ld_ref = ref(mel, x)
        z, ld = _package_flow(sd, cfg, x, mel, inverse=False)
        torch.testing.assert_close(z, z_ref, rtol=1e-10, atol=1e-10)
        torch.testing.assert_close(ld, ld_ref, rtol=1e-10, atol=1e-8)
        x_ref, ldr_ref = ref.reverse(mel, z_ref)
        xr, ldr = _package_flow(sd, cfg, z_ref, mel, inverse=True)
        torch.testing.assert_close(xr, x_ref, rtol=1e-10, atol=1e-10)
        torch.testing.assert_close(ldr, ldr_ref, rtol=1e-10, atol=1e-8)
        torch.testing.assert_close(x_ref, x, rtol=1e-8, atol=1e-8)    # the oracle itself round-trips


def test_model_state_dict_keys():
    model = nvidia.NvidiaWaveGlow(**SMALL)
    _, sd = nvidia.convert_state_dict(nvidia.nvidia_state_dict(_oracle().state_dict()))
    assert set(sd) == set(model.state_dict())
    for k, v in sd.items():
        assert model.state_dict()[k].shape == v.shape, k
    assert model.n_mels == 80 and model.WNs[0].F.aux_chs == 640 and model.WNs[0].F.has_bias


@pytest.fixture
def glow_module(monkeypatch):
    """oracle/nvidia_glow.py's classes importable as NVIDIA's module `glow`, so that a pickled model names glow.*."""
    mod = types.ModuleType("glow")
    for name in ("WaveGlow", "WN", "Invertible1x1Conv"):
        cls = getattr(NG, name)
        monkeypatch.setattr(cls, "__module__", "glow")
        setattr(mod, name, cls)
    monkeypatch.setitem(sys.modules, "glow", mod)
    return mod


def _assert_loaded(model, ref):
    _, sd = nvidia.convert_state_dict(nvidia.nvidia_state_dict(ref.state_dict()))
    got = model.state_dict()
    assert set(got) == set(sd)
    for k, v in sd.items():
        assert torch.equal(got[k], v.float()), k


@pytest.mark.parametrize("zip_format", [True, False])
def test_loader_reads_pickled_model(glow_module, zip_format, tmp_path):
    ref = _oracle().float()
    path = tmp_path / "waveglow.pt"
    torch.save({"model": ref, "iteration": 10}, path, _use_new_zipfile_serialization=zip_format)
    _assert_loaded(nvidia.load_nvidia_waveglow(str(path), device="cpu"), ref)


class _ThnnBackend:
    """What torch 1.0-1.4 stored in every module's `_backend`: it unpickles by calling this global."""

    def __reduce__(self):
        import torch.nn.backends.thnn as thnn
        return (thnn._get_thnn_function_backend, ())


@pytest.mark.parametrize("zip_format", [True, False])
def test_loader_reads_torch1_era_pickle(glow_module, zip_format, tmp_path):
    ref = _oracle().float()
    for m in ref.modules():
        m._backend = _ThnnBackend()
    path = tmp_path / "waveglow.pt"
    torch.save({"model": ref}, path, _use_new_zipfile_serialization=zip_format)
    assert b"_get_thnn_function_backend" in (path.read_bytes() if not zip_format else
                                             __import__("zipfile").ZipFile(path).read("waveglow/data.pkl"))
    _assert_loaded(nvidia.load_nvidia_waveglow(str(path), device="cpu"), ref)


def test_loader_reads_state_dict_forms(tmp_path):
    ref = _oracle(cond_layers=True).float()
    dle = {"state_dict": {"module." + k: v for k, v in ref.state_dict().items()}, "epoch": 3}
    torch.save(dle, tmp_path / "dle.pt")
    _assert_loaded(nvidia.load_nvidia_waveglow(str(tmp_path / "dle.pt"), device="cpu"), ref)
    _assert_loaded(nvidia.load_nvidia_waveglow(ref.state_dict(), device="cpu"), ref)


def test_loader_reads_plain_weights():
    ref = _oracle().float()
    sd = {}
    for k, v in ref.state_dict().items():       # fold weight norm: what remove_weightnorm leaves
        if k.endswith("weight_v"):
            sd[k[:-2]] = FO.weight_norm_weight(ref.state_dict()[k[:-1] + "g"], v)
        elif not k.endswith("weight_g"):
            sd[k] = v
    model = nvidia.load_nvidia_waveglow(sd, device="cpu")
    assert not any(k.endswith("weight_g") for k in model.state_dict())
    assert torch.equal(model.state_dict()["WNs.1.F.start.weight"], sd["WN.1.start.weight"])


class _Evil:
    def __init__(self, marker):
        self.marker = marker

    def __reduce__(self):
        return (os.makedirs, (self.marker,))


@pytest.mark.parametrize("zip_format", [True, False])
def test_loader_refuses_other_globals(zip_format, tmp_path):
    marker = str(tmp_path / "ran")
    path = tmp_path / "evil.pt"
    torch.save({"model": _Evil(marker)}, path, _use_new_zipfile_serialization=zip_format)
    with pytest.raises(pickle.UnpicklingError):
        nvidia.load_nvidia_waveglow(str(path), device="cpu")
    assert not os.path.exists(marker)


@pytest.fixture
def small_ckpt(tmp_path):
    path = tmp_path / "nv.pt"
    torch.save(_oracle().float().state_dict(), path)
    return str(path)


def _vocode_error(argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(["vocode"] + argv)
    assert e.value.code == 2
    return capsys.readouterr().err


def test_vocode_rejects_bad_mel_shape(small_ckpt, tmp_path, capsys):
    bad = tmp_path / "a.npy"
    np.save(bad, np.zeros((2, 80, 5), dtype=np.float32))
    assert "(n_mels, frames)" in _vocode_error([small_ckpt, str(tmp_path / "out"), str(bad)], capsys)
    wrong = tmp_path / "b.pt"
    torch.save(torch.zeros(5, 80), wrong)     # (frames, n_mels): the other orientation is an error
    assert "80 mel channels" in _vocode_error([small_ckpt, str(tmp_path / "out"), str(wrong)], capsys)


def test_vocode_rejects_wrong_n_mels(small_ckpt, tmp_path, capsys):
    m = tmp_path / "a.pt"
    torch.save(torch.zeros(1, 64, 5), m)
    assert "80 mel channels" in _vocode_error([small_ckpt, str(tmp_path / "out"), str(m)], capsys)


def test_vocode_rejects_duplicate_stems(small_ckpt, tmp_path, capsys):
    (tmp_path / "x").mkdir()
    a, b = tmp_path / "a.pt", tmp_path / "x" / "a.npy"
    torch.save(torch.zeros(80, 5), a)
    np.save(b, np.zeros((80, 5), dtype=np.float32))
    assert "distinct names" in _vocode_error([small_ckpt, str(tmp_path / "out"), str(a), str(b)], capsys)


def test_upsample_abi_sizes_and_argument_checks():
    from constant_memory_waveglow_b200 import _lib
    lib = _lib.load()
    assert lib.cmwg_nvidia_upsample_packed_bytes(80, 256, 4) == 256 * 80 * 320 * 2      # K = 4 x 80 = 5 blocks of 64
    whole = lib.cmwg_nvidia_upsample_workspace_bytes(2, 32 * 10, 80, 256, 4, 8)         # whole frames: operand only
    part = lib.cmwg_nvidia_upsample_workspace_bytes(2, 32 * 10 - 5, 80, 256, 4, 8)      # + the whole-frame staging slab
    assert whole >= 2 * 10 * 320 * 2 and part >= whole + 2 * 10 * 20480 * 2 - 1024
    assert lib.cmwg_nvidia_upsample_workspace_bytes(2, 320, 81, 256, 4, 8) == 0          # 648 slab channels: unsupported
    assert lib.cmwg_nvidia_upsample_slab(None, None, None, 0, 0, 1, 81, 4, 256, 4, 8, 32, 2, None, None, None) != 0
    assert lib.cmwg_nvidia_upsample_slab(None, None, None, 0, 0, 1, 80, 4, 256, 4, 8, 32, 2, None, None, None) != 0
    assert lib.cmwg_nvidia_upsample_pack(None, 80, 256, 4, 8, 0, None, None) != 0       # fp32 has no 16-bit operand


def lightning_checkpoint(tmp_path, arch):
    """A small checkpoint of this package's Lightning module (the form `cli train` writes)."""
    from constant_memory_waveglow_b200 import trainer as TR
    cfg = {
        "name": "tiny", "arch": arch,
        "dataset": {"type": "RandomWAVDataset", "args": {"data_dir": str(tmp_path), "size": 4, "segment": 4096}},
        "data_loader": {"batch_size": 2, "shuffle": False, "num_workers": 0, "pin_memory": False},
        "optimizer": {"type": "Adam", "args": {"lr": 1e-3, "weight_decay": 0}},
        "loss": {"type": "WaveGlowLoss", "args": {"sigma": 0.7, "elementwise_mean": True}},
        "conditioner": {"type": "MelSpec", "args": {"sr": 16000, "n_fft": 1024, "hop_length": 256, "f_max": 8000,
                                                    "n_mels": 80}},
    }
    torch.manual_seed(4)
    lm = TR.LightModel(cfg)
    with torch.no_grad():
        for p in lm.model.parameters():
            p.add_(torch.randn_like(p) * 0.02)   # zero-initialised `end` convs would make every flow the identity
    path = tmp_path / "tiny.ckpt"
    torch.save(lm.checkpoint(epoch=0, global_step=0), path)
    return str(path)


TINY_WAVEGLOW = {"type": "WaveGlow", "args": dict(flows=4, n_group=8, n_early_every=2, n_early_size=2, hop_size=256,
                                                  n_mels=80, memory_efficient=True, reverse_mode=False,
                                                  dilation_channels=64, residual_channels=64, skip_channels=64,
                                                  depth=2, radix=3, bias=False)}


def test_vocode_detects_checkpoint_kind(small_ckpt, tmp_path):
    import argparse
    p = argparse.ArgumentParser()
    model, sr = cli._load_vocoder(small_ckpt, p)
    assert type(model) is nvidia.NvidiaWaveGlow and sr == 22050
    model, sr = cli._load_vocoder(lightning_checkpoint(tmp_path, TINY_WAVEGLOW), p)
    assert type(model).__name__ == "WaveGlow" and sr == 16000       # the conditioner's rate
