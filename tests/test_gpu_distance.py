"""Spectral distances on the device (csrc/distance.cu): against the fp64 oracle on ragged batches, batched items against
solo calls (bit for bit), exact identities, and `cli compare` end to end (with `cli vocode` and `--resample`)."""
import math

import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli
from constant_memory_waveglow_b200.datasets import wav_read, wav_write
from oracle import distance_oracle as O

pytestmark = pytest.mark.gpu


def _noise(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, generator=g) * 2 - 1


def _harmonic_with_silence(n, seed):
    t = torch.arange(n, dtype=torch.float64) / 22050.0
    x = 0.3 * torch.sin(2 * math.pi * 220 * t) + 0.2 * torch.sin(2 * math.pi * 660 * t) \
        + 0.1 * torch.sin(2 * math.pi * 1100 * t + seed)
    x[n // 4:n // 2] = 0.0
    x[-(n // 8):] = 0.0
    return x.float()


def _pair(kind, n, seed):
    if kind == "noise":
        return _noise(n, seed), _noise(n, seed + 1000)
    ref = _harmonic_with_silence(n, seed)
    return ref, 0.7 * ref + 0.05 * _noise(n, seed + 1000) * (ref != 0)


def _ragged(items, T):
    """(B, T) pairs of signals, NaN past each length."""
    x = torch.full((len(items), T), float("nan"))
    y = torch.full((len(items), T), float("nan"))
    for b, (r, e) in enumerate(items):
        x[b, :r.numel()], y[b, :e.numel()] = r, e
    return x, y


# The kernel works in fp32 on fp32 input; the oracle gets the same fp32 samples and the module's fp32 filterbank in
# float64.  LSD is the loosest: every bin enters it through log10 of an fp32 power, and low-power bins (the harmonic
# signal's stopband, near the 1e-10 clamp) carry the largest relative error of the FFT's rounding.  The mel sums many bins
# before its log, so the log-mel L1, and the MCD built from the same log-mel differences, are an order of magnitude tighter.
# Observed on the B200, worst item of the batch: LSD 7.7e-6 (noise) and 1.2e-5 (harmonic), log-mel L1 2.1e-8 / 5.3e-7,
# MCD 1.2e-7 / 5.3e-7 relative.  The bounds leave a factor of about 8-20.
RTOL = {"lsd": 1e-4, "mel_l1": 1e-5, "mcd": 1e-5}


@pytest.mark.parametrize("kind", ["noise", "harmonic"])
def test_matches_oracle_ragged_batch(kind):
    lens = [5000, 513, 4096, 22053, 7777]
    items = [_pair(kind, n, 10 + i) for i, n in enumerate(lens)]
    x, y = _ragged(items, max(lens))
    sd = cm.SpectralDistance().cuda()
    got = sd(x.cuda(), y.cuda(), lengths=lens)
    basis = sd.mel_basis.cpu()
    worst = {k: 0.0 for k in RTOL}
    for b, (r, e) in enumerate(items):
        want = O.distances(r.double().numpy(), e.double().numpy(), basis=basis)
        for k, w, g in zip(RTOL, want, got):
            err = abs(float(g[b]) - w) / max(abs(w), 1e-3)
            worst[k] = max(worst[k], err)
            assert err <= RTOL[k], (kind, b, k, float(g[b]), w)
    print(f"\n{kind}: worst relative error vs the fp64 oracle {worst}")


def _same(a, b):
    return all(torch.equal(p, q) for p, q in zip(a, b))


def test_batched_items_equal_solo_calls():
    T = 9000
    lens = [513, 256 * 20, 5001, T, 700]
    items = [_pair("noise" if i % 2 else "harmonic", n, 20 + i) for i, n in enumerate(lens)]
    x, y = _ragged(items, T)
    sd = cm.SpectralDistance().cuda()
    got = sd(x.cuda(), y.cuda(), lengths=lens)
    solos = [sd(r.cuda(), e.cuda()) for r, e in items]
    for b, solo in enumerate(solos):
        assert _same([t[b] for t in got], solo), b
        assert all(bool(torch.isfinite(t)) for t in solo)
    # a longer call on other data leaves stale workspace rows; a rerun is unchanged
    big_lens = [40000, 39000, 38000]
    bx, by = _ragged([_pair("noise", n, 50 + i) for i, n in enumerate(big_lens)], 40000)
    sd(bx.cuda(), by.cuda(), lengths=big_lens)
    sd(bx[:, :38000].contiguous().cuda(), by[:, :38000].contiguous().cuda())
    assert _same(sd(x.cuda(), y.cuda(), lengths=lens), got)


def test_ten_minute_item_next_to_a_short_one():
    n, short = 22050 * 600 + 5, 3000
    g = torch.Generator(device="cuda").manual_seed(0)
    r = torch.rand(n, generator=g, device="cuda") * 2 - 1
    e = 0.8 * r + 0.1 * (torch.rand(n, generator=g, device="cuda") * 2 - 1)
    x = torch.zeros((2, n), device="cuda")
    y = torch.zeros((2, n), device="cuda")
    x[0], y[0] = r, e
    x[1, :short], y[1, :short] = r[:short], e[:short]
    sd = cm.SpectralDistance().cuda()
    got = sd(x, y, lengths=[n, short])
    assert _same([t[0] for t in got], sd(r, e))
    assert _same([t[1] for t in got], sd(r[:short].contiguous(), e[:short].contiguous()))
    lsd, mel_l1, mcd = (float(t[0]) for t in got)
    assert all(math.isfinite(v) and v > 0 for v in (lsd, mel_l1, mcd))


def test_identities():
    sd = cm.SpectralDistance().cuda()
    lens = [6000, 513, 4097]
    items = [_pair("harmonic", n, 30 + i) for i, n in enumerate(lens)]
    x, y = _ragged(items, 6000)
    x, y = x.cuda(), y.cuda()
    zero = sd(x, x.clone(), lengths=lens)
    assert all(bool((t == 0).all()) for t in zero)
    assert _same(sd(x, y, lengths=lens), sd(y, x, lengths=lens))
    r = torch.stack([_noise(6000, 40 + i) for i in range(3)]).cuda()
    half = sd(r, 0.5 * r, lengths=lens)
    assert (half.lsd - 2 * math.log10(2)).abs().max().item() <= 1e-5
    assert (half.mel_l1 - math.log(2)).abs().max().item() <= 1e-5
    assert half.mcd.abs().max().item() <= 1e-3
    one = sd(r[0], 0.5 * r[0])                               # 1-D input: 0-d results, equal to the batched item
    assert one.lsd.dim() == 0 and _same(one, [t[0] for t in half])


# ------------------------------------------------------------------------------------------------------------------
# cli compare
# ------------------------------------------------------------------------------------------------------------------
def _pcm_even(n, seed):
    """Audio on even 16-bit codes: its 0.5-scaled copy is exact in a 16-bit WAV."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(-8000, 8000, (n,), generator=g) * 2).float() / 32768.0


def _lines(capsys):
    return [ln.split("\t") for ln in capsys.readouterr().out.strip().splitlines()]


def test_compare_half_scaled_copies_and_self(tmp_path, capsys):
    synth = tmp_path / "synth"
    synth.mkdir()
    refs = []
    for i, n in enumerate([4000, 22050, 1000]):
        x = _pcm_even(n, i)
        wav_write(str(tmp_path / f"u{i}.wav"), x, 22050)
        wav_write(str(synth / f"u{i}.wav"), 0.5 * x, 22050)
        refs.append(str(tmp_path / f"u{i}.wav"))
    cli.main(["compare", str(synth), *refs, "--max-batch", "2"])
    lines = _lines(capsys)
    assert [ln[0] for ln in lines] == refs + ["mean"] and [int(ln[1]) for ln in lines] == [4000, 22050, 1000, 27050]
    for ln in lines:
        assert abs(float(ln[2]) - 2 * math.log10(2)) <= 1e-5
        assert abs(float(ln[3]) - math.log(2)) <= 1e-5
        assert abs(float(ln[4])) <= 1e-3
    cli.main(["compare", str(tmp_path), *refs])               # each file against itself
    for ln in _lines(capsys):
        assert ln[2:] == ["0.000000"] * 3


def _nvidia_ckpt(tmp_path):
    from oracle import nvidia_glow as NG
    cfg = dict(n_mel_channels=80, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
               WN_config=dict(n_layers=3, n_channels=64, kernel_size=3))
    path = tmp_path / "nv.pt"
    torch.save(NG.randomize(NG.WaveGlow(**cfg).double(), seed=0).float().state_dict(), path)
    return str(path)


def test_vocode_then_compare(tmp_path, capsys):
    counts = [3000, 5120, 1203]
    refs = []
    for i, n in enumerate(counts):
        refs.append(str(tmp_path / f"w{i}.wav"))
        wav_write(refs[-1], (_noise(n, 60 + i) * 0.4).unsqueeze(0), 22050)
    out = tmp_path / "out"
    cli.main(["vocode", _nvidia_ckpt(tmp_path), str(out), *refs, "--max-batch", "2"])
    capsys.readouterr()
    cli.main(["compare", str(out), *refs, "--max-batch", "2"])
    lines = _lines(capsys)
    assert [int(ln[1]) for ln in lines[:-1]] == counts
    assert all(math.isfinite(float(v)) and float(v) > 0 for ln in lines for v in ln[2:])


def test_compare_resample_equals_resampling_first(tmp_path):
    import argparse
    synth = tmp_path / "synth"
    synth.mkdir()
    refs, pairs = [], []
    for i, n in enumerate([3000, 8000, 2203]):
        x, e = _noise(n, 70 + i) * 0.5, _noise(n, 80 + i) * 0.5
        wav_write(str(tmp_path / f"r{i}.wav"), x, 16000)
        wav_write(str(synth / f"r{i}.wav"), e, 16000)
        refs.append(str(tmp_path / f"r{i}.wav"))
        pairs.append((wav_read(refs[-1]).mean(0), wav_read(str(synth / f"r{i}.wav")).mean(0)))
    got = cli.compare_files(str(synth), refs, 22050, 2, argparse.ArgumentParser(), resample=True)
    rs = cm.Resample(16000, 22050).cuda()
    sd = cm.SpectralDistance().cuda()
    for (name, n, lsd, mel_l1, mcd), ref, (x, e) in zip(got, refs, pairs):
        xr, er = rs(x.cuda()), rs(e.cuda())
        assert name == ref and n == xr.numel() == er.numel()
        want = sd(xr, er)
        assert (lsd, mel_l1, mcd) == tuple(float(t) for t in want)
