"""Band-limited resampling on the GPU: the kernel against the fp64 oracle, per-item lengths against solo calls (bit for
bit), 64-bit output lengths, equal rates, and `cli vocode --resample` / `--output-rate` and `cli score --resample`."""
import argparse

import numpy as np
import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli
from constant_memory_waveglow_b200.datasets import wav_info, wav_read, wav_write
from oracle import resample_oracle as R
from tests._util import rel_l2

pytestmark = pytest.mark.gpu

PAIRS = [(48000, 22050), (44100, 22050), (24000, 22050), (16000, 22050), (22050, 48000), (22050, 16000), (8000, 22050),
         (2, 3), (22050, 22050)]


def _signal(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, generator=g, dtype=torch.float64) * 2 - 1


@pytest.mark.parametrize("method", ["sinc_interp_hann", "sinc_interp_kaiser"])
@pytest.mark.parametrize("orig,new", PAIRS)
def test_kernel_matches_oracle(orig, new, method):
    r = cm.Resample(orig, new, method).cuda()
    for n in sorted({1, max(1, r.width - 1), 3 * r.O + 1, max(orig, 1000)}):
        x = _signal(n, n).float()
        got = r(x.cuda()).cpu().double()
        want = torch.from_numpy(R.resample_full(x.double().numpy(), orig, new, method=method))
        assert got.shape == want.shape == (r.output_lengths([n])[0],)
        assert (got - want).abs().max().item() <= 1e-6, (n, (got - want).abs().max().item())
        if n >= 1000:
            assert rel_l2(got, want) <= 3e-7, (n, rel_l2(got, want))


def _ragged(lens, T, seed):
    x = torch.full((len(lens), T), float("nan"))
    for b, n in enumerate(lens):
        x[b, :n] = _signal(n, seed + b).float()
    return x


@pytest.mark.parametrize("orig,new", [(48000, 22050), (16000, 22050), (22050, 48000), (22050, 16000), (2, 3),
                                      (22050, 22050), (44100, 22051)])
def test_lengths_match_solo_calls(orig, new):
    r = cm.Resample(orig, new).cuda()
    lens = [5000, 1, min(3 * r.O + 1, 4998), 4999, 17, 2500]
    x = _ragged(lens, 5000, 7).cuda()
    y = r(x, lengths=lens)
    assert y.shape == (len(lens), r.output_lengths([5000])[0])
    for b, (n, m) in enumerate(zip(lens, r.output_lengths(lens))):
        solo = r(x[b, :n].contiguous())
        assert solo.shape == (m,)
        assert torch.equal(y[b, :m], solo), b
        assert bool((y[b, m:] == 0).all()), b
        assert not torch.isnan(y[b]).any()


def test_same_buffers_after_a_longer_call_on_other_data():
    r = cm.Resample(48000, 22050).cuda()
    lens = [3000, 1200, 4000]
    x = _ragged(lens, 4000, 1).cuda()
    want = r(x, lengths=lens).clone()
    big = _ragged([40000, 39000, 38000, 40000], 40000, 99).cuda()
    r(big, lengths=[40000, 39000, 38000, 40000])
    r(big)
    assert torch.equal(r(x, lengths=lens), want)


def test_ten_minutes_at_48k():
    # N * len = 147 * 28.8e6 > 2**31: the output length and the kernel's sample test use 64-bit integers
    n = 48000 * 600 + 7
    r = cm.Resample(48000, 22050).cuda()
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(n, generator=g, device="cuda") * 2 - 1
    y = r(x)
    m = r.output_lengths([n])[0]
    assert y.shape == (m,) and m == (147 * n + 319) // 320
    xs = x.cpu().double().numpy()
    for start in (0, m // 2, m - 2000):                      # windows of the output against the oracle
        # a slice from a multiple of O that starts and ends further from the window than the filter reaches
        lo = max(0, (start // 147 - 2) * 320)
        piece = R.resample_full(xs[lo:lo + 320 * 20] if start < m - 2000 else xs[lo:], 48000, 22050)
        off = lo // 320 * 147
        want = torch.from_numpy(piece[start - off:start - off + 2000])
        got = y[start:start + want.numel()].cpu().double()
        assert (got - want).abs().max().item() <= 1e-6
    # as an item of a batch with a short one
    xb = torch.zeros((2, n), device="cuda")
    xb[0] = x
    xb[1, :1000] = x[:1000]
    yb = r(xb, lengths=[n, 1000])
    assert torch.equal(yb[0], y) and torch.equal(yb[1, :r.output_lengths([1000])[0]], r(x[:1000].contiguous()))


def test_equal_rates_copy_the_input():
    r = cm.Resample(22050, 22050).cuda()
    x = _ragged([3000, 100], 3000, 3)
    x[0, 5] = -0.0
    y = r(x.cuda(), lengths=[3000, 100]).cpu()
    assert torch.equal(y[0], x[0]) and torch.signbit(y[0, 5])
    assert torch.equal(y[1, :100], x[1, :100]) and bool((y[1, 100:] == 0).all())


def test_kernel_argument_checks():
    import ctypes as C
    from constant_memory_waveglow_b200 import _lib as L
    r = cm.Resample(48000, 22050).cuda()
    x = torch.zeros(2, 640, device="cuda")
    y = torch.zeros(2, 294, device="cuda")
    lib = L.load()

    def call(lens, T_out=294):
        lh = None if lens is None else (C.c_int * 2)(*lens)
        ld = None if lens is None else torch.tensor(lens, dtype=torch.int32, device="cuda")
        return lib.cmwg_resample(x.data_ptr(), 640, 2, 640, lh, L.ptr(ld), r.table.data_ptr(), r.first.data_ptr(), 320,
                                 147, r.table.shape[0], r.width, y.data_ptr(), 294, T_out, L.stream_ptr())
    assert call([640, 1]) == 0 and call(None) == 0
    assert call([641, 1]) != 0 and "outside" in lib.cmwg_last_error().decode()
    assert call([0, 1]) != 0
    assert call(None, T_out=293) != 0 and "T_out" in lib.cmwg_last_error().decode()
    assert lib.cmwg_resample(x.data_ptr(), 640, 2, 640, (C.c_int * 2)(640, 640), None, r.table.data_ptr(),
                             r.first.data_ptr(), 320, 147, r.table.shape[0], r.width, y.data_ptr(), 294, 294,
                             L.stream_ptr()) != 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# CLI
# ------------------------------------------------------------------------------------------------------------------
def _nvidia_ckpt(tmp_path):
    from oracle import nvidia_glow as NG
    cfg = dict(n_mel_channels=80, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
               WN_config=dict(n_layers=3, n_channels=64, kernel_size=3))
    path = tmp_path / "nv.pt"
    torch.save(NG.randomize(NG.WaveGlow(**cfg).double(), seed=0).float().state_dict(), path)
    return str(path)


def _wavs(tmp_path, rates_lens):
    files = []
    for i, (sr, n) in enumerate(rates_lens):
        f = tmp_path / f"w{i}.wav"
        g = torch.Generator().manual_seed(100 + i)
        wav_write(str(f), (torch.rand(1, n, generator=g) - 0.5) * 0.8, sr)
        files.append(str(f))
    return files


def _model_rate_signal(f):
    """What vocode/score make of a file: resampled alone to 22.05 kHz by cm.Resample."""
    x = wav_read(f).mean(0)
    sr = wav_info(f).sample_rate
    if sr == 22050:
        return x
    return cm.Resample(sr, 22050).cuda()(x.cuda()).cpu()


def _pcm(x):
    return (x.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round()


def test_vocode_resample_matches_resample_then_vocode(tmp_path):
    ck = _nvidia_ckpt(tmp_path)
    files = _wavs(tmp_path, [(16000, 3000), (48000, 9000), (16000, 2203), (48000, 4801), (22050, 3000)])
    out = tmp_path / "out"
    cli.main(["vocode", ck, str(out), *files, "--max-batch", "2", "--seed", "3", "--resample"])
    model, _, frontend = cli._load_vocoder_frontend(ck, argparse.ArgumentParser())
    model, frontend = model.cuda().eval(), frontend.cuda()
    for i, f in enumerate(files):
        x = _model_rate_signal(f)
        n = x.numel()
        with torch.no_grad():
            mel = frontend(x.cuda().unsqueeze(0))
            frames = mel.shape[-1]
            z = cli.item_noise(3, i, frames * 256, 0.6).cuda()
            want = model.infer(mel, 0.6, z=z.unsqueeze(0)).reshape(-1)[:n].cpu()
        got = wav_read(str(out / f"w{i}.wav")).reshape(-1)
        assert got.shape[0] == n
        assert torch.equal((got * 32768.0).round(), _pcm(want)), i


def test_vocode_output_rate(tmp_path):
    ck = _nvidia_ckpt(tmp_path)
    files = _wavs(tmp_path, [(22050, 3000), (22050, 5120), (22050, 1203)])
    ref, out = tmp_path / "ref", tmp_path / "out"
    cli.main(["vocode", ck, str(ref), *files, "--max-batch", "2", "--seed", "5"])
    cli.main(["vocode", ck, str(out), *files, "--max-batch", "2", "--seed", "5", "--output-rate", "16000"])
    model, _, frontend = cli._load_vocoder_frontend(ck, argparse.ArgumentParser())
    model, frontend = model.cuda().eval(), frontend.cuda()
    rs = cm.Resample(22050, 16000).cuda()
    for i, f in enumerate(files):
        x = wav_read(f).mean(0)
        with torch.no_grad():
            mel = frontend(x.cuda().unsqueeze(0))
            z = cli.item_noise(5, i, mel.shape[-1] * 256, 0.6).cuda()
            audio = model.infer(mel, 0.6, z=z.unsqueeze(0)).reshape(-1)[:x.numel()]
            want = rs(audio.contiguous()).cpu()
        got = wav_read(str(out / f"w{i}.wav")).reshape(-1)
        assert wav_info(str(out / f"w{i}.wav")).sample_rate == 16000
        assert wav_info(str(ref / f"w{i}.wav")).sample_rate == 22050
        assert got.shape[0] == want.shape[0] == -(-x.numel() * 320 // 441)
        assert torch.equal((got * 32768.0).round(), _pcm(want)), i


def test_score_resample(tmp_path, capsys):
    ck = _nvidia_ckpt(tmp_path)
    files = _wavs(tmp_path, [(16000, 3000), (48000, 9001), (16000, 2203), (22050, 4003)])
    got = cli.score_files(ck, files, 1.0, 3, argparse.ArgumentParser(), resample=True)
    model, _, frontend = cli._load_vocoder_frontend(ck, argparse.ArgumentParser())
    model, frontend = model.cuda().eval(), frontend.cuda()
    loss = cm.WaveGlowLoss(1.0)
    for (path, n, nll), f in zip(got, files):
        x = _model_rate_signal(f)
        assert path == f and n == x.numel() - x.numel() % 8
        x = x[:n].cuda().unsqueeze(0)
        with torch.no_grad():
            z, logdet = model(x, frontend(x))
            want = float(loss(z, logdet))
        assert nll == want, (f, nll, want)
    cli.main(["score", ck, *files, "--resample"])
    lines = capsys.readouterr().out.strip().splitlines()
    assert [int(ln.split("\t")[1]) for ln in lines] == [n for _, n, _ in got]
