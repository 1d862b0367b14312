"""Tacotron2's mel front end on the GPU: TacotronSTFT against the fp64 oracle, per-item lengths of TacotronSTFT and
MelSpec against each item's own call (bit for bit), and copy synthesis / scoring of WAV files through the CLI."""
import argparse

import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli
from constant_memory_waveglow_b200.condition import MelSpec
from constant_memory_waveglow_b200.datasets import wav_read, wav_write
from oracle import tacotron_stft as O
from tests._util import rel_l2

pytestmark = pytest.mark.gpu


def audio(B, T, seed=0):
    g = torch.Generator().manual_seed(seed)
    y = torch.rand(B, T, generator=g) * 2 - 1
    y[:, T // 3:T // 2] *= 1e-3                              # quiet stretch: mels near the clamp
    y[:, T // 2:T // 2 + 700] = 0                            # silence: mels clamped at 1e-5
    return y


@pytest.mark.parametrize("n_fft,hop,win,n_mels,sr", [(1024, 256, 1024, 80, 22050), (256, 64, 256, 40, 16000),
                                                     (2048, 512, 2048, 128, 44100), (1024, 256, 800, 80, 22050)])
def test_mel_spectrogram_matches_oracle(n_fft, hop, win, n_mels, sr):
    t = cm.TacotronSTFT(n_fft, hop, win, n_mels, sr).cuda()
    y = audio(3, 9000, seed=n_fft + win)
    got = t.mel_spectrogram(y.cuda()).cpu().double()
    assert got.shape == (3, n_mels, 9000 // hop + 1)
    kw = dict(filter_length=n_fft, hop_length=hop, win_length=win, n_mel_channels=n_mels, sampling_rate=sr)
    # the same fp32 filterbank: what is left is the fp32 STFT and mel sum
    want = O.mel_spectrogram(y.double(), basis=t.mel_basis.cpu(), **kw)
    assert (got - want).abs().max().item() < 5e-3
    assert rel_l2(got.exp(), want.exp()) < 2e-6
    # librosa's fp64 filterbank
    want64 = O.mel_spectrogram(y.double(), **kw)
    assert rel_l2(got.exp(), want64.exp()) < 2e-6
    # (T,) in, (n_mels, frames) out
    assert torch.equal(t.mel_spectrogram(y[1].cuda()).cpu().double(), got[1])


def _ragged(T, lens, seed):
    y = audio(len(lens), T, seed=seed)
    yp = y.clone()
    for b, n in enumerate(lens):
        yp[b, n:] = 1e3                                      # garbage past each length
    return y, yp


def _check_items(out, solo_fn, y, lens, hop):
    for b, n in enumerate(lens):
        f = n // hop + 1
        solo = solo_fn(y[b, :n].cuda().unsqueeze(0))[0]
        assert solo.shape[-1] == f
        assert torch.equal(out[b, :, :f], solo), (b, n)
        assert torch.equal(out[b, :, f:], torch.zeros_like(out[b, :, f:])), (b, n)


@pytest.mark.parametrize("n_fft,hop,win,lens", [
    (1024, 256, 1024, [513, 1000, 2560, 6000, 256 * 9 + 3]),      # just above n_fft/2, not a multiple, a multiple, T
    (256, 160, 256, [160, 129, 777, 1600]),                       # one hop, just above n_fft/2, T
    (1024, 256, 800, [6000, 700, 4096])])
def test_tacotron_lengths_match_solo_calls(n_fft, hop, win, lens):
    t = cm.TacotronSTFT(n_fft, hop, win).cuda()
    T = max(lens)
    y, yp = _ragged(T, lens, seed=len(lens))
    out = t.mel_spectrogram(yp.cuda(), lengths=lens)
    assert out.shape == (len(lens), 80, T // hop + 1)
    _check_items(out, t.mel_spectrogram, y, lens, hop)
    # an all-full batch with lengths equals the call without them
    assert torch.equal(t.mel_spectrogram(y[:, :T].cuda(), lengths=[T] * len(lens)), t.mel_spectrogram(y.cuda()))


@pytest.mark.parametrize("kw", [dict(), dict(power=1.0, win_length=800), dict(n_fft=256, hop_length=64, n_mels=40)])
def test_melspec_lengths_match_existing_kernel(kw):
    args = dict(sr=22050, n_fft=1024, hop_length=256, n_mels=80)
    args.update(kw)
    m = MelSpec(**args).cuda()
    hop, pad = m.hop_length, m.n_fft // 2 + m.hop_length // 2
    lens = [pad + 1, hop * 7, hop * 11 + 5, 4000]
    T = max(lens)
    y, yp = _ragged(T, lens, seed=7)
    out = m(yp.cuda(), lengths=lens)
    # the solo reference is MelSpec without lengths: the existing kernel
    _check_items(out, m, y, lens, hop)


def test_kernel_argument_checks():
    from constant_memory_waveglow_b200 import _lib as L
    import ctypes as C
    lib = L.load()
    t = cm.TacotronSTFT().cuda()
    w, fbt, lo, hi = t._device_tables(torch.device("cuda"))
    x = torch.zeros(2, 2000, device="cuda")
    out = torch.empty(2, 80, 2000 // 256 + 1, device="cuda")
    lens = torch.tensor([2000, 600], dtype=torch.int32, device="cuda")

    def call(lh, log_mode=2, eps=1e-5, pad_left=512):
        return lib.cmwg_melspec_fwd_varlen(x.data_ptr(), 2000, 2, 2000, lh, lens.data_ptr() if lh else None, w.data_ptr(),
                                           fbt.data_ptr(), lo.data_ptr(), hi.data_ptr(), 1024, 256, 80, pad_left, 1,
                                           log_mode, eps, out.data_ptr(), L.stream_ptr())
    assert call((C.c_int * 2)(2000, 600)) == 0
    for bad in ((2000, 512), (2001, 600), (0, 600)):
        assert call((C.c_int * 2)(*bad)) != 0
    assert call((C.c_int * 2)(2000, 641), pad_left=384) == 0        # MelSpec's pads (384, 640)
    assert call((C.c_int * 2)(2000, 640), pad_left=384) != 0        # n_fft - pad_left = 640: not enough
    assert call(None, log_mode=3) != 0
    assert call(None, eps=-1.0) != 0
    assert call(None, eps=float("inf")) != 0
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
    return str(path), 22050


def _lightning_ckpt(tmp_path):
    from tests.test_nvidia_host import TINY_WAVEGLOW, lightning_checkpoint
    return lightning_checkpoint(tmp_path, TINY_WAVEGLOW), 16000


CKPTS = {"nvidia": _nvidia_ckpt, "lightning": _lightning_ckpt}


def _wavs(tmp_path, sr, lens):
    files = []
    for i, n in enumerate(lens):
        f = tmp_path / f"w{i}.wav"
        g = torch.Generator().manual_seed(100 + i)
        wav_write(str(f), (torch.rand(2, n, generator=g) - 0.5) * 0.8, sr)      # two channels: averaged
        files.append(str(f))
    return files


@pytest.mark.parametrize("kind", ["nvidia", "lightning"])
def test_vocode_wavs_match_solo_infer(kind, tmp_path):
    ck, sr = CKPTS[kind](tmp_path)
    lens = [3000, 5120, 1203, 4000]
    files = _wavs(tmp_path, sr, lens)
    out = tmp_path / "out"
    cli.main(["vocode", ck, str(out), *files, "--max-batch", "3", "--seed", "3", "-s", "0.6"])
    model, _, frontend = cli._load_vocoder_frontend(ck, argparse.ArgumentParser())
    model, frontend = model.cuda().eval(), frontend.cuda()
    for i, (f, n) in enumerate(zip(files, lens)):
        with torch.no_grad():
            mel = frontend(wav_read(f).mean(0).cuda().unsqueeze(0))
            frames = mel.shape[-1]
            assert frames == n // 256 + 1
            z = cli.item_noise(3, i, frames * 256, 0.6).cuda()
            want = model.infer(mel, 0.6, z=z.unsqueeze(0)).reshape(-1)[:n].cpu()
        got = wav_read(str(out / f"w{i}.wav")).reshape(-1)
        assert got.shape[0] == n
        assert torch.equal((got * 32768.0).round(), (want.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round()), i


@pytest.mark.parametrize("kind", ["nvidia", "lightning"])
def test_score_matches_solo_loss(kind, tmp_path, capsys):
    ck, sr = CKPTS[kind](tmp_path)
    lens = [3000, 5120, 1203, 4003, 2048, 3001]               # multiples of the hop, and of neither hop nor n_group
    files = _wavs(tmp_path, sr, lens)
    got = cli.score_files(ck, files, 1.0, 3, argparse.ArgumentParser())
    model, _, frontend = cli._load_vocoder_frontend(ck, argparse.ArgumentParser())
    model, frontend = model.cuda().eval(), frontend.cuda()
    loss = cm.WaveGlowLoss(1.0)
    for (path, n, nll), f, n_in in zip(got, files, lens):
        assert path == f and n == n_in - n_in % 8
        x = wav_read(f).mean(0)[:n].cuda().unsqueeze(0)
        with torch.no_grad():
            z, logdet = model(x, frontend(x))
            want = float(loss(z, logdet))
        assert nll == want, (f, nll, want)
    cli.main(["score", ck, *files, "--max-batch", "4"])
    lines = capsys.readouterr().out.strip().splitlines()
    assert [ln.split("\t")[0] for ln in lines] == files
    assert [int(ln.split("\t")[1]) for ln in lines] == [n for _, n, _ in got]
