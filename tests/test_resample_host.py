"""Band-limited resampling without a GPU: the fp64 oracle against torchaudio.functional.resample, the compact table
against the oracle, output lengths, argument checks, and the --resample / --output-rate flags of `cli vocode` / `cli score`."""
import numpy as np
import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import cli, ops
from constant_memory_waveglow_b200.datasets import wav_write
from constant_memory_waveglow_b200.resample import resample_table
from oracle import resample_oracle as R

PAIRS = [(48000, 22050), (44100, 22050), (24000, 22050), (16000, 22050), (22050, 48000), (22050, 16000), (8000, 22050),
         (2, 3), (22050, 22050)]
METHODS = ["sinc_interp_hann", "sinc_interp_kaiser"]


def _lengths(orig, new):
    """1, shorter than w, not a multiple of O, and about 1 s."""
    O, _ = R.reduced(orig, new)
    w = 0 if orig == new else R.kernel(orig, new)[2]
    return sorted({1, max(1, w - 1), 3 * O + 1, max(orig, 1000)})


def _signal(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, generator=g, dtype=torch.float64) * 2 - 1


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("orig,new", PAIRS)
def test_oracle_matches_torchaudio(orig, new, method):
    torchaudio = pytest.importorskip("torchaudio")
    table, first, w = R.compact_table(orig, new, method=method) if orig != new else (None, None, 0)
    for n in _lengths(orig, new):
        x = _signal(n, n)
        want = torchaudio.functional.resample(x, orig, new, resampling_method=method).numpy()
        full = R.resample_full(x.numpy(), orig, new, method=method)
        assert full.shape == want.shape == (R.output_length(n, orig, new),)
        assert np.abs(full - want).max(initial=0.0) <= 1e-12
        if table is not None:
            compact = R.resample_compact(x.numpy(), table, first, w, orig, new)
            assert np.abs(compact - want).max(initial=0.0) <= 1e-12


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("orig,new", [p for p in PAIRS if p[0] != p[1]])
def test_table_keeps_exactly_the_taps_inside_the_window(orig, new, method):
    table, first, O, N, w = resample_table(orig, new, method)
    K, t, w_ref = R.kernel(orig, new, method=method)
    assert (O, N) == R.reduced(orig, new) and w == w_ref and table.dtype == torch.float32 and first.dtype == torch.int32
    L = table.shape[0]
    assert table.shape == (L, N)
    for j in range(N):
        keep = np.nonzero(np.abs(t[j]) < 6)[0]
        assert keep.size and int(first[j]) == keep[0] and np.array_equal(keep, np.arange(keep[0], keep[-1] + 1))
        assert torch.equal(table[:keep.size, j], torch.from_numpy(K[j, keep]).float())
        assert torch.equal(table[keep.size:, j], torch.zeros(L - keep.size))
        # the dropped taps are rounding residue of a zero
        dropped = np.delete(K[j], keep)
        assert np.abs(dropped).max(initial=0.0) < 1e-15
    L_max = max(np.count_nonzero(np.abs(t[j]) < 6) for j in range(N))
    assert L == L_max
    ref, ref_first, _ = R.compact_table(orig, new, method=method)
    assert torch.equal(table, torch.from_numpy(ref).float()) and torch.equal(first.long(), torch.from_numpy(ref_first))


@pytest.mark.parametrize("method", METHODS)
def test_table_of_an_odd_ratio(method):
    # 44.1 -> 22.051 kHz: N = 22051 phases of a 44126-tap kernel; the table is built without the full kernel
    table, first, O, N, w = resample_table(44100, 22051, method)
    assert (O, N, w) == (44100, 22051, 13) and table.shape == (25, N)
    phases = np.r_[0:40, N // 2 - 20:N // 2 + 20, N - 40:N]
    K, t, _ = R.kernel(44100, 22051, method=method, phases=phases)
    for r, j in enumerate(phases):
        keep = np.nonzero(np.abs(t[r]) < 6)[0]
        assert int(first[j]) == keep[0] and np.array_equal(keep, np.arange(keep[0], keep[-1] + 1))
        assert torch.equal(table[:keep.size, j], torch.from_numpy(K[r, keep]).float())
        assert torch.equal(table[keep.size:, j], torch.zeros(table.shape[0] - keep.size))


def test_table_sizes_of_common_pairs():
    # taps per phase inside the window (torchaudio's kernels have 348, 334, 459 and 161)
    for (orig, new), L in {(48000, 22050): 27, (16000, 22050): 13, (22050, 16000): 17, (22050, 48000): 13}.items():
        assert resample_table(orig, new)[0].shape[0] == L


def test_equal_rates_give_the_identity_table():
    table, first, O, N, w = resample_table(22050, 22050)
    assert torch.equal(table, torch.ones(1, 1)) and torch.equal(first, torch.zeros(1, dtype=torch.int32))
    assert (O, N, w) == (1, 1, 0)


def test_output_lengths():
    r = cm.Resample(48000, 22050)
    assert r.output_lengths([1, 320, 321, 48000]) == [1, 147, 148, 22050]
    assert r.output_lengths(torch.tensor([1000])) == [-(-147 * 1000 // 320)]
    # 10 minutes at 48 kHz: N * len = 4.2e9 > 2**31
    n = 48000 * 600
    assert 147 * n > 2 ** 31 and r.output_lengths([n]) == [22050 * 600] == [R.output_length(n, 48000, 22050)]
    n = 48000 * 600 + 7
    assert r.output_lengths([n]) == [(147 * n + 319) // 320] == [R.output_length(n, 48000, 22050)]
    assert cm.Resample(16000, 22050).output_lengths([16001]) == [22052]
    assert cm.Resample(22050, 22050).output_lengths([5, 7]) == [5, 7]


def test_constructor_checks():
    with pytest.raises(ValueError, match="integer type"):
        cm.Resample(44100.5, 22050)
    with pytest.raises(ValueError, match="should be positive"):
        cm.Resample(0, 22050)
    with pytest.raises(ValueError, match="should be positive"):
        cm.Resample(16000, -1)
    with pytest.raises(ValueError, match="Low pass filter width should be positive"):
        cm.Resample(16000, 22050, lowpass_filter_width=0)
    with pytest.raises(ValueError, match="lowpass_filter_width"):
        cm.Resample(16000, 22050, lowpass_filter_width=6.5)
    for bad in (0.0, 1.01, -0.5, float("nan")):
        with pytest.raises(ValueError, match="rolloff"):
            cm.Resample(16000, 22050, rolloff=bad)
    with pytest.raises(ValueError, match="Invalid resampling method"):
        cm.Resample(16000, 22050, resampling_method="linear")
    with pytest.raises(ValueError, match="beta"):
        cm.Resample(16000, 22050, resampling_method="sinc_interp_kaiser", beta=float("inf"))
    # integral floats are taken; beta is ignored with the Hann window, as torchaudio ignores it
    r = cm.Resample(16000.0, 22050.0, beta=float("nan"))
    assert (r.orig_freq, r.new_freq, r.beta) == (16000, 22050, None)
    assert cm.Resample(16000, 22050, "sinc_interp_kaiser").beta == 14.769656459379492
    t1, _, _, _, _ = resample_table(16000, 22050, "sinc_interp_kaiser", beta=8.0)
    t2, _, _, _, _ = resample_table(16000, 22050, "sinc_interp_kaiser")
    assert not torch.equal(t1, t2)


def test_table_is_a_non_persistent_buffer():
    r = cm.Resample(48000, 22050)
    assert list(r.state_dict()) == [] and {n for n, _ in r.named_buffers()} == {"table", "first"}


def test_forward_argument_checks():
    r = cm.Resample(48000, 22050)
    x = torch.zeros(3, 2000)
    for bad in ([2000, 2000], [2001, 600, 600], [0, 600, 600], [600.0, 600, 600]):
        with pytest.raises((ValueError, TypeError)):
            r(x, lengths=bad)
    with pytest.raises(ValueError):
        r(torch.zeros(2, 2, 600))
    with pytest.raises(RuntimeError, match="CUDA"):
        r(x)
    with pytest.raises(RuntimeError, match="CUDA"):
        r(x, lengths=[2000, 1, 5])
    with pytest.raises(TypeError):
        r(x, lengths=torch.tensor([2000.0, 1.0, 5.0]))
    assert ops.resample_lengths(x, [1, 2000, 7]) == [1, 2000, 7]
    # more than 2**31 - 1 output samples: refused before anything is allocated (an expanded input holds no memory)
    with pytest.raises(ValueError, match="2\\*\\*31"):
        cm.Resample(22050, 48000)(torch.zeros(1).expand(1_000_000_000))


def _wav(tmp_path, name, sr, n=4000):
    f = tmp_path / name
    wav_write(str(f), torch.zeros(1, n), sr)
    return str(f)


def _error(verb, argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main([verb] + argv)
    assert e.value.code == 2
    return capsys.readouterr().err


def test_cli_resample_flags_parse(tmp_path, capsys):
    wav = _wav(tmp_path, "a.wav", 16000)
    out = str(tmp_path / "out")
    assert "--output-rate" in _error("vocode", ["x.pt", out, wav, "--output-rate", "0"], capsys)
    for verb in ("vocode", "score"):
        with pytest.raises(SystemExit) as e:
            cli.main([verb, "-h"])
        assert e.value.code == 0
        text = capsys.readouterr().out
        assert "--resample" in text
        if verb == "vocode":
            assert "--output-rate" in text and "--sampling-rate" in text
        else:
            assert "resampled signal" in " ".join(text.split())


def test_cli_refusal_without_resample_names_both_rates_and_the_flag(tmp_path, capsys):
    from tests.test_frontend_host import _nvidia_checkpoint
    wav = _wav(tmp_path, "a.wav", 16000)
    ck = _nvidia_checkpoint(tmp_path)
    for verb, extra in (("vocode", [str(tmp_path / "out")]), ("score", [])):
        err = _error(verb, [ck] + extra + [wav], capsys)
        assert "16000 Hz" in err and "22050 Hz" in err and "--resample" in err


def test_cli_reads_wavs_at_other_rates_with_resample(tmp_path):
    import argparse
    wav = _wav(tmp_path, "a.wav", 48000, 4801)
    x, sr = cli._read_wav_mono(wav, 22050, argparse.ArgumentParser(), resample=True)
    assert sr == 48000 and x.shape == (4801,)
    same = [torch.zeros(5)]
    assert cli._resample_batches(same, [22050], 22050, 4, torch.device("cpu"))[0] is same[0]
