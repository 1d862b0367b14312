"""bench.py's command line and its --dump-outputs files (host logic only)."""
import os
import sys

import numpy as np
import pytest
import torch

import bench
import constant_memory_waveglow_b200 as cm


def _model_with_grads(seed):
    torch.manual_seed(seed)
    m = cm.WaveGlow(4, 8, 2, 2, 16, 8, True, zero_init=False, dilation_channels=8, residual_channels=8,
                    skip_channels=8, depth=1)
    for p in m.parameters():
        p.grad = torch.randn_like(p)
    return m


def _read(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_files_and_positions(tmp_path, monkeypatch):
    m = _model_with_grads(0)
    bench.dump_outputs(str(tmp_path / "full"), m, torch.tensor(1.25))
    full = _read(tmp_path / "full")
    assert set(full) == {"loss.npy", "grad_sample.npy", "param_sample.npy"}
    assert full["loss.npy"].dtype == np.float64 and full["loss.npy"].shape == () and full["loss.npy"] == 1.25
    assert full["grad_sample.npy"].dtype == full["param_sample.npy"].dtype == np.float32
    # every tensor of this model is smaller than the per-tensor sample: the files hold all of it, in parameter order
    assert all(p.numel() <= bench.DUMP_SAMPLE_PER_TENSOR for p in m.parameters())
    assert np.array_equal(full["param_sample.npy"], torch.cat([p.detach().reshape(-1) for p in m.parameters()]).numpy())
    assert np.array_equal(full["grad_sample.npy"], torch.cat([p.grad.reshape(-1) for p in m.parameters()]).numpy())

    # sampled tensors: the positions depend on the shapes alone, so a doubled model state reads back exactly doubled
    monkeypatch.setattr(bench, "DUMP_SAMPLE_PER_TENSOR", 100)
    bench.dump_outputs(str(tmp_path / "a"), m, torch.tensor(1.25))
    with torch.no_grad():
        for p in m.parameters():
            p.mul_(2)
            p.grad.mul_(2)
    bench.dump_outputs(str(tmp_path / "b"), m, torch.tensor(2.5))
    a, b = _read(tmp_path / "a"), _read(tmp_path / "b")
    n = sum(min(p.numel(), 100) for p in m.parameters())
    assert a["param_sample.npy"].shape == a["grad_sample.npy"].shape == (n,) and n < full["param_sample.npy"].size
    for f in a:
        assert np.array_equal(2 * a[f], b[f]), f


def test_dump_outputs_refuses_more_than_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    with pytest.raises(AssertionError, match="exceed"):
        bench.dump_outputs(str(tmp_path / "d"), _model_with_grads(0), torch.tensor(1.0))
    assert os.listdir(tmp_path / "d") == []


@pytest.mark.parametrize("argv", [["--gpus", "1", "--steps", "0", "--warmup", "1"],
                                  ["--impl", "reference", "--ref-task", "parity"]])
def test_command_line_is_checked_before_any_work(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    monkeypatch.setattr(bench, "run_b200", lambda args: pytest.fail("ran"))
    monkeypatch.setattr(bench, "run_reference", lambda args: pytest.fail("ran"))
    with pytest.raises(SystemExit):
        bench.main()
