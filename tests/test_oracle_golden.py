"""The CPU oracle (oracle/flow_oracle.py) against the fixtures produced by the unmodified
reference (tests/golden/make_golden.py).  No GPU needed."""
import os

import pytest
import torch

from oracle import flow_oracle as O
from tests._util import load_wsrglow_golden

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)


def rel_l2(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("c", [2, 4, 8])
def test_conv1x1_against_reference(c):
    fx = load(f"conv1x1_c{c}.pt")
    w, x, sigma = fx["state"]["weight"], fx["x"], fx["sigma"]
    B = x.shape[0]
    for direction, fn in (("forward", O.conv1x1_forward), ("reverse", O.conv1x1_reverse)):
        ref = fx[direction]
        ww = w.clone().requires_grad_(True)
        xx = x.clone().requires_grad_(True)
        out, ld = fn(ww, xx)
        assert torch.allclose(out, ref["out"], atol=1e-6, rtol=1e-6)
        assert torch.allclose(ld, ref["logdet"], atol=1e-5, rtol=1e-6)
        loss = O.waveglow_loss(out.reshape(B, -1), ld, sigma)
        dw, dx = torch.autograd.grad(loss, [ww, xx])
        assert torch.allclose(loss, ref["loss"], rtol=1e-6)
        assert torch.allclose(dx, ref["dx"], atol=1e-9, rtol=1e-5)
        assert torch.allclose(dw, ref["dweight"], atol=5e-7, rtol=1e-5)
        # closed-form backward restatement
        dz = (out / (sigma ** 2 * B * out[0].numel())).detach()
        dl = torch.tensor(-1.0 / (out[0].numel()))
        if direction == "forward":
            dx2, dw2 = O.conv1x1_backward(w, x, dz, dl)
        else:
            dx2, dw2 = O.invconv1x1_backward(w, x, dz, dl)
        assert torch.allclose(dx2, ref["dx"], atol=1e-9, rtol=1e-5)
        assert torch.allclose(dw2, ref["dweight"], atol=5e-7, rtol=1e-4)
    # restore-input step of the reversible backward
    assert torch.allclose(O.conv1x1_restore_input(w, fx["forward"]["out"]), x, atol=1e-6)


@pytest.mark.parametrize("name", ["a", "b"])
def test_coupling_against_reference(name):
    fx = load(f"coupling_{name}.pt")
    sd, x, y = fx["state"], fx["x"], fx["y"]
    B = x.shape[0]
    n = x[0].numel()
    for direction in ("forward", "reverse"):
        ref = fx[direction]
        fn = O.coupling_reverse if direction == "reverse" else O.coupling_forward
        out, ls = fn(sd, "F.", x, y)
        assert torch.allclose(out, ref["out"], atol=1e-6, rtol=1e-5)
        assert torch.allclose(ls, ref["log_s"], atol=1e-6, rtol=1e-5)
        # loss = mean_b(0.5*sum z^2 - sum log_s)/n  -> cotangents
        dz = ref["out"] / (B * n)
        dls = torch.full_like(ls, -1.0 / (B * n))
        _, _, dx, dparams, dy = O.coupling_grads(sd, "F.", x, y, dz, dls, reverse=direction == "reverse",
                                                 need_dy=True)
        assert rel_l2(dx, ref["dx"]) < 1e-5
        assert rel_l2(dy, ref["dy"]) < 1e-5
        for k, g in ref["dparams"].items():
            assert rel_l2(dparams[k], g) < 2e-5, k
    # restore-input step (forward direction): x from z
    xr = O.coupling_restore_input(sd, "F.", fx["forward"]["out"], y)
    assert torch.allclose(xr, x, atol=1e-6)
    assert fx["param_order"][0] == "V.weight_g" and fx["param_order"][-1] == "end.weight"


def test_waveglow_tiny_against_reference():
    fx = load("waveglow_tiny.pt")
    sd = fx["state"]
    spec = O.WaveGlowSpec(**fx["arch"])
    z, logdet, loss, grads = O.waveglow_train_step(sd, spec, fx["x"], fx["h"], fx["sigma"])
    assert rel_l2(z, fx["z"]) < 1e-6
    # logdet is a cancelling sum of ~1e4 fp32 terms: order-of-summation noise is ~1e-6 relative
    assert rel_l2(logdet, fx["logdet"]) < 2e-5
    assert torch.allclose(loss, fx["loss"], rtol=1e-6)
    assert set(grads) == set(fx["grads"])
    for k, g in fx["grads"].items():
        assert rel_l2(grads[k], g) < 5e-5, k
    xr, ldr = O.waveglow_reverse(sd, spec, fx["z"], fx["h"])
    assert torch.allclose(xr, fx["x_roundtrip"], atol=2e-6)
    assert torch.allclose(xr, fx["x"], atol=1e-5)
    assert rel_l2(ldr, fx["logdet_reverse"]) < 2e-5
    audio = O.waveglow_infer(sd, spec, fx["h"], fx["infer_z"])
    assert torch.allclose(audio, fx["infer_audio"], atol=2e-6)


def test_spec_matches_reference_channel_schedule():
    spec = O.WaveGlowSpec(12, 8, 4, 2, 256, 80)
    assert spec.channels == [8] * 4 + [6] * 4 + [4] * 4
    assert spec.z_split_sizes == [2, 2, 4]
    assert spec.upsample_factor == 32 and spec.sub_win == 65 and spec.up_pad == 16


def test_random_state_has_reference_keys():
    fx = load("waveglow_tiny.pt")
    spec = O.WaveGlowSpec(**fx["arch"])
    sd = O.random_state(spec, 32, 3, seed=1)
    assert set(sd) == set(fx["state"])
    for k in sd:
        assert sd[k].shape == fx["state"][k].shape, k


def test_wsrglow_tiny_against_reference():
    """WSRGlow 2x (model/wsrglow.py): conditioning front end + flow, outputs and gradients from the
    unmodified reference; weights are regenerated from the seed the fixture records."""
    fx = load_wsrglow_golden()
    ga = fx["gen_args"]
    sd = O.wsrglow_random_state(**ga)
    assert list(sd.keys()) == fx["state_keys"] or set(sd.keys()) == set(fx["state_keys"])
    spec = O.wsrglow_spec(ga["upsample_rate"])
    assert spec.n_mels == 3659 and spec.n_group == 16 and spec.upsample_factor == 1 and spec.sub_win == 3
    cond = O.wsrglow_cond(sd, fx["c"])
    assert cond.shape == (2, 3659, 128)
    assert torch.allclose(cond[:, ::61, ::7], fx["cond_sample"], atol=1e-5)
    assert abs(cond.double().abs().sum().item() - fx["cond_abs_sum"].item()) < 1e-6 * fx["cond_abs_sum"].item()
    z, logdet, loss, grads = O.wsrglow_train_step(sd, spec, fx["x"], fx["c"], fx["sigma"])
    assert rel_l2(z, fx["z"]) < 1e-6
    assert rel_l2(logdet, fx["logdet"]) < 2e-5
    assert torch.allclose(loss, fx["loss"], rtol=1e-6)
    for k, g in fx["grads"].items():
        assert rel_l2(grads[k], g) < 5e-5, k
    for k, n in fx["grad_norms"].items():
        assert abs(grads[k].double().norm().item() - n.item()) < 1e-4 * max(n.item(), 1e-12), k
    xr, _ = O.wsrglow_reverse(sd, spec, fx["z"], fx["c"])
    assert torch.allclose(xr, fx["x_roundtrip"], atol=2e-6)
    assert torch.allclose(xr, fx["x"], atol=2e-5)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_waveflow_against_reference(tag):
    """WaveFlow (model/waveflow.py): 2-D WN forward, plain-autograd gradients, row-recurrent reverse."""
    fx = load(f"waveflow_tiny_{tag}.pt")
    sd, x, h = fx["state"], fx["x"], fx["h"]
    spec = O.WaveFlowSpec(**fx["arch"])
    assert torch.allclose(O.waveflow_upsample_h(sd, spec, h), fx["upsampled"], atol=1e-6, rtol=1e-6)
    z, logdet, loss, grads = O.waveflow_train_step(sd, spec, x, h, fx["sigma"])
    assert torch.allclose(z, fx["z"], atol=2e-6, rtol=1e-5)
    assert torch.allclose(logdet, fx["logdet"], atol=1e-4, rtol=1e-6)
    assert torch.allclose(loss, fx["loss"], rtol=1e-6)
    assert set(grads) == set(fx["grads"])
    for n, g in fx["grads"].items():
        # d start.weight_v is analytically zero (one input channel: w = g * sign(v)); only rounding noise is left
        tol = 1e-8 if n.endswith("start.weight_v") else 2e-5 * g.norm().item() + 1e-9
        assert (grads[n] - g).norm().item() <= tol, n
    xr, ldr = O.waveflow_reverse(sd, spec, fx["z"], h)
    assert torch.allclose(xr, fx["x_roundtrip"], atol=2e-6)
    assert torch.allclose(ldr, fx["logdet_reverse"], atol=1e-4, rtol=1e-6)
    assert torch.allclose(xr, x, atol=1e-5)
    audio, lds = O.waveflow_reverse(sd, spec, fx["infer_z"], h)
    assert torch.allclose(audio, fx["infer_audio"], atol=2e-6, rtol=1e-5)
    assert torch.allclose(lds, fx["infer_logdet"], atol=1e-4, rtol=1e-6)
    # the row-recurrent reverse equals running the full-image WN once per generated row (what the CUDA path does)
    zi = O.waveflow_squeeze(fx["infer_z"], spec.n_group)
    y = O.waveflow_upsample_h(sd, spec, h)[..., :zi.size(-1)]
    k = spec.flows - 1
    if not spec.use_conv1x1:
        zi = zi.flip(2)
    else:
        zi = O.conv1x1_reverse(sd[f"invconv1x1.{k}.weight"], zi.squeeze(1))[0].unsqueeze(1)
    img = zi.clone()
    for i in range(1, spec.n_group):
        ls, t = O.wn2d_forward(sd, f"WNs.{k}.", img[:, :, :i], y, spec.h_dilations)
        img[:, :, i] = (zi[:, :, i] - t[:, :, i - 1]) / ls[:, :, i - 1].exp()
    rows = [zi[:, :, :1]]
    cond = torch.nn.functional.conv1d(y, O.resolve_weight(sd, f"WNs.{k}.V.")).unsqueeze(2).chunk(8, 1)
    buffers, xnew = None, zi[:, :, :1]
    for i in range(1, spec.n_group):
        ls, t, buffers = O.wn2d_reverse_step(sd, f"WNs.{k}.", xnew, cond, buffers, spec.h_dilations)
        xnew = (zi[:, :, i:i + 1] - t) / ls.exp()
        rows.append(xnew)
    assert torch.allclose(img, torch.cat(rows, 2), atol=2e-6, rtol=1e-5)


def test_waveflow_random_state_layout():
    fx = load("waveflow_tiny_b.pt")
    spec = O.WaveFlowSpec(**fx["arch"])
    rs = O.waveflow_random_state(spec, 16, seed=3)
    assert list(sorted(rs)) == list(sorted(fx["state"]))
    for k, v in fx["state"].items():
        assert rs[k].shape == v.shape, k
