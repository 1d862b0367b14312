"""Model-level parity the reference's own tests lack: WaveGlow against the golden fixture of the unmodified reference and
against the CPU oracle, per precision mode.  Block level: chains of 1x1 convs and affine couplings with the constant-memory
backward against the same chains storing their activations (input storage freed and restored, gradients, invertibility),
the properties the reference's own tests/test_fwd_bwd.py checks."""
import pytest
import torch
from torch import nn

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import precision
from oracle import flow_oracle as O
from tests._util import TOL, load_golden, rel_l2, to_double

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _exact_mode():
    # tests/test_fwd_bwd.py:10-11 of the reference
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, precision.get_precision())
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    precision.set_precision("auto")
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old[0], old[1]
    precision.set_precision(old[2])


# ------------------------------------------------------------------------------------------------
# model level
# ------------------------------------------------------------------------------------------------
def test_waveglow_against_reference_golden():
    fx = load_golden("waveglow_tiny.pt")
    m = cm.WaveGlow(memory_efficient=True, **fx["arch"], **fx["wn_kwargs"])
    m.load_state_dict(fx["state"])
    m = m.cuda().train()
    x, h = fx["x"].cuda(), fx["h"].cuda()
    z, logdet = m(x.clone(), h)
    assert rel_l2(z, fx["z"]) < 5e-6, rel_l2(z, fx["z"])
    assert rel_l2(logdet, fx["logdet"]) < 5e-5
    loss = cm.WaveGlowLoss(fx["sigma"])(z, logdet)
    assert abs(loss.item() - fx["loss"].item()) < 1e-5 * abs(fx["loss"].item())
    loss.backward()
    for n, p in m.named_parameters():
        assert p.grad is not None, n
        assert rel_l2(p.grad, fx["grads"][n]) < 2e-4, (n, rel_l2(p.grad, fx["grads"][n]))
    with torch.no_grad():
        xr, ldr = m.reverse(z.detach().clone(), h)
        assert torch.allclose(xr.cpu(), fx["x"], atol=2e-5)
        assert rel_l2(ldr, fx["logdet_reverse"]) < 5e-5
        audio = m.infer(h, 0.6, z=fx["infer_z"].cuda())
        assert torch.allclose(audio.cpu(), fx["infer_audio"], atol=2e-5)
        m.apply(cm.remove_weight_norms)          # inference.py:17
        audio2 = m.infer(h, 0.6, z=fx["infer_z"].cuda())
        assert torch.allclose(audio2.cpu(), fx["infer_audio"], atol=2e-5)


@pytest.mark.parametrize("prec", ["fp32", "fp16", "bf16"])
def test_waveglow_128ch_against_oracle(prec):
    """Config 1b of SURVEY 8(d): 12 flows, 128 channels, depth 4, B=2, T=16000, sigma 0.7."""
    precision.set_precision(prec)
    spec = O.WaveGlowSpec(12, 8, 4, 2, 256, 80)
    sd = O.random_state(spec, 128, 4, seed=0)
    g = torch.Generator().manual_seed(0)
    x = torch.rand(2, 16000, generator=g) * 2 - 1
    h = torch.randn(2, 80, 63, generator=g)
    z_ref, ld_ref, loss_ref, grads_ref = O.waveglow_train_step(sd, spec, x, h, 0.7)
    m = cm.WaveGlow(12, 8, 4, 2, 256, 80, True, dilation_channels=128, residual_channels=128, skip_channels=128,
                    depth=4, zero_init=False)
    m.load_state_dict(sd)
    m = m.cuda().train()
    z, logdet = m(x.cuda(), h.cuda())
    loss = cm.WaveGlowLoss(0.7)(z, logdet)
    loss.backward()
    tol = TOL[prec]
    # the oracle here is fp32 (not fp64): allow its own round-off on top of ours
    assert rel_l2(z, z_ref) < max(tol["out"], 2e-5), rel_l2(z, z_ref)
    assert rel_l2(logdet, ld_ref) < max(tol["logdet"], 1e-4), rel_l2(logdet, ld_ref)
    num = den = 0.0
    for n, p in m.named_parameters():
        gr = grads_ref[n].double()
        num += (p.grad.double().cpu() - gr).pow(2).sum().item()
        den += gr.pow(2).sum().item()
    agg = (num / den) ** 0.5
    assert agg < max(tol["grad"], 2e-4), agg
    with torch.no_grad():
        xr, _ = m.reverse(z.detach().clone(), h.cuda())
    assert rel_l2(xr, x) < max(tol["roundtrip"], 2e-5), rel_l2(xr, x)


# ------------------------------------------------------------------------------------------------
# block level
# ------------------------------------------------------------------------------------------------
def _chain(efficient, reverse_mode, cin, aux, ch, depth):
    torch.manual_seed(0)
    return nn.ModuleList([m for _ in range(2) for m in (
        cm.InvertibleConv1x1(2 * cin, efficient, reverse_mode),
        cm.AffineCouplingBlock(cm.WN, efficient, reverse_mode, in_channels=cin, aux_channels=aux, zero_init=False,
                               dilation_channels=ch, residual_channels=ch, skip_channels=ch, depth=depth))]).cuda()


def _run(blocks, x, y, inverse=False):
    h, logdet = x, 0
    for b in (reversed(blocks) if inverse else blocks):
        args = (h, y) if isinstance(b, cm.AffineCouplingBlock) else (h,)
        h, ld = b.reverse(*args) if inverse else b(*args)
        logdet = logdet + ld.sum()
    return h, logdet


@pytest.mark.parametrize("reverse_mode", [False, True])
@pytest.mark.parametrize("cin,aux,ch,depth,B,T", [(4, 12, 32, 2, 2, 300), (8, 40, 128, 4, 2, 1000)])
def test_constant_memory_chain_matches_stored_activations(cin, aux, ch, depth, B, T, reverse_mode):
    """Two flows (1x1 conv -> affine coupling), so every block's freed input is the previous block's output: the
    constant-memory chain frees its input, restores it in the backward and gives the outputs and gradients of the chain
    that stores its activations; the inverse chain returns the input."""
    precision.set_precision("fp32")
    g = torch.Generator().manual_seed(1)
    x = (torch.rand(B, 2 * cin, T, generator=g) * 2 - 1).cuda()
    y = torch.randn(B, aux, T, generator=g).cuda()
    dz = torch.randn(B, 2 * cin, T, generator=g).cuda()
    stored = _chain(False, reverse_mode, cin, aux, ch, depth)
    res = {}
    for efficient in (False, True):
        blocks = stored if not efficient else _chain(True, reverse_mode, cin, aux, ch, depth)
        blocks.load_state_dict(stored.state_dict())
        xg, yg = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        xin = xg.clone()
        z, logdet = _run(blocks, xin, yg)
        assert (xin.untyped_storage().size() == 0) == efficient          # only the constant-memory chain frees it
        ((z * dz).sum() + logdet).backward()
        assert xin.untyped_storage().size() > 0 and rel_l2(xin, x) < 1e-5  # restored in place by the backward
        with torch.no_grad():
            xr, ldr = _run(blocks, z.detach().clone(), y, inverse=True)
        assert rel_l2(xr, x) < 1e-5 and abs(ldr.item() + logdet.item()) < 1e-4 * max(abs(logdet.item()), 1.0)
        res[efficient] = dict(z=z.detach(), logdet=logdet.detach(), dx=xg.grad, dy=yg.grad,
                              **{n: p.grad for n, p in blocks.named_parameters()})
    for k, want in res[False].items():
        got = res[True][k]
        assert got is not None and want is not None, k
        assert rel_l2(got, want) < 2e-5, (k, rel_l2(got, want))
