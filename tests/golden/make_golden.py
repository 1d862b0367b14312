"""Generate golden fixtures by running the UNMODIFIED reference (CPU, fp32).

Run in the authoring container only (``/root/reference`` does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference is imported from ``/root/reference`` with an in-memory stub for the missing
``pytorch_lightning`` module (only ``model/lightning.py`` needs it; none of the flow code does).
Every fixture stores the seeded inputs, the reference state-dict, the reference outputs and the
gradients produced by the reference's *memory-efficient* (constant-memory) path, so the oracle
(and through it the CUDA product) is pinned against the real reversible backward.
"""
import os
import sys
import types
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
REF = os.environ.get("CMWG_REFERENCE", "/root/reference")
OUT = os.path.dirname(os.path.abspath(__file__))


def import_reference():
    pl = types.ModuleType("pytorch_lightning")

    class _LM(torch.nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

    pl.LightningModule = _LM
    pl.Callback = object
    pl.Trainer = object
    sys.modules["pytorch_lightning"] = pl
    # the reference must win over this repo's drop-in ``model`` package
    sys.path.insert(0, REF)
    for name in list(sys.modules):
        if name == "model" or name.startswith("model.") or name == "utils":
            del sys.modules[name]
    from model.efficient_modules import AffineCouplingBlock, InvertibleConv1x1
    from model.waveglow import WN, WaveGlow
    from model.loss import WaveGlowLoss
    assert sys.modules["model.waveglow"].__file__.startswith(REF)
    return AffineCouplingBlock, InvertibleConv1x1, WN, WaveGlow, WaveGlowLoss


def set_seed(seed):
    np.random.seed(seed)
    torch.manual_seed(seed)


def cpu_state(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def main():
    torch.set_num_threads(4)
    AffineCouplingBlock, InvertibleConv1x1, WN, WaveGlow, WaveGlowLoss = import_reference()

    # ---- 1. invertible 1x1 conv, both directions, efficient mode --------------------------------
    for c in (2, 4, 8):
        set_seed(100 + c)
        B, T = 3, 257
        m = InvertibleConv1x1(c, True)
        sd = cpu_state(m)
        x = torch.rand(B, c, T) * 2 - 1
        loss_fn = WaveGlowLoss(0.7)
        fx = {"state": sd, "x": x, "sigma": 0.7}
        for direction in ("forward", "reverse"):
            m.zero_grad()
            xin = x.clone().requires_grad_(True)
            xc = xin.clone()
            y, ld = (m(xc) if direction == "forward" else m.reverse(xc))
            loss = loss_fn(y.reshape(B, -1), ld)
            loss.backward()
            fx[direction] = {"out": y.detach().clone(), "logdet": ld.detach().clone(),
                             "loss": loss.detach().clone(), "dx": xin.grad.clone(),
                             "dweight": m.weight.grad.clone()}
        torch.save(fx, os.path.join(OUT, f"conv1x1_c{c}.pt"))

    # ---- 2. affine coupling block with WN transform --------------------------------------------
    for name, ch, wn_ch, depth, aux, T in (("a", 16, 32, 2, 20, 300), ("b", 8, 32, 3, 12, 211)):
        set_seed(7 + depth)
        B = 2
        kw = dict(in_channels=ch // 2, aux_channels=aux, zero_init=False, dilation_channels=wn_ch,
                  residual_channels=wn_ch, skip_channels=wn_ch, depth=depth)
        m = AffineCouplingBlock(WN, True, **kw)
        sd = cpu_state(m)
        x = torch.rand(B, ch, T) * 2 - 1
        y = torch.randn(B, aux, T)
        loss_fn = WaveGlowLoss(1.0)
        fx = {"state": sd, "x": x, "y": y, "kwargs": kw, "param_order": [n for n, _ in m.F.named_parameters()]}
        for direction in ("forward", "reverse"):
            m.zero_grad()
            xin = x.clone().requires_grad_(True)
            yin = y.clone().requires_grad_(True)
            xc = xin.clone()
            out, ls = (m(xc, yin) if direction == "forward" else m.reverse(xc, yin))
            loss = loss_fn(out.reshape(B, -1), ls.sum((1, 2)))
            loss.backward()
            fx[direction] = {"out": out.detach().clone(), "log_s": ls.detach().clone(),
                             "loss": loss.detach().clone(), "dx": xin.grad.clone(), "dy": yin.grad.clone(),
                             "dparams": {"F." + n: p.grad.clone() for n, p in m.F.named_parameters()}}
        torch.save(fx, os.path.join(OUT, f"coupling_{name}.pt"))

    # ---- 3. tiny WaveGlow: forward, loss, reversible backward, reverse, infer ---------------------
    set_seed(0)
    arch = dict(flows=4, n_group=8, n_early_every=2, n_early_size=2, hop_size=256, n_mels=8)
    wkw = dict(dilation_channels=32, residual_channels=32, skip_channels=32, depth=3, radix=3,
               bias=False, zero_init=False)
    B, T, frames = 2, 2048, 8
    m = WaveGlow(memory_efficient=True, **arch, **wkw)
    sd = cpu_state(m)
    x = torch.rand(B, T) * 2 - 1
    h = torch.randn(B, arch["n_mels"], frames)
    loss_fn = WaveGlowLoss(0.7)
    m.zero_grad()
    z, logdet = m(x.clone(), h)
    loss = loss_fn(z, logdet)
    loss.backward()
    grads = {n: p.grad.clone() for n, p in m.named_parameters()}
    with torch.no_grad():
        m2 = WaveGlow(memory_efficient=False, **arch, **wkw)
        m2.load_state_dict(sd)
        xr, logdet_r = m2.reverse(z.detach().clone(), h)
        zs = torch.randn(B, frames * arch["hop_size"]) * 0.6
        audio, _ = m2.reverse_computation(zs.clone(), h)
    torch.save({"state": sd, "arch": arch, "wn_kwargs": wkw, "x": x, "h": h, "sigma": 0.7,
                "z": z.detach().clone(), "logdet": logdet.detach().clone(), "loss": loss.detach().clone(),
                "grads": grads, "x_roundtrip": xr, "logdet_reverse": logdet_r,
                "infer_z": zs, "infer_audio": audio},
               os.path.join(OUT, "waveglow_tiny.pt"))
    # ---- 4. WSRGlow 2x (model/wsrglow.py): weights come from the oracle's seeded generator (the state is
    # ~45 MB, too big for a fixture), the REFERENCE model computes outputs and gradients -------------------
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from oracle import flow_oracle as O
    from model.wsrglow import WSRGlow
    assert sys.modules["model.wsrglow"].__file__.startswith(REF)
    gen_args = dict(upsample_rate=2, wn_channels=64, depth=2, seed=5)
    sdw = O.wsrglow_random_state(**gen_args)
    wkw = dict(dilation_channels=64, residual_channels=64, skip_channels=64, depth=2, radix=3, bias=False,
               zero_init=False)
    set_seed(11)
    B, T = 2, 2048
    x = torch.rand(B, T) * 2 - 1
    c = torch.rand(B, T // 2) * 2.2 - 1.1          # a few samples outside [-1, 1]: exercises the clip
    m = WSRGlow(upsample_rate=2, memory_efficient=True, **wkw)
    missing = m.load_state_dict(sdw, strict=True)
    m.zero_grad()
    cond = m._get_cond(c.clone()).detach().clone()
    z, logdet = m(x.clone(), c.clone())
    loss = WaveGlowLoss(0.7)(z, logdet)
    loss.backward()
    grads = {n: p.grad.clone() for n, p in m.named_parameters()}
    # full gradients only for the embeddings, the upsampler, the 1x1 convs and flows 0 / 5 / 11 (minus V.weight_v);
    # every other tensor is pinned through its norm
    keep = {n: g for n, g in grads.items()
            if not n.endswith("V.weight_v") and g.numel() <= 130000 and
            (not n.startswith("WNs.") or n.split(".")[1] in ("0", "5", "11"))}
    with torch.no_grad():
        m2 = WSRGlow(upsample_rate=2, memory_efficient=False, **wkw)
        m2.load_state_dict(sdw)
        xr, _ = m2.reverse(z.detach().clone(), c.clone())
    torch.save({"gen_args": gen_args, "wn_kwargs": wkw, "x": x, "c": c, "sigma": 0.7,
                "state_keys": list(m.state_dict().keys()),
                "cond_sum": cond.double().sum(), "cond_abs_sum": cond.double().abs().sum(),
                "cond_sample": cond[:, ::61, ::7].clone(),
                "z": z.detach().clone(), "logdet": logdet.detach().clone(), "loss": loss.detach().clone(),
                "grads": {n: g for n, g in keep.items() if not n.startswith("WNs.")},
                "grad_norms": {n: g.double().norm() for n, g in grads.items()},
                "x_roundtrip": xr},
               os.path.join(OUT, "wsrglow_tiny.pt"))
    # the flows' gradients in a file of their own, to keep each fixture under 1 MB (tests/_util.load_wsrglow_golden)
    torch.save({n: g for n, g in keep.items() if n.startswith("WNs.")}, os.path.join(OUT, "wsrglow_tiny_wn_grads.pt"))
    # ---- 5. tiny WaveFlow (model/waveflow.py): forward, loss, plain-autograd backward, row-recurrent reverse ------
    from model.waveflow import WaveFlow
    assert sys.modules["model.waveflow"].__file__.startswith(REF)
    for tag, ng, conv in (("a", 32, False), ("b", 16, True)):
        set_seed(21 + ng)
        arch = dict(flows=2, n_group=ng, n_mels=8, use_conv1x1=conv)
        wkw = dict(dilation_channels=16, residual_channels=16, skip_channels=16, bias=False, zero_init=False)
        B, frames = 2, 3
        T = frames * 256
        m = WaveFlow(memory_efficient=False, **arch, **wkw)
        sd = cpu_state(m)
        x = torch.rand(B, T) * 2 - 1
        h = torch.randn(B, arch["n_mels"], frames)
        m.zero_grad()
        z, logdet = m(x.clone(), h)
        loss = WaveGlowLoss(0.7)(z, logdet)
        loss.backward()
        grads = {n: p.grad.clone() for n, p in m.named_parameters()}
        with torch.no_grad():
            xr, logdet_r = m.reverse(z.detach().clone(), h)
            zs = torch.randn(B, T) * 0.6
            audio, logdet_s = m.reverse_computation(zs.clone(), h)
            up = m._upsample_h(h).clone()
        torch.save({"state": sd, "arch": arch, "wn_kwargs": wkw, "x": x, "h": h, "sigma": 0.7,
                    "upsampled": up, "z": z.detach().clone(), "logdet": logdet.detach().clone(),
                    "loss": loss.detach().clone(), "grads": grads, "x_roundtrip": xr, "logdet_reverse": logdet_r,
                    "infer_z": zs, "infer_audio": audio, "infer_logdet": logdet_s},
                   os.path.join(OUT, f"waveflow_tiny_{tag}.pt"))
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".pt"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
