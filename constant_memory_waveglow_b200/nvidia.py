"""NVIDIA's published WaveGlow (NVIDIA/waveglow ``glow.py``; the DeepLearningExamples checkpoint ``torch.hub`` serves).

The flow is the package's WaveGlow -- invertible 1x1 conv, affine coupling, the same WN layers, gate order, residual / skip
split and early outputs -- with three differences that this module absorbs:

* conditioning: a dense ``ConvTranspose1d(80, 80, 1024, stride=256)`` with bias at the sample rate, unfolded by
  ``n_group`` into 640 channels at the squeezed rate.  With 16-bit operands it runs as one tcgen05 GEMM that writes the
  WN conditioning slab directly (``cmwg_nvidia_upsample_slab``), once per call, shared by all flows; in fp32 (the exact
  engine) as ``cmwg_upsample_dense_fwd`` + unfold + ``cmwg_cond_pack``;
* a bias on every WN conv (``WN(..., bias=True)``: the layered pipeline);
* key names, and the row order of the ``end`` conv: NVIDIA's gives ``[b, log_s]``, this package's ``[log_s, t]``.

``load_nvidia_waveglow`` reads the checkpoint forms in circulation without running code from them.
"""
from __future__ import annotations

import collections
import io
import os
import pickle
import types
import warnings
import zipfile
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib as L
from . import ops, precision
from .base import FlowBase
from .efficient_modules import AffineCouplingBlock, InvertibleConv1x1
from .waveglow import WN, CondSlab, WaveGlow, pack_generation

HOP = 256        # NVIDIA's upsampler: ConvTranspose1d(n_mel, n_mel, 1024, stride=256)
UP_KERNEL = 1024


class NvidiaWaveGlow(WaveGlow):
    """NVIDIA's WaveGlow, built with NVIDIA's constructor arguments; inference only.

    ``forward(x, h, lengths=None)``, ``reverse(z, h, lengths=None)`` and ``infer(h, sigma, z=None, lengths=None)`` keep the
    package's contracts: audio (B, T) with T a multiple of ``n_group``, a per-item log-det, ``lengths`` in samples (frames for
    ``infer``) and zero tails.  ``infer`` gives ``frames * 256`` samples, NVIDIA's ``infer`` (which trims the last 768 samples
    of the upsampled mel).  With autograd enabled every entry point raises ``NotImplementedError``.

    Load NVIDIA's checkpoints with ``load_nvidia_waveglow``; state-dict keys here are this package's (``WNs.k.F.V`` for
    NVIDIA's ``WN.k.cond_layer`` and so on)."""

    def __init__(self, n_mel_channels: int = 80, n_flows: int = 12, n_group: int = 8, n_early_every: int = 4,
                 n_early_size: int = 2, WN_config: Optional[dict] = None):
        FlowBase.__init__(self, HOP, False)
        cfg = {"n_layers": 8, "n_channels": 256, "kernel_size": 3}
        cfg.update(WN_config or {})
        if HOP % n_group:
            raise ValueError(f"NvidiaWaveGlow: n_group={n_group} must divide the hop {HOP}")
        self.n_group, self.n_early_every, self.n_early_size = n_group, n_early_every, n_early_size
        self.n_mels = n_mel_channels
        self.mem_efficient = False
        self.upsample = nn.ConvTranspose1d(n_mel_channels, n_mel_channels, UP_KERNEL, stride=HOP)
        self.invconv1x1 = nn.ModuleList()
        self.WNs = nn.ModuleList()
        remaining = n_group
        self.z_split_sizes = []
        for k in range(n_flows):
            if k % n_early_every == 0 and k:
                remaining -= n_early_size
                self.z_split_sizes.append(n_early_size)
            self.invconv1x1.append(InvertibleConv1x1(remaining))
            self.WNs.append(AffineCouplingBlock(WN, memory_efficient=False, in_channels=remaining // 2,
                                                aux_channels=n_mel_channels * n_group,
                                                dilation_channels=cfg["n_channels"], residual_channels=cfg["n_channels"],
                                                skip_channels=cfg["n_channels"], depth=cfg["n_layers"],
                                                radix=cfg["kernel_size"], bias=True))
        self.z_split_sizes.append(remaining)
        self._ups_pack: Dict[str, tuple] = {}

    def _upsample_h(self, h):
        raise NotImplementedError("NvidiaWaveGlow: the conditioning is built by _conditioning")

    def _require_no_grad(self, x: Tensor, h: Tensor, what: str) -> None:
        if torch.is_grad_enabled() and (x.requires_grad or h.requires_grad or any(p.requires_grad for p in self.parameters())):
            raise NotImplementedError(f"{what}: NvidiaWaveGlow is inference only; run under torch.no_grad()")

    # ---- conditioning ----------------------------------------------------------------------------------------------
    def _packed_upsampler(self, prec: str) -> Tensor:
        """The upsampler weight as the GEMM's B operand (cmwg_nvidia_upsample_pack), re-packed when the weight changed."""
        w = self.upsample.weight
        key = (pack_generation(), w.data_ptr(), w._version, w.device)
        ent = self._ups_pack.get(prec)
        if ent is not None and ent[0] == key:
            return ent[1]
        lib = L.load()
        C_, _, K = w.shape
        buf = torch.empty(int(lib.cmwg_nvidia_upsample_packed_bytes(C_, HOP, K // HOP)), device=w.device, dtype=torch.uint8)
        L.check(lib.cmwg_nvidia_upsample_pack(w.detach().contiguous().data_ptr(), C_, HOP, K // HOP, self.n_group,
                                              L.PREC_NAMES[prec], buf.data_ptr(), L.stream_ptr(w.device)),
                "nvidia_upsample_pack")
        self._ups_pack[prec] = (key, buf)
        return buf

    def _conditioning(self, h: Tensor, Tq: int, prec: str):
        """Conditioning of Tq squeezed steps: channel c of step t is up[c // n_group, n_group t + c % n_group], up = the
        upsampled mel.  A CondSlab for the 16-bit engines, the (B, n_mels * n_group, Tq) fp32 tensor for the exact one."""
        lib = L.load()
        B, Cm, F = h.shape
        up = self.upsample
        if Tq * self.n_group > (F - 1) * HOP + UP_KERNEL:
            raise ValueError(f"NvidiaWaveGlow: {Tq * self.n_group} samples need more than the {F} mel frames given")
        bias = up.bias.detach().float().contiguous()
        if prec == "fp32":
            Tout = (F - 1) * HOP + UP_KERNEL
            y = torch.empty((B, Cm, Tout), device=h.device, dtype=torch.float32)
            ws = torch.empty(int(lib.cmwg_upsample_dense_workspace(Cm, UP_KERNEL)), device=h.device, dtype=torch.uint8)
            w = up.weight.detach().float().contiguous()
            L.check(lib.cmwg_upsample_dense_fwd(h.data_ptr(), None, w.data_ptr(), bias.data_ptr(), B, Cm, F, UP_KERNEL, HOP,
                                                0, 0, 1.0, y.data_ptr(), ws.data_ptr(), L.stream_ptr(h.device)),
                    "upsample_dense_fwd")
            g = self.n_group
            return y[..., :Tq * g].reshape(B, Cm, Tq, g).permute(0, 1, 3, 2).reshape(B, Cm * g, Tq)
        packed = self._packed_upsampler(prec)
        width = Cm * self.n_group
        slab = torch.empty((B * Tq * width,), device=h.device, dtype=torch.int16)
        ws = torch.empty(int(lib.cmwg_nvidia_upsample_workspace_bytes(B, Tq, Cm, HOP, UP_KERNEL // HOP, self.n_group)),
                         device=h.device, dtype=torch.uint8)
        L.check(lib.cmwg_nvidia_upsample_slab(packed.data_ptr(), bias.data_ptr(), h.data_ptr(), h.stride(0), h.stride(1),
                                              B, Cm, F, HOP, UP_KERNEL // HOP, self.n_group, Tq, L.PREC_NAMES[prec],
                                              slab.data_ptr(), ws.data_ptr(), L.stream_ptr(h.device)),
                "nvidia_upsample_slab")
        return CondSlab(slab, (B, width, Tq), prec)

    def _prepare(self, x: Tensor, h: Tensor, lens: Optional[List[int]]):
        """The arguments of the direct loop: squeezed input, conditioning, the squeezed lengths (host, device) or (None,
        None), and the WN precision, resolved once because the conditioning is built in it."""
        L.require_cuda(x, h, op="NvidiaWaveGlow")
        if h.shape[1] != self.n_mels:
            raise ValueError(f"NvidiaWaveGlow: expected {self.n_mels} mel channels, got {h.shape[1]}")
        x = x.float()
        h = h.float()
        cols = None
        if lens is not None:
            # zero frames add nothing to the transposed conv: each item's conditioning equals its own call's
            frames = torch.tensor([-(-n // HOP) for n in lens], device=h.device)
            h = torch.where(torch.arange(h.shape[2], device=h.device)[None, None, :] < frames[:, None, None], h, 0.)
            x = torch.where(torch.arange(x.shape[1], device=x.device)[None, :] <
                            torch.tensor(lens, device=x.device)[:, None], x, 0.)
            cols = [n // self.n_group for n in lens]
        cols_host, cols_dev = ops.lengths_arg(cols, x.device)
        h = h.contiguous()
        xs = ops.squeeze(x.contiguous(), self.n_group, False)
        prec = precision.resolve(self.WNs[0].F._tc_supported(), training=False)
        return xs, self._conditioning(h, xs.shape[2], prec), cols_host, cols_dev, prec

    def _lens(self, x: Tensor, h: Tensor, lengths, what: str) -> Optional[List[int]]:
        self._require_no_grad(x, h, what)
        if x.dim() != 2 or h.dim() != 3 or h.shape[0] != x.shape[0]:
            raise ValueError(f"{what}: expected x (B, T) and h (B, n_mels, frames), got {tuple(x.shape)} and {tuple(h.shape)}")
        if x.shape[1] % self.n_group:
            raise ValueError(f"{what}: {x.shape[1]} samples is not a multiple of n_group={self.n_group}")
        if lengths is None:
            return None
        lens = self._check_lengths(x, h, lengths, what)
        return lens if any(n != x.shape[1] for n in lens) else None   # all full: the ordinary call, same bits

    def _direct_inputs(self, x: Tensor, h: Tensor, lengths, what: str):
        """Every call takes the direct loop, with per-item lengths or without."""
        return self._prepare(x, h, self._lens(x, h, lengths, what))


# ---------------------------------------------------------------------------------------------------------------------
# checkpoints
# ---------------------------------------------------------------------------------------------------------------------
class _PickledModule:
    """Stand-in for a class named in a pickled NVIDIA model: unpickling only records the object's state dict."""

    def __setstate__(self, state):
        self.state = state


_STUB_NAMES = ("glow.WaveGlow", "glow.WN", "glow.Invertible1x1Conv", "torch.nn.modules.conv.Conv1d",
               "torch.nn.modules.conv.ConvTranspose1d", "torch.nn.modules.container.ModuleList",
               "torch.nn.utils.weight_norm.WeightNorm")
_STUBS = {n: type(n.rsplit(".", 1)[1], (_PickledModule,), {"__module__": __name__}) for n in _STUB_NAMES}


def _no_backend():
    """Stand-in for torch.nn.backends.thnn._get_thnn_function_backend: every module pickled by torch 1.0-1.4 (the era of
    NVIDIA's published checkpoints, written in the legacy format) carries a `_backend` attribute that unpickles through
    it.  torch's own version is a no-op kept for these pickles; this one returns None without importing anything."""
    return None


# names a checkpoint may use besides the stubs and what tensors are built from
_FUNCTIONS = {"torch.nn.backends.thnn._get_thnn_function_backend": _no_backend}


class _RestrictedUnpickler(pickle.Unpickler):
    """Unpickler of the legacy (pre-zip) format that resolves only the allowlisted names: the stubs and what tensors and
    state dicts are built from.  torch's weights_only reader refuses this format's records of a pickled module's class."""
    _ALLOWED = dict(_STUBS, **_FUNCTIONS, **{"collections.OrderedDict": collections.OrderedDict, "builtins.set": set,
                               "__builtin__.set": set, "torch._utils._rebuild_tensor_v2": torch._utils._rebuild_tensor_v2,
                               "torch._utils._rebuild_parameter": torch._utils._rebuild_parameter})

    def find_class(self, module, name):
        obj = self._ALLOWED.get(f"{module}.{name}")
        if obj is None:
            raise pickle.UnpicklingError(f"load_nvidia_waveglow: the checkpoint names {module}.{name}, which is not allowed")
        return obj


def _read_checkpoint(path_or_file):
    """torch.load(weights_only=True) with the stubs allowed; a legacy-format file that pickles module classes goes
    through the same allowlist in _RestrictedUnpickler (torch's legacy reader, storages restored on the CPU)."""
    data = path_or_file.read() if hasattr(path_or_file, "read") else open(path_or_file, "rb").read()
    allowed = [(obj, name) for name, obj in {**_STUBS, **_FUNCTIONS}.items()] + [set]
    with torch.serialization.safe_globals(allowed):
        try:
            return torch.load(io.BytesIO(data), map_location="cpu", weights_only=True)
        except pickle.UnpicklingError:
            if zipfile.is_zipfile(io.BytesIO(data)):
                raise
    module = types.SimpleNamespace(Unpickler=_RestrictedUnpickler, __name__="restricted_pickle",
                                   load=lambda f, **kw: _RestrictedUnpickler(f, **kw).load())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # the class source saved in the file is not compared with the stubs
        return torch.serialization._legacy_load(io.BytesIO(data), "cpu", module)


def _flatten(obj: _PickledModule, prefix: str, out: Dict[str, Tensor]) -> None:
    st = obj.state
    for name, t in st.get("_parameters", {}).items():
        if t is not None:
            out[prefix + name] = t
    for name, t in st.get("_buffers", {}).items():
        if t is not None:
            out[prefix + name] = t
    for name, m in st.get("_modules", {}).items():
        if m is not None:
            _flatten(m, prefix + name + ".", out)


def nvidia_state_dict(ckpt) -> Dict[str, Tensor]:
    """NVIDIA-keyed state dict from any of the three checkpoint forms (already unpickled)."""
    if isinstance(ckpt, dict) and isinstance(ckpt.get("model"), _PickledModule):
        out: Dict[str, Tensor] = {}
        _flatten(ckpt["model"], "", out)
        return out
    sd = ckpt["state_dict"] if isinstance(ckpt, dict) and isinstance(ckpt.get("state_dict"), dict) else ckpt
    if not isinstance(sd, dict) or not all(isinstance(v, Tensor) for v in sd.values()):
        raise ValueError("load_nvidia_waveglow: expected {'model': WaveGlow}, {'state_dict': ...} or a state dict")
    return {(k[len("module."):] if k.startswith("module.") else k): v for k, v in sd.items()}


def _conv(sd: Dict[str, Tensor], src: str) -> Dict[str, Tensor]:
    """Parameters of conv `src` (weight_g / weight_v or plain weight, and bias) keyed by their local names."""
    return {n: sd[src + n] for n in ("weight_g", "weight_v", "weight", "bias") if src + n in sd}


def _cond_layer(sd: Dict[str, Tensor], src: str, n_layers: int) -> Dict[str, Tensor]:
    if src + "cond_layer.bias" in sd:
        return _conv(sd, src + "cond_layer.")
    # per-layer cond_layers.i: weight norm is per output channel, so stacking the layers in order is exact
    parts = [_conv(sd, f"{src}cond_layers.{i}.") for i in range(n_layers)]
    return {n: torch.cat([p[n] for p in parts], 0) for n in parts[0]}


def convert_state_dict(sd: Dict[str, Tensor]) -> Tuple[dict, Dict[str, Tensor]]:
    """(constructor arguments of NvidiaWaveGlow, package-keyed state dict) from an NVIDIA-keyed state dict; every
    dimension is read from the tensor shapes."""
    n_flows = 0
    while f"convinv.{n_flows}.conv.weight" in sd:
        n_flows += 1
    if n_flows == 0 or "upsample.weight" not in sd:
        raise ValueError("load_nvidia_waveglow: no NVIDIA WaveGlow weights (convinv.*.conv.weight, upsample.weight) found")
    n_mel = sd["upsample.weight"].shape[0]
    if tuple(sd["upsample.weight"].shape) != (n_mel, n_mel, UP_KERNEL):
        raise ValueError(f"load_nvidia_waveglow: upsample weight {tuple(sd['upsample.weight'].shape)} is not "
                         f"({n_mel}, {n_mel}, {UP_KERNEL})")
    sizes = [sd[f"convinv.{k}.conv.weight"].shape[0] for k in range(n_flows)]
    n_group = sizes[0]
    drops = [(k, sizes[k - 1] - sizes[k]) for k in range(1, n_flows) if sizes[k] != sizes[k - 1]]
    n_early_every = drops[0][0] if drops else n_flows
    n_early_size = drops[0][1] if drops else 2
    n_layers = 0
    while f"WN.0.in_layers.{n_layers}.bias" in sd:
        n_layers += 1
    w0 = _conv(sd, "WN.0.in_layers.0.")
    w0 = w0.get("weight_v", w0.get("weight"))
    cfg = dict(n_mel_channels=n_mel, n_flows=n_flows, n_group=n_group, n_early_every=n_early_every,
               n_early_size=n_early_size,
               WN_config=dict(n_layers=n_layers, n_channels=w0.shape[1], kernel_size=w0.shape[2]))
    out = {"upsample.weight": sd["upsample.weight"], "upsample.bias": sd["upsample.bias"]}
    for k in range(n_flows):
        out[f"invconv1x1.{k}.weight"] = sd[f"convinv.{k}.conv.weight"]
        src, dst = f"WN.{k}.", f"WNs.{k}.F."
        pieces = {"V.": _cond_layer(sd, src, n_layers), "start.": _conv(sd, src + "start.")}
        for i in range(n_layers):
            pieces[f"layers.{i}.W."] = _conv(sd, f"{src}in_layers.{i}.")
            pieces[f"layers.{i}.W_o."] = _conv(sd, f"{src}res_skip_layers.{i}.")
        end = _conv(sd, src + "end.")
        for n, t in end.items():   # [b, log_s] -> [log_s, t]
            half = t.shape[0] // 2
            end[n] = torch.cat((t[half:], t[:half]), 0)
        pieces["end."] = end
        for p, params in pieces.items():
            for n, t in params.items():
                out[dst + p + n] = t
    return cfg, out


def load_nvidia_waveglow(path_or_obj, device="cuda") -> NvidiaWaveGlow:
    """An NvidiaWaveGlow with the weights of an NVIDIA WaveGlow checkpoint, in eval mode on `device`.

    Accepts a path or file object, or an already loaded object, of: the pickled ``{'model': glow.WaveGlow}`` of NVIDIA/waveglow
    (zip or legacy serialization), DeepLearningExamples' ``{'state_dict': ...}`` (``module.`` prefixes), or a plain state
    dict; weight-normed (``weight_g`` / ``weight_v``) or plain weights; one ``cond_layer`` or per-layer ``cond_layers``.
    Files are read without running code from them: only tensors, containers and stand-ins for NVIDIA's module classes are
    unpickled."""
    if isinstance(path_or_obj, (str, os.PathLike)) or hasattr(path_or_obj, "read"):
        path_or_obj = _read_checkpoint(path_or_obj)
    cfg, sd = convert_state_dict(nvidia_state_dict(path_or_obj))
    model = NvidiaWaveGlow(**cfg)
    if not any(k.endswith("weight_g") for k in sd):
        from .utils import remove_weight_norms
        model.apply(remove_weight_norms)
    model.load_state_dict({k: v.float() for k, v in sd.items()})
    return model.to(device).eval()
