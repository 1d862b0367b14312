"""WN transform and the WaveGlow model: host-side mirror of the reference's ``model/waveglow.py``.

Same class names, constructor signatures, attribute names and state-dict keys as the reference
(``fused_gate`` :13-15, ``NonCausalLayer`` :18-46, ``WN`` :49-105, ``WaveGlow`` :108-212), so
checkpoints, ``train.py``, ``inference.py`` and ``tests/test_fwd_bwd.py`` work unchanged.  The
modules only OWN parameters; the arithmetic runs in libcmwg_b200.so:

  WN.forward        -> cmwg_wn_pack (once per weight version) + cmwg_cond_pack (once per conditioning
                       tensor, shared by all flows) + cmwg_wn_forward / cmwg_wn_backward
  WaveGlow glue     -> cmwg_upsample_*, cmwg_squeeze, cmwg_sum_per_batch
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib as L
from . import ops, precision
from .base import FlowBase, Lengths, lengths_list
from .efficient_modules import AffineCouplingBlock, InvertibleConv1x1, grad_hint, graph_possible
from .parallel import grad_buffer
from .utils import add_weight_norms


def fused_gate(x1: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
    """tanh(x1) * sigmoid(x2) (reference ``model/waveglow.py:13-15``).  Kept for importers
    (``waveflow`` / ``melglow`` style transforms); WN's own gate runs inside the GEMM epilogue."""
    return x1.tanh() * x2.sigmoid()


class NonCausalLayer(nn.Module):
    """Parameter container of one WN layer (reference ``model/waveglow.py:18-46``): ``W`` dilated
    conv Cr -> 2*Cd (kernel ``radix``, padding = dilation*(radix-1)//2) and ``W_o`` 1x1 conv
    Cd -> Cr+Cs (last layer: Cd -> Cs)."""

    def __init__(self, dilation, dilation_channels, residual_channels, skip_channels, radix, bias,
                 last_layer=False):
        super().__init__()
        self.W = nn.Conv1d(residual_channels, dilation_channels * 2, kernel_size=radix,
                           padding=dilation * (radix - 1) // 2, dilation=dilation, bias=bias)
        out_ch = skip_channels if last_layer else residual_channels + skip_channels
        self.W_o = nn.Conv1d(dilation_channels, out_ch, 1, bias=bias)
        self.chs_split = [skip_channels] if last_layer else [residual_channels, skip_channels]

    def forward(self, x, y):
        # Generic per-layer entry for external transforms that reuse this class; WN itself never
        # calls it (its layers run fused in cmwg_wn_forward).
        zw, zf = (self.W(x) + y).chunk(2, 1)
        out = self.W_o(fused_gate(zw, zf))
        if len(self.chs_split) == 2:
            res, skip = out.split(self.chs_split, 1)
            return res + x, skip
        return None, out


# ---------------------------------------------------------------------------------------------
# conditioning cache: the slab-layout copy of y is built once and reused by all flows / recomputes
# ---------------------------------------------------------------------------------------------
class CondSlab:
    """Conditioning already in the slab layout ``cmwg_cond_pack`` writes ([B*T][auxp], the operand type of `prec`), for a
    model that produces it directly (NvidiaWaveGlow's upsampler GEMM).  The WN entry points take it in place of the
    (B, aux, T) fp32 tensor; `shape` is that tensor's shape."""
    __slots__ = ("data", "shape", "prec")

    def __init__(self, data: Tensor, shape: Tuple[int, int, int], prec: str):
        self.data, self.shape, self.prec = data, tuple(shape), prec


class _CondCache:
    def __init__(self, capacity: int = 3):
        self.capacity = capacity
        self.entries: "OrderedDict[tuple, tuple]" = OrderedDict()

    def get(self, y: Tensor, cfg: L.WnConfig) -> Tensor:
        auxp = L.load().cmwg_wn_aux_padded(C.byref(cfg))
        if isinstance(y, CondSlab):
            if L.PREC_NAMES[y.prec] != cfg.precision or y.data.numel() != y.shape[0] * y.shape[2] * auxp:
                raise RuntimeError(f"WN: conditioning slab of precision {y.prec} and {y.data.numel()} elements does not "
                                   f"match this WN ({auxp} padded channels, precision code {cfg.precision})")
            return y.data
        key = (y.untyped_storage().data_ptr(), y.storage_offset(), tuple(y.shape), tuple(y.stride()), y._version,
               auxp, cfg.precision, y.device.index)
        hit = self.entries.get(key)
        if hit is not None:
            # the constant-memory ops release a tensor's memory with storage.resize_(0) while the tensor object lives on, so
            # holding `y` does not pin its address: the entry is valid only while the held tensor still owns the keyed memory
            st = hit[0].untyped_storage()
            if st.data_ptr() == key[0] and st.size() > 0:
                self.entries.move_to_end(key)
                return hit[1]
            del self.entries[key]
        B, aux, T = y.shape
        elem = torch.float32 if cfg.precision == L.PREC_FP32 else torch.int16
        ycl = torch.empty((B, T, auxp), device=y.device, dtype=elem)
        L.check(L.load().cmwg_cond_pack(C.byref(cfg), y.data_ptr(), y.stride(0), y.stride(1), y.stride(2), B, T,
                                        ycl.data_ptr(), L.stream_ptr(y.device)), "cond_pack")
        self.entries[key] = (y, ycl)
        while len(self.entries) > self.capacity:
            self.entries.popitem(last=False)
        return ycl

    def clear(self):
        self.entries.clear()


_cond_cache = _CondCache()


# ---------------------------------------------------------------------------------------------
# Weight-pack invalidation.  A pack (effective weights after weight norm, re-laid-out as GEMM operands) is keyed on
# (address, version counter) of every parameter -- but in-place updates that bypass the version counter exist and are
# common: torch's FUSED optimizers (`Adam(..., fused=True)` leaves `p._version` untouched), `p.data.copy_(...)`, EMA
# swaps.  So the key also carries a process-wide generation number that every optimizer step bumps (a global
# optimizer-step post hook), that `load_state_dict` / `.to()` / `.cuda()` bump through the module hooks below, and that
# user code which edits `.data` directly can bump with `invalidate_packs()`.
# ---------------------------------------------------------------------------------------------
_pack_generation = [0]


def invalidate_packs() -> None:
    """Force every WN to re-pack its weights at its next call (and WaveFlow to drop its captured synthesis graphs)."""
    _pack_generation[0] += 1


def pack_generation() -> int:
    return _pack_generation[0]


try:
    from torch.optim.optimizer import register_optimizer_step_post_hook as _reg_post
    _reg_post(lambda _opt, _args, _kwargs: invalidate_packs())
except Exception:  # pragma: no cover  (very old torch: fall back to the version counters alone)
    pass


class _WNState:
    """What one fused WN forward leaves behind for its backward."""
    __slots__ = ("cfg", "packed", "params", "ycl", "saved", "B", "T", "prec")


class WN(nn.Module):
    """WaveNet-style transform (reference ``model/waveglow.py:49-105``).

    forward(x, y) -> (log_s, t): ``start`` 1x1, ``V`` conditioning 1x1 for all layers, ``depth``
    NonCausalLayers with dilation 2^i accumulating skips, ``end`` 1x1 (no weight norm, zero-init
    unless ``zero_init=False``).  Parameter registration order (V, start, layers, end) is the
    reference's, which fixes ``parameters()`` order and therefore the gradient order the coupling
    Functions return.
    """
    _cmwg_fused = True  # AffineCouplingBlock engages the fused kernels for this transform type

    def __init__(self, in_channels, aux_channels, dilation_channels=256, residual_channels=256,
                 skip_channels=256, depth=8, radix=3, bias=False, zero_init=True):
        super().__init__()
        self.dilations = [2 ** i for i in range(depth)]
        self.in_chs = in_channels
        self.aux_chs = aux_channels
        self.res_chs = residual_channels
        self.dil_chs = dilation_channels
        self.skp_chs = skip_channels
        self.rdx = radix
        self.has_bias = bool(bias)
        self.r_field = sum(self.dilations) + 1

        self.V = nn.Conv1d(aux_channels, dilation_channels * 2 * depth, 1, bias=bias)
        self.V.apply(add_weight_norms)
        self.start = nn.Conv1d(in_channels, residual_channels, 1, bias=bias)
        self.start.apply(add_weight_norms)
        self.layers = nn.ModuleList(
            NonCausalLayer(d, dilation_channels, residual_channels, skip_channels, radix, bias,
                           last_layer=(i == depth - 1)) for i, d in enumerate(self.dilations))
        self.layers.apply(add_weight_norms)
        self.end = nn.Conv1d(skip_channels, in_channels * 2, 1, bias=bias)
        if zero_init:
            self.end.weight.data.zero_()
            if bias:
                self.end.bias.data.zero_()
        self._pack_cache = {}

    # ---- parameter plumbing ------------------------------------------------------------------
    def _convs(self):
        yield "V", self.V
        yield "start", self.start
        for i, layer in enumerate(self.layers):
            yield ("W", i), layer.W
            yield ("W_o", i), layer.W_o
        yield "end", self.end

    @staticmethod
    def _gvb(mod):
        if hasattr(mod, "weight_g"):
            return mod.weight_g, mod.weight_v, mod.bias
        return None, mod.weight, mod.bias

    def _config(self, prec: str, height: int = 0) -> L.WnConfig:
        return L.WnConfig(self.in_chs, self.aux_chs, self.dil_chs, self.res_chs, self.skp_chs, len(self.layers),
                          self.rdx, int(self.has_bias), L.PREC_NAMES[prec])

    def _params_struct(self) -> L.WnParams:
        ps = L.WnParams()
        for key, mod in self._convs():
            g, v, b = self._gvb(mod)
            for t in (g, v, b):
                if t is not None and (not t.is_contiguous() or t.dtype != torch.float32):
                    raise RuntimeError("cmwg_b200: WN parameters must be contiguous fp32 tensors")
            cp = L.ConvParam(L.ptr(g), L.ptr(v), L.ptr(b))
            if isinstance(key, tuple):
                getattr(ps, key[0])[key[1]] = cp
            else:
                setattr(ps, key, cp)
        return ps

    def _tc_supported(self) -> bool:
        return bool(L.load().cmwg_wn_tc_supported(C.byref(self._config("fp32"))))

    def _prepare(self, prec: str, device, height: int = 0):
        """(cfg, packed weights, params struct) for `prec`; re-packs only when a parameter changed."""
        params = list(self.parameters())
        L.require_cuda(*params, op="WN")
        cfg = self._config(prec, height)
        key = (_pack_generation[0],) + tuple((p.data_ptr(), p._version) for p in params)
        ent = self._pack_cache.get(prec)
        ps = self._params_struct()
        if ent is not None and ent[0] == key and ent[1].device == device:
            return cfg, ent[1], ps
        nbytes = int(L.load().cmwg_wn_packed_bytes(C.byref(cfg)))
        if nbytes == 0:
            L.check(-1, "wn_packed_bytes")
        buf = ent[1] if (ent is not None and ent[1].numel() == nbytes and ent[1].device == device) else \
            torch.empty(nbytes, device=device, dtype=torch.uint8)
        L.check(L.load().cmwg_wn_pack(C.byref(cfg), C.byref(ps), buf.data_ptr(), L.stream_ptr(device)), "wn_pack")
        self._pack_cache[prec] = (key, buf)   # one entry per precision: captured CUDA graphs and stored-mode states keep
        return cfg, buf, ps                   # pointing at the buffer of THEIR precision

    def _apply(self, fn, *args, **kwargs):          # .to() / .cuda() / .float(): parameters are replaced or rewritten
        invalidate_packs()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):   # load_state_dict copies into .data without a version bump guarantee
        invalidate_packs()
        return super()._load_from_state_dict(*args, **kwargs)

    # ---- scratch: per (device, stream, purpose) buffers that persist between calls ---------------------------------
    # The kernels address every slab through TMA descriptors that the library caches by ADDRESS; a fresh torch.empty per
    # call lands wherever the caching allocator has room, and a step whose workspaces land on new addresses re-encodes a few
    # thousand descriptors (60-100 ms once measured).  Work on one stream is ordered, so one buffer per stream is safe.
    _scratch: dict = {}
    _SCRATCH_MAX = 6 << 30     # larger requests (long-utterance batches) are not kept

    @classmethod
    def _scratch_buf(cls, nbytes: int, device, purpose: str) -> Tensor:
        if nbytes > cls._SCRATCH_MAX or torch.cuda.is_current_stream_capturing():
            # too large to keep, or a CUDA graph is being captured (its allocations belong to the graph's private pool)
            return torch.empty(nbytes, device=device, dtype=torch.uint8)
        key = (device.index, torch.cuda.current_stream(device).cuda_stream, purpose)
        buf = cls._scratch.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(nbytes, device=device, dtype=torch.uint8)
            cls._scratch[key] = buf
        return buf

    # ---- fused entry points used by the coupling Functions --------------------------------------
    def _cmwg_forward(self, x: Tensor, y: Tensor, save: bool, prec: Optional[str] = None, transient: bool = False):
        """x: (B, >=cin, T) NCL whose first `cin` channels are the WN input.  Returns (lst, state):
        lst (B, 2cin, T) = [log_s ; t].  `transient`: the saved activations are consumed by a `_cmwg_backward` call that
        follows immediately (the constant-memory recompute), so they may live in the per-stream scratch buffer."""
        L.require_cuda(x, y.data if isinstance(y, CondSlab) else y, op="WN.forward")
        if prec is None:
            prec = precision.resolve(self._tc_supported(), training=save)
        cfg, packed, ps = self._prepare(prec, x.device)
        lib = L.load()
        x = ops._ncl(x)
        B, _, T = x.shape
        if y.shape[0] != B or y.shape[1] != self.aux_chs or y.shape[2] != T:
            raise RuntimeError(f"WN: conditioning shape {tuple(y.shape)} does not match input {(B, self.aux_chs, T)}")
        if not isinstance(y, CondSlab) and y.dtype != torch.float32:
            y = y.float()
        ycl = _cond_cache.get(y, cfg)
        ws = self._scratch_buf(int(lib.cmwg_wn_workspace_bytes(C.byref(cfg), B, T)), x.device, "ws")
        saved = None
        if save:
            nsv = int(lib.cmwg_wn_saved_bytes(C.byref(cfg), B, T))
            saved = self._scratch_buf(nsv, x.device, "saved") if transient else \
                torch.empty(nsv, device=x.device, dtype=torch.uint8)
        lst = torch.empty((B, 2 * self.in_chs, T), device=x.device, dtype=torch.float32)
        L.check(lib.cmwg_wn_forward(C.byref(cfg), packed.data_ptr(), x.data_ptr(), ops._bstride(x), ycl.data_ptr(), B, T,
                                    ws.data_ptr(), L.ptr(saved), lst.data_ptr(), L.stream_ptr(x.device)), "wn_forward")
        st = _WNState()
        st.cfg, st.packed, st.params, st.ycl, st.saved, st.B, st.T, st.prec = cfg, packed, ps, ycl, saved, B, T, prec
        return lst, st

    def _cmwg_forward_varlen(self, x: Tensor, y: Tensor, lengths_host, lengths_dev: Tensor, prec: str) -> Tensor:
        """Inference over a padded batch: lst (B, 2cin, T) whose columns t < lengths[b] equal the WN of item b alone
        (cmwg_wn_forward_varlen); lengths_host is a ctypes int array, lengths_dev the same values as a device int32 tensor."""
        L.require_cuda(x, y.data if isinstance(y, CondSlab) else y, op="WN.forward")
        cfg, packed, _ = self._prepare(prec, x.device)
        lib = L.load()
        x = ops._ncl(x)
        B, _, T = x.shape
        if y.shape[0] != B or y.shape[1] != self.aux_chs or y.shape[2] != T:
            raise RuntimeError(f"WN: conditioning shape {tuple(y.shape)} does not match input {(B, self.aux_chs, T)}")
        ycl = _cond_cache.get(y if isinstance(y, CondSlab) or y.dtype == torch.float32 else y.float(), cfg)
        ws = self._scratch_buf(int(lib.cmwg_wn_varlen_workspace_bytes(C.byref(cfg), B, T)), x.device, "ws")
        lst = torch.empty((B, 2 * self.in_chs, T), device=x.device, dtype=torch.float32)
        L.check(lib.cmwg_wn_forward_varlen(C.byref(cfg), packed.data_ptr(), x.data_ptr(), ops._bstride(x), ycl.data_ptr(),
                                           B, T, lengths_host, lengths_dev.data_ptr(), ws.data_ptr(), lst.data_ptr(),
                                           L.stream_ptr(x.device)), "wn_forward_varlen")
        return lst

    def _grads_struct(self):
        """(cmwg_wn_grads, {id(param): destination tensor}); destinations are views of the data-parallel
        communication buffers when available."""
        grads = L.WnGrads()
        by_param = {}
        for key, mod in self._convs():
            g, v, b = self._gvb(mod)
            dg = grad_buffer(g) if g is not None else None
            dv = grad_buffer(v)
            db = grad_buffer(b) if b is not None else None
            cg = L.ConvGrad(L.ptr(dg), L.ptr(dv), L.ptr(db))
            if isinstance(key, tuple):
                getattr(grads, key[0])[key[1]] = cg
            else:
                setattr(grads, key, cg)
            for p, d in ((g, dg), (v, dv), (b, db)):
                if p is not None:
                    by_param[id(p)] = d
        return grads, by_param

    def _cmwg_backward(self, st: _WNState, x: Tensor, dlst: Tensor, dx: Tensor, need_dy: bool):
        """Accumulates d(xa) into dx[:, :cin]; returns (grads in self.parameters() order, dy or None)."""
        lib = L.load()
        x = ops._ncl(x)
        dlst = dlst.contiguous()
        dev = x.device
        grads, by_param = self._grads_struct()
        aux_p = lib.cmwg_wn_aux_padded(C.byref(st.cfg))
        dycl = torch.empty((st.B, st.T, aux_p), device=dev, dtype=torch.float32) if need_dy else None
        ws = self._scratch_buf(int(lib.cmwg_wn_workspace_bytes(C.byref(st.cfg), st.B, st.T)), dev, "ws")
        L.check(lib.cmwg_wn_backward(C.byref(st.cfg), C.byref(st.params), st.packed.data_ptr(), x.data_ptr(),
                                     ops._bstride(x), st.ycl.data_ptr(), st.B, st.T, ws.data_ptr(),
                                     st.saved.data_ptr(), dlst.data_ptr(), dx.data_ptr(), ops._bstride(dx),
                                     L.ptr(dycl), C.byref(grads), L.stream_ptr(dev)), "wn_backward")
        dy = None
        if need_dy:
            dy = torch.empty((st.B, self.aux_chs, st.T), device=dev, dtype=torch.float32)
            L.check(lib.cmwg_cond_unpack_grad(C.byref(st.cfg), dycl.data_ptr(), st.B, st.T, dy.data_ptr(),
                                              L.stream_ptr(dev)), "cond_unpack_grad")
        return [by_param[id(p)] for p in self.parameters()], dy

    def forward(self, x, y):
        with grad_hint():
            lst = _WNFunction.apply(x, y, self, *self.parameters())
        return lst.chunk(2, 1)


class _WNFunction(torch.autograd.Function):
    """WN as an ordinary (activation-storing) autograd node: what the reference's naive mode gets
    from autograd over ``WN.forward``."""

    @staticmethod
    def forward(ctx, x, y, wn, *params):
        need = any(ctx.needs_input_grad) and graph_possible()
        xd = ops._ncl(x.detach())
        lst, st = wn._cmwg_forward(xd, y.detach(), save=need)
        ctx.wn, ctx.st = wn, st
        ctx.save_for_backward(xd)
        ctx.y_shape = y.shape
        return lst

    @staticmethod
    def backward(ctx, dlst):
        (x,) = ctx.saved_tensors
        wn, st = ctx.wn, ctx.st
        dx = torch.zeros_like(x, memory_format=torch.contiguous_format)
        grads, dy = wn._cmwg_backward(st, x, dlst, dx, need_dy=ctx.needs_input_grad[1])
        ctx.st = None
        return (dx if ctx.needs_input_grad[0] else None, dy, None) + tuple(grads)


# ---------------------------------------------------------------------------------------------
# WaveGlow glue ops with autograd
# ---------------------------------------------------------------------------------------------
class _UpsampleFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, g, v, bias, stride, pad):
        ctx.save_for_backward(h, g, v)
        ctx.params = (g, v, bias)
        ctx.stride, ctx.pad, ctx.has_bias = stride, pad, bias is not None
        return ops.upsample_fwd(h.detach(), None if g is None else g.detach(), v.detach(),
                                None if bias is None else bias.detach(), stride, pad)

    @staticmethod
    def backward(ctx, dy):
        h, g, v = ctx.saved_tensors
        dh = None
        if ctx.needs_input_grad[0]:  # trainable conditioning (WSRGlow's embedding tables)
            dh = ops.upsample_bwd_input(g, v, dy, h.shape[2], ctx.stride, ctx.pad)
        pg, pv, pb = ctx.params
        out = (grad_buffer(pg) if pg is not None else None, grad_buffer(pv), grad_buffer(pb) if pb is not None else None)
        dg, dv, db = ops.upsample_bwd(h, g, v, dy, ctx.stride, ctx.pad, ctx.has_bias, out=out)
        return dh, dg, dv, db, None, None


class _SqueezeFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, n_group, inverse):
        ctx.n_group, ctx.inverse = n_group, inverse
        return ops.squeeze(x.detach(), n_group, inverse)

    @staticmethod
    def backward(ctx, g):
        return ops.squeeze(g, ctx.n_group, not ctx.inverse), None, None


class _SumPerBatch(torch.autograd.Function):
    """log_s.sum((1, 2)) of ``model/waveglow.py:175``."""

    @staticmethod
    def forward(ctx, a):
        ctx.shape = a.shape
        return ops.sum_per_batch(a.detach())

    @staticmethod
    def backward(ctx, g):
        return g.view(-1, 1, 1).expand(ctx.shape)


class _LogdetAccumulate(torch.autograd.Function):
    """``logdet + log_det_W + log_s.sum((1, 2))`` of ``model/waveglow.py:175,199`` as one kernel (three launches as torch ops)."""

    @staticmethod
    def forward(ctx, prev, log_det_w, log_s):
        ctx.shape = log_s.shape
        ctx.has_prev = prev is not None
        return ops.logdet_accumulate(log_s.detach(), prev, log_det_w)

    @staticmethod
    def backward(ctx, g):
        # every flow of the chain receives the SAME cotangent tensor: its batch sum (the cotangent of the 0-dim log_det_W)
        # is formed once and handed down the chain with it
        gs = getattr(g, "_cmwg_batch_sum", None)
        if gs is None:
            gs = g.sum()
            try:
                g._cmwg_batch_sum = gs
            except Exception:  # pragma: no cover
                pass
        return (g if ctx.has_prev else None), (gs if ctx.needs_input_grad[1] else None), g.view(-1, 1, 1).expand(ctx.shape)


class WaveGlow(FlowBase):
    """Reference ``model/waveglow.py:108-212``: upsampler, squeeze, ``flows`` x (invertible 1x1 conv ->
    affine coupling with WN), early outputs every ``n_early_every`` flows.

    ``forward(x, h, lengths=...)`` / ``reverse(z, h, lengths=...)`` run a zero-padded batch of different-length items in one
    call (inference only): ``lengths`` are valid SAMPLES per item, multiples of ``n_group``.  Item b then gets exactly what
    the call on ``(x[b, :len_b], h[b, :, :ceil(len_b / hop)])`` alone gives on its valid samples (bit for bit in fp32 and
    fp16), zeros after them, and a log-det over its valid samples only."""
    _supports_lengths = True

    def __init__(self, flows, n_group, n_early_every, n_early_size, hop_size, n_mels, memory_efficient,
                 reverse_mode=False, **kwargs):
        super().__init__(hop_size, reverse_mode)
        self.n_group = n_group
        self.n_early_every = n_early_every
        self.n_early_size = n_early_size
        self.n_mels = n_mels
        self.mem_efficient = memory_efficient

        self.upsample_factor = self._hop_length // n_group
        sub_win_size = self.upsample_factor * 2 + 1
        self.upsampler = nn.ConvTranspose1d(n_mels, n_mels, sub_win_size, self.upsample_factor,
                                            padding=sub_win_size // 2 - self.upsample_factor // 2, groups=n_mels)
        self.upsampler.apply(add_weight_norms)

        self.invconv1x1 = nn.ModuleList()
        self.WNs = nn.ModuleList()
        remaining = n_group
        self.z_split_sizes = []
        for k in range(flows):
            if k % self.n_early_every == 0 and k:
                remaining -= n_early_size
                self.z_split_sizes.append(n_early_size)
            self.invconv1x1.append(InvertibleConv1x1(remaining, memory_efficient=memory_efficient,
                                                     reverse_mode=reverse_mode))
            self.WNs.append(AffineCouplingBlock(WN, memory_efficient=memory_efficient, in_channels=remaining // 2,
                                                aux_channels=n_mels, reverse_mode=reverse_mode, **kwargs))
        self.z_split_sizes.append(remaining)

    def _upsample_h(self, h):
        up = self.upsampler
        g, v, b = WN._gvb(up)
        return _UpsampleFunction.apply(h, g, v, b, up.stride[0], up.padding[0])

    # ---- per-item lengths (inference on a padded batch) -------------------------------------------------------------
    def _check_lengths(self, x: Tensor, h: Tensor, lengths: Lengths, what: str) -> List[int]:
        if x.dim() != 2 or h.dim() != 3 or h.shape[0] != x.shape[0]:
            raise ValueError(f"{what}: expected x (B, T) and h (B, n_mels, frames), got {tuple(x.shape)} and {tuple(h.shape)}")
        B, T = x.shape
        lens = lengths_list(lengths, B, what, "samples")
        for n in lens:
            if not 1 <= n <= T or n % self.n_group:
                raise ValueError(f"{what}: length {n} must be a multiple of n_group={self.n_group} in [1, {T}] "
                                 "(lengths are in samples here; FlowBase.infer takes mel frames)")
        if torch.is_grad_enabled() and (x.requires_grad or h.requires_grad or any(p.requires_grad for p in self.parameters())):
            raise NotImplementedError(f"{what}: per-item lengths are inference only; run under torch.no_grad() "
                                      "(training on variable-length batches is not supported)")
        return lens

    def _varlen_prepare(self, x: Tensor, h: Tensor, lens: List[int]):
        """x and h with their padding zeroed -> the squeezed input, the upsampled conditioning and the per-item lengths in
        squeezed columns (host ctypes array and device int32 tensor)."""
        L.require_cuda(x, h, op="WaveGlow")
        B, T = x.shape
        hop = self._hop_length
        frames = [-(-n // hop) for n in lens]
        t_idx = torch.arange(T, device=x.device)
        f_idx = torch.arange(h.shape[2], device=h.device)
        len_t = torch.tensor(lens, device=x.device)
        x = torch.where(t_idx[None, :] < len_t[:, None], x.float(), 0.)
        # a zero frame adds nothing to the transposed conv, so the upsampled conditioning equals the item's own on its samples
        h = torch.where(f_idx[None, None, :] < torch.tensor(frames, device=h.device)[:, None, None], h.float(), 0.)
        up = self.upsampler
        g, v, b = WN._gvb(up)
        y = ops.upsample_fwd(h, g, v, b, up.stride[0], up.padding[0])
        xs = ops.squeeze(x, self.n_group, False)
        assert xs.size(2) <= y.size(2)
        y = y[..., :xs.size(2)]
        cols = [n // self.n_group for n in lens]
        cols_host = (C.c_int * B)(*cols)
        cols_dev = torch.tensor(cols, dtype=torch.int32).to(x.device)
        return xs, y, cols_host, cols_dev

    # One flow's two steps on a padded batch.  `inverse` is the direction the model asks for; a module built with
    # reverse_mode=True swaps it (Reversible._direction), exactly as the ordinary path's module calls do.
    def _varlen_conv(self, k: int, x: Tensor, inverse: bool) -> Tuple[Tensor, Tensor]:
        conv = self.invconv1x1[k]
        inv = inverse != bool(conv._reverse_mode)
        w2 = conv.weight.detach().reshape(conv.weight.shape[0], -1).float().contiguous()
        winv, ld = ops.small_inverse_logdet(w2)
        return ops.conv1x1_apply(winv if inv else w2, x), (-ld if inv else ld)

    def _varlen_coupling(self, k: int, x: Tensor, y: Tensor, cols_host, cols_dev: Tensor,
                         inverse: bool) -> Tuple[Tensor, Tensor]:
        coup = self.WNs[k]
        inv = inverse != bool(coup._reverse_mode)
        F = coup.F
        lst = F._cmwg_forward_varlen(x, y, cols_host, cols_dev, precision.resolve(F._tc_supported(), training=False))
        z, neg_log_s = ops.coupling_apply_varlen(x, lst, cols_dev, inverse=inv)
        return z, (neg_log_s if inv else lst[:, :F.in_chs])

    def _forward_varlen(self, x: Tensor, h: Tensor, lens: List[int]) -> Tuple[Tensor, Tensor]:
        batch = x.size(0)
        x, y, cols_host, cols_dev = self._varlen_prepare(x, h, lens)
        early: List[Tensor] = []
        logdet = None
        for k in range(len(self.WNs)):
            if k % self.n_early_every == 0 and k:
                e, x = x.split([self.n_early_size, x.size(1) - self.n_early_size], 1)
                early.append(e)
            x, ldw = self._varlen_conv(k, x, False)
            x, log_s = self._varlen_coupling(k, x, y, cols_host, cols_dev, False)
            logdet = ops.logdet_accumulate_varlen(log_s, cols_dev, logdet, ldw)
        early.append(x)
        z = ops.squeeze(torch.cat(early, 1), self.n_group, True)
        return z.view(batch, -1), logdet

    def _reverse_varlen(self, z: Tensor, h: Tensor, lens: List[int]) -> Tuple[Tensor, Tensor]:
        batch = z.size(0)
        z, y, cols_host, cols_dev = self._varlen_prepare(z, h, lens)
        parts = list(z.split(self.z_split_sizes, 1))
        z = parts.pop()
        logdet = None
        for k in range(len(self.WNs) - 1, -1, -1):
            z, log_s = self._varlen_coupling(k, z, y, cols_host, cols_dev, True)
            z, ldw = self._varlen_conv(k, z, True)
            logdet = ops.logdet_accumulate_varlen(log_s, cols_dev, logdet, ldw)
            if k % self.n_early_every == 0 and k:
                z = torch.cat((parts.pop(), z), 1)
        x = ops.squeeze(z, self.n_group, True)
        return x.view(batch, -1), logdet

    def forward_computation(self, x: Tensor, h: Tensor, lengths: Optional[Lengths] = None) -> Tuple[Tensor, Tensor]:
        if lengths is not None:
            lens = self._check_lengths(x, h, lengths, "WaveGlow.forward")
            if any(n != x.shape[1] for n in lens):   # all lengths == T: the ordinary call, same bits
                return self._forward_varlen(x, h, lens)
        L.require_cuda(x, h, op="WaveGlow.forward")
        y = self._upsample_h(h)
        batch = x.size(0)
        x = _SqueezeFunction.apply(x, self.n_group, False)
        assert x.size(2) <= y.size(2)
        y = y[..., :x.size(2)]

        early: List[Tensor] = []
        logdet = None
        for k, (invconv, coup) in enumerate(zip(self.invconv1x1, self.WNs)):
            if k % self.n_early_every == 0 and k:
                e, x = x.split([self.n_early_size, x.size(1) - self.n_early_size], 1)
                early.append(e)
                if self.mem_efficient:
                    x = x.clone()  # the efficient ops consume (free) their input
            x, log_det_w = invconv(x)
            x, log_s = coup(x, y)
            logdet = _LogdetAccumulate.apply(logdet, log_det_w, log_s)
        early.append(x)
        z = _SqueezeFunction.apply(torch.cat(early, 1), self.n_group, True)
        return z.view(batch, -1), logdet

    def reverse_computation(self, z: Tensor, h: Tensor, lengths: Optional[Lengths] = None) -> Tuple[Tensor, Tensor]:
        if lengths is not None:
            lens = self._check_lengths(z, h, lengths, "WaveGlow.reverse")
            if any(n != z.shape[1] for n in lens):
                return self._reverse_varlen(z, h, lens)
        L.require_cuda(z, h, op="WaveGlow.reverse")
        y = self._upsample_h(h)
        batch = z.size(0)
        z = _SqueezeFunction.apply(z, self.n_group, False)
        assert z.size(2) <= y.size(2)
        y = y[..., :z.size(2)]

        parts = list(z.split(self.z_split_sizes, 1))
        if self.mem_efficient:
            parts = [p.clone() for p in parts]
        z = parts.pop()
        logdet = None
        for k in range(len(self.WNs) - 1, -1, -1):
            z, log_s = self.WNs[k].reverse(z, y)
            z, log_det_w = self.invconv1x1[k].reverse(z)
            logdet = _LogdetAccumulate.apply(logdet, log_det_w, log_s)
            if k % self.n_early_every == 0 and k:
                z = torch.cat((parts.pop(), z), 1)
        x = _SqueezeFunction.apply(z, self.n_group, True)
        return x.view(batch, -1), logdet
