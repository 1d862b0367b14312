"""Tensor-level wrappers around the C ABI (no autograd here; see efficient_modules.py / waveglow.py).

Every function takes CUDA fp32 tensors, launches on torch's current stream and returns freshly
allocated outputs.  Layout notes: "NCL" = (B, C, T) with T contiguous and channel stride T; the
batch stride is free so channel slices of a wider tensor are passed without copies.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
from typing import List, Optional, Tuple

import torch

from . import _lib as L
from .base import audio_lengths


def _ncl(t: torch.Tensor) -> torch.Tensor:
    """Return t if it is (B, C, T) with unit time stride and channel stride T, else a contiguous copy."""
    if t.dim() != 3:
        raise ValueError(f"expected a (B, C, T) tensor, got shape {tuple(t.shape)}")
    if t.dtype != torch.float32:
        t = t.float()
    B, Cc, T = t.shape
    if T == 0 or B == 0 or Cc == 0:
        return t.contiguous()
    if t.stride(2) == 1 and (Cc == 1 or t.stride(1) == T) and (B == 1 or t.stride(0) >= Cc * T):
        return t
    return t.contiguous()


def _bstride(t: torch.Tensor) -> int:
    return t.stride(0) if t.shape[0] > 1 else t.shape[1] * t.shape[2]


# ---------------------------------------------------------------------------------------------
# invertible 1x1 conv
# ---------------------------------------------------------------------------------------------
def small_inverse_logdet(w2d: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    L.require_cuda(w2d, op="small_inverse_logdet")
    w2d = w2d.detach().contiguous().float()
    c = w2d.shape[0]
    winv = torch.empty_like(w2d)
    logdet = torch.empty((), device=w2d.device, dtype=torch.float32)
    L.check(L.load().cmwg_small_inverse_logdet(w2d.data_ptr(), c, winv.data_ptr(), logdet.data_ptr(),
                                               L.stream_ptr(w2d.device)), "small_inverse_logdet")
    return winv, logdet


def conv1x1_apply(w2d: torch.Tensor, x: torch.Tensor, transpose: bool = False,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    L.require_cuda(w2d, x, op="conv1x1_apply")
    w2d = w2d.contiguous()  # row-major c x c (QR factors come out column-major)
    x = _ncl(x)
    B, Cc, T = x.shape
    if out is None:
        out = torch.empty((B, Cc, T), device=x.device, dtype=torch.float32)
    L.check(L.load().cmwg_conv1x1_apply(w2d.data_ptr(), int(transpose), x.data_ptr(), _bstride(x), out.data_ptr(),
                                        _bstride(out), B, Cc, T, L.stream_ptr(x.device)), "conv1x1_apply")
    return out


def conv1x1_wgrad(dz: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    L.require_cuda(dz, x, op="conv1x1_wgrad")
    dz, x = _ncl(dz), _ncl(x)
    B, Cc, T = x.shape
    lib = L.load()
    ws = torch.empty(max(int(lib.cmwg_conv1x1_wgrad_workspace(B, Cc, T)), 4), device=x.device, dtype=torch.uint8)
    dm = torch.empty((Cc, Cc), device=x.device, dtype=torch.float32)
    L.check(lib.cmwg_conv1x1_wgrad(dz.data_ptr(), _bstride(dz), x.data_ptr(), _bstride(x), B, Cc, T, dm.data_ptr(),
                                   ws.data_ptr(), L.stream_ptr(x.device)), "conv1x1_wgrad")
    return dm


def conv1x1_dw_finalize(dm: torch.Tensor, winv: torch.Tensor, dlogdet: torch.Tensor, T: int,
                        inverse_mode: bool, out: torch.Tensor = None) -> torch.Tensor:
    c = dm.shape[0]
    dlogdet = dlogdet.detach().reshape(()).float().contiguous()
    dw = out if out is not None else torch.empty_like(dm)
    L.check(L.load().cmwg_conv1x1_dw_finalize(dm.data_ptr(), winv.data_ptr(), dlogdet.data_ptr(), c, T,
                                              int(inverse_mode), dw.data_ptr(), L.stream_ptr(dm.device)),
            "conv1x1_dw_finalize")
    return dw


def conv1x1_backward(w: torch.Tensor, winv: torch.Tensor, inverse: bool, out: torch.Tensor, dout: torch.Tensor,
                     dlogdet, restored, dw_out):
    """Restore the forward call's input into `restored` (contiguous (B, C, T) or None), return din; `dw_out` (C x C view
    or None) receives the weight gradient.  One fused sweep + one finalise launch for even C <= 8."""
    out, dout = _ncl(out), _ncl(dout)
    B, Cc, T = out.shape
    lib = L.load()
    din = torch.empty((B, Cc, T), device=out.device, dtype=torch.float32)
    ws = None
    if dw_out is not None:
        ws = torch.empty(int(lib.cmwg_conv1x1_backward_workspace(B, Cc, T)), device=out.device, dtype=torch.uint8)
        if dlogdet is not None:
            dlogdet = dlogdet.detach().reshape(()).float().contiguous()
    L.check(lib.cmwg_conv1x1_backward(w.data_ptr(), winv.data_ptr(), int(inverse), out.data_ptr(), _bstride(out),
                                      dout.data_ptr(), _bstride(dout), L.ptr(dlogdet) if dw_out is not None else 0, B, Cc, T,
                                      L.ptr(restored), Cc * T, din.data_ptr(), Cc * T, L.ptr(dw_out), L.ptr(ws),
                                      L.stream_ptr(out.device)), "conv1x1_backward")
    return din


# ---------------------------------------------------------------------------------------------
# affine coupling
# ---------------------------------------------------------------------------------------------
def coupling_apply(x: torch.Tensor, lst: torch.Tensor, inverse: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """z = cat(xa, xb*exp(ls)+t) or cat(xa, (xb-t)/exp(ls)); returns (z, -log_s or None)."""
    x = _ncl(x)
    B, c, T = x.shape
    cin = c // 2
    z = torch.empty((B, c, T), device=x.device, dtype=torch.float32)
    neg = torch.empty((B, cin, T), device=x.device, dtype=torch.float32) if inverse else None
    L.check(L.load().cmwg_coupling_apply(x.data_ptr(), _bstride(x), lst.data_ptr(), z.data_ptr(), _bstride(z),
                                         L.ptr(neg), B, cin, T, int(inverse), L.stream_ptr(x.device)),
            "coupling_apply")
    return z, neg


def coupling_apply_varlen(x: torch.Tensor, lst: torch.Tensor, lengths_dev: torch.Tensor,
                          inverse: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """coupling_apply on a padded batch: columns t >= lengths_dev[b] of z and -log_s are 0."""
    x = _ncl(x)
    B, c, T = x.shape
    cin = c // 2
    z = torch.empty((B, c, T), device=x.device, dtype=torch.float32)
    neg = torch.empty((B, cin, T), device=x.device, dtype=torch.float32) if inverse else None
    L.check(L.load().cmwg_coupling_apply_varlen(x.data_ptr(), _bstride(x), lst.data_ptr(), z.data_ptr(), _bstride(z),
                                                L.ptr(neg), B, cin, T, lengths_dev.data_ptr(), int(inverse),
                                                L.stream_ptr(x.device)), "coupling_apply_varlen")
    return z, neg


def coupling_bwd(out: torch.Tensor, lst: torch.Tensor, dout: torch.Tensor, dls: torch.Tensor,
                 restored: torch.Tensor, inverse: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    """Writes the re-materialised input into `restored` (contiguous (B, c, T)); returns (dlst, din)."""
    out, dout, dls = _ncl(out), _ncl(dout), _ncl(dls)
    B, c, T = out.shape
    cin = c // 2
    dlst = torch.empty((B, c, T), device=out.device, dtype=torch.float32)
    din = torch.empty((B, c, T), device=out.device, dtype=torch.float32)
    L.check(L.load().cmwg_coupling_bwd(out.data_ptr(), _bstride(out), lst.data_ptr(), dout.data_ptr(), _bstride(dout),
                                       dls.data_ptr(), _bstride(dls), restored.data_ptr(), dlst.data_ptr(),
                                       din.data_ptr(), B, cin, T, int(inverse), L.stream_ptr(out.device)),
            "coupling_bwd")
    return dlst, din


# ---------------------------------------------------------------------------------------------
# glue
# ---------------------------------------------------------------------------------------------
def squeeze(x: torch.Tensor, n_group: int, inverse: bool = False) -> torch.Tensor:
    """forward: (B, T) -> (B, n_group, T/n_group); inverse: (B, G, T') -> (B, G*T')."""
    L.require_cuda(x, op="squeeze")
    x = x.contiguous().float()
    if not inverse:
        B, T = x.shape
        out = torch.empty((B, n_group, T // n_group), device=x.device, dtype=torch.float32)
    else:
        B, G, Tq = x.shape
        T = G * Tq
        out = torch.empty((B, T), device=x.device, dtype=torch.float32)
    L.check(L.load().cmwg_squeeze(x.data_ptr(), out.data_ptr(), B, T, n_group, int(inverse), L.stream_ptr(x.device)),
            "squeeze")
    return out


def sum_per_batch(a: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    a = _ncl(a) if a.dim() == 3 else a.contiguous()
    B = a.shape[0]
    N = a[0].numel()
    if a.dim() == 3 and not a.is_contiguous():
        # channel slice: rows are contiguous per batch item
        pass
    out = torch.empty((B,), device=a.device, dtype=torch.float32)
    L.check(L.load().cmwg_sum_per_batch(a.data_ptr(), a.stride(0) if B > 1 else N, B, N, out.data_ptr(), 0,
                                        float(scale), L.stream_ptr(a.device)), "sum_per_batch")
    return out


def logdet_accumulate(log_s: torch.Tensor, prev, log_det_w) -> torch.Tensor:
    """prev (B,) or None  +  log_det_w (0-dim) or None  +  log_s.sum((1, 2)), one launch."""
    a = _ncl(log_s)
    B = a.shape[0]
    N = a[0].numel()
    out = torch.empty((B,), device=a.device, dtype=torch.float32)
    if log_det_w is not None:
        log_det_w = log_det_w.detach().reshape(()).float().contiguous()
    if prev is not None:
        prev = prev.detach().float().contiguous()
    L.check(L.load().cmwg_logdet_accumulate(a.data_ptr(), a.stride(0) if B > 1 else N, B, N, L.ptr(prev), L.ptr(log_det_w),
                                            out.data_ptr(), L.stream_ptr(a.device)), "logdet_accumulate")
    return out


def logdet_accumulate_varlen(a: torch.Tensor, lengths_dev: torch.Tensor, prev, log_det_w_col) -> torch.Tensor:
    """prev (B,) or None + log_det_w_col (0-dim: the log-det of one column) * len_b + a[b, :, :len_b].sum()."""
    if a.dim() != 3 or a.stride(2) != 1 or (a.shape[1] > 1 and a.stride(1) != a.shape[2]):
        a = a.contiguous()
    B, Cc, T = a.shape
    out = torch.empty((B,), device=a.device, dtype=torch.float32)
    if log_det_w_col is not None:
        log_det_w_col = log_det_w_col.detach().reshape(()).float().contiguous()
    if prev is not None:
        prev = prev.detach().float().contiguous()
    L.check(L.load().cmwg_logdet_accumulate_varlen(a.data_ptr(), a.stride(0) if B > 1 else Cc * T, B, Cc, T,
                                                   lengths_dev.data_ptr(), L.ptr(prev), L.ptr(log_det_w_col),
                                                   out.data_ptr(), L.stream_ptr(a.device)), "logdet_accumulate_varlen")
    return out


def nll_loss(z: torch.Tensor, logdet: torch.Tensor, sigma: float, mean: bool, want_dz: bool):
    L.require_cuda(z, logdet, op="nll_loss")
    z = z.contiguous().float()
    B, T = z.shape
    logdet = logdet.detach().float().expand(B).contiguous() if logdet.dim() == 0 else logdet.contiguous().float()
    loss = torch.empty((), device=z.device, dtype=torch.float32)
    dz = torch.empty_like(z) if want_dz else None
    ws = torch.empty((B + 1,), device=z.device, dtype=torch.float32)
    L.check(L.load().cmwg_nll_loss(z.data_ptr(), logdet.data_ptr(), B, T, float(sigma), int(mean), loss.data_ptr(),
                                   L.ptr(dz), ws.data_ptr(), L.stream_ptr(z.device)), "nll_loss")
    return loss, dz


# ---------------------------------------------------------------------------------------------
# upsampler
# ---------------------------------------------------------------------------------------------
def upsample_fwd(h, g, v, bias, stride: int, pad: int) -> torch.Tensor:
    L.require_cuda(h, v, op="upsample_fwd")
    h = h.contiguous().float()
    B, Cc, F = h.shape
    K = v.shape[-1]
    Tout = (F - 1) * stride - 2 * pad + K
    y = torch.empty((B, Cc, Tout), device=h.device, dtype=torch.float32)
    L.check(L.load().cmwg_upsample_fwd(h.data_ptr(), L.ptr(g), v.data_ptr(), L.ptr(bias), B, Cc, F, K, stride, pad,
                                       y.data_ptr(), L.stream_ptr(h.device)), "upsample_fwd")
    return y


def upsample_bwd(h, g, v, dy, stride: int, pad: int, want_bias: bool, out=None):
    """`out` = (dg, dv, db) destination tensors (e.g. views of the data-parallel gradient buckets) or None."""
    h = h.contiguous().float()
    B, Cc, F = h.shape
    K = v.shape[-1]
    if dy.stride(2) != 1:
        dy = dy.contiguous()
    if out is not None:
        dg, dv, db = out
    else:
        dg = torch.empty_like(g) if g is not None else None
        dv = torch.empty_like(v)
        db = torch.empty((Cc,), device=h.device, dtype=torch.float32) if want_bias else None
    lib = L.load()
    ws = torch.empty(max(int(lib.cmwg_upsample_bwd_workspace(B, Cc, K)), 4), device=h.device, dtype=torch.uint8)
    L.check(lib.cmwg_upsample_bwd(h.data_ptr(), L.ptr(g), v.data_ptr(), dy.data_ptr(), dy.stride(0), dy.stride(1),
                                  B, Cc, F, K, stride, pad, dy.shape[2], L.ptr(dg), dv.data_ptr(), L.ptr(db), ws.data_ptr(),
                                  L.stream_ptr(h.device)), "upsample_bwd")
    return dg, dv, db


def upsample_bwd_input(g, v, dy, F: int, stride: int, pad: int) -> torch.Tensor:
    """Gradient w.r.t. the upsampler input h (B, C, F)."""
    B, Cc, Tv = dy.shape
    K = v.shape[-1]
    if dy.stride(2) != 1:
        dy = dy.contiguous()
    dh = torch.empty((B, Cc, F), device=dy.device, dtype=torch.float32)
    L.check(L.load().cmwg_upsample_bwd_input(L.ptr(g), v.data_ptr(), dy.data_ptr(), dy.stride(0), dy.stride(1), B, Cc,
                                             F, K, stride, pad, Tv, dh.data_ptr(), L.stream_ptr(dy.device)),
            "upsample_bwd_input")
    return dh


# ---------------------------------------------------------------------------------------------
# denoiser (bias-spectrum subtraction)
# ---------------------------------------------------------------------------------------------
def stft_frame_magnitude(x: torch.Tensor, window: torch.Tensor, hop: int, frame: int = 0) -> torch.Tensor:
    """|torch.stft(x, n_fft, hop, window, center=True, pad_mode="reflect")[:, frame]| of a 1-D signal, n_fft = len(window)."""
    L.require_cuda(x, window, op="stft_frame_magnitude")
    x = x.detach().reshape(-1).float().contiguous()
    n_fft = window.numel()
    mag = torch.empty((n_fft // 2 + 1,), device=x.device, dtype=torch.float32)
    L.check(L.load().cmwg_stft_frame_magnitude(x.data_ptr(), x.numel(), window.data_ptr(), n_fft, int(hop), int(frame),
                                               mag.data_ptr(), L.stream_ptr(x.device)), "stft_frame_magnitude")
    return mag


def lengths_arg(lens: Optional[List[int]], device) -> Tuple[Optional[C.Array], Optional[torch.Tensor]]:
    """Per-item lengths as the C ABI takes them: a ctypes int array on the host and the same values as an int32 tensor on
    `device`, or (None, None).  The upload waits for the stream (a blocking copy from pageable memory), so callers make it
    just before the launch: host work between the two would leave the GPU idle."""
    if lens is None:
        return None, None
    return (C.c_int * len(lens))(*lens), torch.tensor(lens, dtype=torch.int32).to(device)


def audio_batch(x: torch.Tensor) -> Tuple[torch.Tensor, bool]:
    """x (T,) or (B, T) as a (B, T) float32 tensor with unit time stride (x itself when it is one), and whether to index the
    result back to x's rank."""
    squeeze = x.dim() == 1
    x = x.detach()
    if squeeze:
        x = x.unsqueeze(0)
    if x.dtype != torch.float32 or x.stride(1) != 1:
        x = x.float().contiguous()
    return x, squeeze


def denoise(audio: torch.Tensor, window: torch.Tensor, bias_mag: torch.Tensor, strength: float, hop: int,
            lengths=None, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Bias-spectrum subtraction (cmwg_denoise) of audio (T,) or (B, T) with optional per-item `lengths` in samples; returns
    a tensor of audio's shape, 0 after each item's length.  `workspace`: uint8 tensor of at least
    cmwg_denoise_workspace_bytes bytes (allocated here when None).  Each length must exceed n_fft / 2."""
    n_fft = window.numel()
    if isinstance(strength, bool) or not isinstance(strength, numbers.Real) or not 0 <= strength < math.inf:
        raise ValueError(f"denoise: strength must be a finite number >= 0, got {strength!r}")
    lens = audio_lengths(audio, lengths, n_fft // 2, "denoise")
    L.require_cuda(audio, window, bias_mag, op="denoise")
    x, squeeze = audio_batch(audio)
    B, T = x.shape
    out = torch.empty((B, T), device=x.device, dtype=torch.float32)
    lib = L.load()
    need = int(lib.cmwg_denoise_workspace_bytes(B, T, n_fft, int(hop)))
    if workspace is None:
        workspace = torch.empty((max(need, 4),), device=x.device, dtype=torch.uint8)
    elif workspace.numel() * workspace.element_size() < need:
        raise ValueError(f"denoise: workspace of {workspace.numel() * workspace.element_size()} bytes, {need} needed")
    lens_host, lens_dev = lengths_arg(lens, x.device)
    L.check(lib.cmwg_denoise(x.data_ptr(), x.stride(0) if B > 1 else T, B, T, lens_host, L.ptr(lens_dev),
                             window.data_ptr(), bias_mag.data_ptr(), float(strength), n_fft, int(hop),
                             workspace.data_ptr(), out.data_ptr(), L.stream_ptr(x.device)), "denoise")
    return out[0] if squeeze else out


# ---------------------------------------------------------------------------------------------
# band-limited resampling
# ---------------------------------------------------------------------------------------------
def resample_lengths(x: Tensor, lengths) -> Optional[List[int]]:
    """audio_lengths for resample: each length in [1, T]; T itself is not bounded, so an empty signal resamples to an empty
    one."""
    return audio_lengths(x, lengths, 0, "Resample", check_full=False)


def resample(x: Tensor, table: Tensor, first: Tensor, O: int, N: int, w: int, lengths=None) -> Tensor:
    """cmwg_resample (band-limited resampling, resample.py) of x (B, T) or (T,) on the GPU -> (B, ceil(N T / O)) or (ceil(N T / O),) float32; item b (len_b
    samples) holds its ceil(N len_b / O) resampled samples, then zeros.  table (L, N) float32 and first (N,) int32 on x's
    device come from resample_table."""
    lens = resample_lengths(x, lengths)
    T = x.shape[-1]
    if (N * T + O - 1) // O > 2 ** 31 - 1:
        raise ValueError(f"resample: {T} samples give {(N * T + O - 1) // O} output samples, more than the 2**31 - 1 a "
                         "call can write")
    L.require_cuda(x, table, first, op="resample")
    if table.dtype != torch.float32 or table.dim() != 2 or table.shape[1] != N or first.dtype != torch.int32 \
            or first.shape != (N,):
        raise ValueError(f"resample: expected table (L, {N}) float32 and first ({N},) int32, got {tuple(table.shape)} "
                         f"{table.dtype} and {tuple(first.shape)} {first.dtype}")
    table, first = table.contiguous(), first.contiguous()
    x, squeeze = audio_batch(x)
    B, T = x.shape
    T_out = (N * T + O - 1) // O
    y = torch.empty((B, T_out), device=x.device, dtype=torch.float32)
    lens_host, lens_dev = lengths_arg(lens, x.device)
    L.check(L.load().cmwg_resample(x.data_ptr(), x.stride(0) if B > 1 else T, B, T, lens_host, L.ptr(lens_dev),
                                   table.data_ptr(), first.data_ptr(), O, N, table.shape[0], w, y.data_ptr(),
                                   T_out, T_out, L.stream_ptr(x.device)), "resample")
    return y[0] if squeeze else y


def selftest_tc_gemm(a: torch.Tensor, b: torch.Tensor, M: int, N: int, K: int, variant: int) -> torch.Tensor:
    """16-bit operands through the tcgen05 engine; see cmwg_selftest_tc_gemm."""
    is_fp16 = int(a.dtype == torch.float16)
    d = torch.zeros((M, N), device=a.device, dtype=torch.float32)
    L.check(L.load().cmwg_selftest_tc_gemm(a.data_ptr(), b.data_ptr(), d.data_ptr(), M, N, K, is_fp16, variant,
                                           L.stream_ptr(a.device)), "selftest_tc_gemm")
    return d
