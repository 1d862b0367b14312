"""WSRGlow (audio super-resolution flow): host-side mirror of the reference's ``model/wsrglow.py``.

``WSRGlow`` (:21-56) is a ``WaveGlow`` with 12 flows, ``n_group = hop = 8 * upsample_rate``, early outputs
4 / 2 and a 3659-channel conditioning built from the low-rate signal by ``_get_cond`` (:37-50): mu-law code
embedding (3200 rows), 9 STFT magnitudes and 9 x 50 phase-embedding rows, at one conditioning column per
squeezed time step (upsample factor 1).  The flow itself -- 1x1 convs, couplings, the WN stack whose ``V``
conv is now 3659 -> 2*Cd*depth and dominates the FLOPs (78 %) -- runs on the same libcmwg_b200.so kernels as
WaveGlow; the conditioning front end is ONE kernel, ``cmwg_wsrglow_cond`` (csrc/wsrglow_cond.cu: clip, mu-law codes, table
gathers, the 16-point windowed DFT, phase codes, written straight into the (B, 3659, F) layout), whose backward scatters the
cotangent into the two embedding tables.  ``_get_cond_torch`` keeps the op-by-op form the kernel is tested against.
"""
from __future__ import annotations

import math

import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib as L
from .waveglow import WaveGlow


class _CondFunction(torch.autograd.Function):
    """cmwg_wsrglow_cond with the gradient of the two embedding tables (the signal itself gets none: its path goes through
    integer codes, as in the reference)."""

    @staticmethod
    def forward(ctx, c, emb, aemb, window):
        L.require_cuda(c, emb, aemb, op="WSRGlow._get_cond")
        if c.dim() != 2 or c.dtype != torch.float32 or not c.is_contiguous():
            raise RuntimeError("WSRGlow: the low-rate signal must be a contiguous fp32 (B, T) tensor")
        B, Tc = c.shape
        E, P = emb.shape[1], aemb.shape[1]
        nf = Tc // 8
        need = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        out = torch.empty((B, 8 * E + 9 + 9 * P, nf), device=c.device, dtype=torch.float32)
        codes = torch.empty((B, Tc), device=c.device, dtype=torch.int32) if need else None
        phase = torch.empty((B, 9, nf), device=c.device, dtype=torch.int32) if need else None
        L.check(L.load().cmwg_wsrglow_cond(c.data_ptr(), B, Tc, emb.detach().contiguous().data_ptr(), E, emb.shape[0],
                                           aemb.detach().contiguous().data_ptr(), P, aemb.shape[0],
                                           window.contiguous().data_ptr(), out.data_ptr(), L.ptr(codes), L.ptr(phase),
                                           L.stream_ptr(c.device)), "wsrglow_cond")
        ctx.mark_dirty(c)                      # clipped in place, like the reference's c.clip_(-1, 1)
        ctx.save_for_backward(codes, phase)
        ctx.dims = (B, nf, E, P, emb.shape[0], aemb.shape[0])
        return out, c

    @staticmethod
    def backward(ctx, dout, _dc):
        codes, phase = ctx.saved_tensors
        B, nf, E, P, n_codes, n_phase = ctx.dims
        d_emb = d_aemb = None
        if ctx.needs_input_grad[1]:
            src = dout[:, :8 * E].reshape(B, 8, E, nf).permute(0, 3, 1, 2).reshape(-1, E)       # sample 8f + j <- row j*E + e
            d_emb = torch.zeros((n_codes, E), device=dout.device, dtype=dout.dtype).index_add_(0, codes.flatten().long(), src)
        if ctx.needs_input_grad[2]:
            src = dout[:, 8 * E + 9:].reshape(B, 9, P, nf).permute(0, 1, 3, 2).reshape(-1, P)
            d_aemb = torch.zeros((n_phase, P), device=dout.device, dtype=dout.dtype).index_add_(0, phase.flatten().long(), src)
        return None, d_emb, d_aemb, None


class AngleEmbedding(nn.Module):
    """Reference ``model/wsrglow.py:8-18``: quantise an angle in [-pi, pi] to ``embed_num`` codes."""

    def __init__(self, embed_num, hidden_dim):
        super().__init__()
        self.embed_num = embed_num
        self.embed = nn.Embedding(num_embeddings=embed_num, embedding_dim=hidden_dim)

    def forward(self, index):
        embed_num = self.embed_num
        index = ((index / torch.pi + 1) * 0.5 * (embed_num - 1)).long()
        return self.embed(index)


class MuLawEncoding(nn.Module):
    """torchaudio.transforms.MuLawEncoding(quantization_channels) without the torchaudio dependency."""

    def __init__(self, quantization_channels: int = 256):
        super().__init__()
        self.quantization_channels = quantization_channels

    def forward(self, x):
        mu = torch.tensor(self.quantization_channels - 1.0, dtype=x.dtype, device=x.device)
        x_mu = torch.sign(x) * torch.log1p(mu * torch.abs(x)) / torch.log1p(mu)
        return ((x_mu + 1) / 2 * mu + 0.5).to(torch.int64)


class WSRGlow(WaveGlow):
    """Reference ``model/wsrglow.py:21-56`` (same constructor, attributes and state-dict keys:
    ``mu_enc.1.weight``, ``angle_embed.embed.weight``, buffer ``window``)."""
    _supports_lengths = False   # WaveGlow's per-item lengths do not cover the low-rate conditioning front end

    def __init__(self, upsample_rate: int = 2, memory_efficient: bool = False, **kwargs) -> None:
        super().__init__(12, 8 * upsample_rate, 4, 2, 8 * upsample_rate, 8 * 400 + 51 * 9,
                         memory_efficient=memory_efficient, **kwargs)
        self.mu_enc = nn.Sequential(MuLawEncoding(256), nn.Embedding(256, 400))
        self.angle_embed = AngleEmbedding(embed_num=120, hidden_dim=50)
        self.n_fft = 16
        self.hop_length = 8
        self.register_buffer('window', torch.hann_window(self.n_fft))
        k = torch.arange(self.n_fft // 2 + 1, dtype=torch.float64).view(-1, 1)
        n = torch.arange(self.n_fft, dtype=torch.float64).view(1, -1)
        ang = 2 * math.pi * k * n / self.n_fft
        sin = torch.sin(ang)
        sin[0] = 0.0                   # DC and Nyquist bins of a real signal are exactly real: a real FFT returns
        sin[self.n_fft // 2] = 0.0     # imag = +0.0 there, and atan2(+0, re < 0) = +pi picks the LAST phase code
        self.register_buffer('_dft_cos', torch.cos(ang).float(), persistent=False)
        self.register_buffer('_dft_sin', sin.float(), persistent=False)

    def _stft(self, c):
        """torch.stft(pad_reflect(c, 4), n_fft=16, hop=8, window, center=False) as a windowed DFT:
        returns (re, im), each (B, 9, frames)."""
        xp = F.pad(c.unsqueeze(1), (4, 4), mode='reflect').squeeze(1)
        frames = xp.unfold(-1, self.n_fft, self.hop_length) * self.window          # (B, frames, 16)
        fr = frames.unsqueeze(1)                                                    # (B, 1, frames, 16)
        re = (fr * self._dft_cos.view(1, -1, 1, self.n_fft)).sum(-1)
        s = (fr * self._dft_sin.view(1, -1, 1, self.n_fft)).sum(-1)
        im = torch.zeros_like(s) - s   # (+0) - (+-0) = +0: keeps the sign convention of the real FFT
        return re, im

    def _get_cond(self, c):
        if not c.is_cuda:
            raise RuntimeError("cmwg_b200 WSRGlow: expected CUDA tensors; this package has no CPU implementation")
        cond, _ = _CondFunction.apply(c, self.mu_enc[1].weight, self.angle_embed.embed.weight, self.window)
        return cond

    def _get_cond_torch(self, c):
        """The same computation op by op (test reference for the kernel; not on the product path)."""
        c = c.clip_(-1, 1)
        c_emb = self.mu_enc(c).view(c.shape[0], -1, 8 * 400).transpose(1, 2)
        re, im = self._stft(c)
        mag = torch.sqrt(re * re + im * im)
        phase_emb = self.angle_embed(torch.atan2(im, re)).permute(0, 1, 3, 2).reshape(re.shape[0], 50 * 9, -1)
        return torch.cat([c_emb, mag, phase_emb], dim=1)

    def forward_computation(self, x, h):
        return super().forward_computation(x, self._get_cond(h))

    def reverse_computation(self, z, h):
        return super().reverse_computation(z, self._get_cond(h))
