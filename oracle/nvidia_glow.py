"""NVIDIA's WaveGlow (NVIDIA/waveglow ``glow.py``) restated in plain PyTorch, for tests and benchmarks only.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (see ``flow_oracle.py``).  Class and attribute names are NVIDIA's, so a
``state_dict()`` of ``WaveGlow`` has NVIDIA's keys (``upsample``, ``WN.k.cond_layer``, ``WN.k.in_layers.i``,
``WN.k.res_skip_layers.i``, ``WN.k.start``, ``WN.k.end``, ``convinv.k.conv``); ``cond_layers=True`` builds the older
per-layer ``cond_layers.i`` form that DeepLearningExamples keeps.  Runs in any dtype (fp64 for the parity tests).

Differences from ``glow.py``, none of which changes the arithmetic: ``forward`` and ``reverse`` take the audio / noise as
(B, T) and return ``(audio, per-item log-det)`` in the package's convention (NVIDIA's ``log_det_W`` is summed over the
batch); ``infer`` takes the noise instead of drawing it, as the package's ``infer(z=...)`` does, splitting it the same way.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor, nn


def fused_add_tanh_sigmoid_multiply(input_a: Tensor, input_b: Tensor, n_channels: int) -> Tensor:
    in_act = input_a + input_b
    return torch.tanh(in_act[:, :n_channels]) * torch.sigmoid(in_act[:, n_channels:])


class Invertible1x1Conv(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.conv = nn.Conv1d(c, c, kernel_size=1, stride=1, padding=0, bias=False)
        W = torch.linalg.qr(torch.randn(c, c))[0]
        if torch.det(W) < 0:
            W[:, 0] = -1 * W[:, 0]
        self.conv.weight.data = W.view(c, c, 1)

    def forward(self, z: Tensor) -> Tuple[Tensor, Tensor]:
        """z -> (W z, log|det W| of ONE column)."""
        W = self.conv.weight.squeeze(-1)
        return self.conv(z), torch.logdet(W)

    def reverse(self, z: Tensor) -> Tensor:
        W = self.conv.weight.squeeze(-1)
        if W.dtype == torch.float16:    # as glow.py: the inverse in fp32, applied in fp16
            return F.conv1d(z, W.float().inverse().half().unsqueeze(-1))
        return F.conv1d(z, W.inverse().unsqueeze(-1))


class WN(nn.Module):
    def __init__(self, n_in_channels: int, n_mel_channels: int, n_layers: int, n_channels: int, kernel_size: int,
                 cond_layers: bool = False):
        super().__init__()
        wn = nn.utils.weight_norm
        self.n_layers, self.n_channels = n_layers, n_channels
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        self.start = wn(nn.Conv1d(n_in_channels, n_channels, 1), name="weight")
        end = nn.Conv1d(n_channels, 2 * n_in_channels, 1)   # NVIDIA zero-initialises it; tests set random values
        self.end = end
        if cond_layers:
            self.cond_layers = nn.ModuleList(wn(nn.Conv1d(n_mel_channels, 2 * n_channels, 1), name="weight")
                                             for _ in range(n_layers))
        else:
            self.cond_layer = wn(nn.Conv1d(n_mel_channels, 2 * n_channels * n_layers, 1), name="weight")
        for i in range(n_layers):
            dilation = 2 ** i
            padding = int((kernel_size * dilation - dilation) / 2)
            self.in_layers.append(wn(nn.Conv1d(n_channels, 2 * n_channels, kernel_size, dilation=dilation,
                                               padding=padding), name="weight"))
            rs = 2 * n_channels if i < n_layers - 1 else n_channels
            self.res_skip_layers.append(wn(nn.Conv1d(n_channels, rs, 1), name="weight"))

    def forward(self, audio: Tensor, spect: Tensor) -> Tensor:
        audio = self.start(audio)
        output = torch.zeros_like(audio)
        if hasattr(self, "cond_layer"):
            spect = self.cond_layer(spect)
        for i in range(self.n_layers):
            if hasattr(self, "cond_layer"):
                off = i * 2 * self.n_channels
                spect_i = spect[:, off:off + 2 * self.n_channels]
            else:
                spect_i = self.cond_layers[i](spect)
            acts = fused_add_tanh_sigmoid_multiply(self.in_layers[i](audio), spect_i, self.n_channels)
            res_skip = self.res_skip_layers[i](acts)
            if i < self.n_layers - 1:
                audio = audio + res_skip[:, :self.n_channels]
                output = output + res_skip[:, self.n_channels:]
            else:
                output = output + res_skip
        return self.end(output)          # [b, log_s]


class WaveGlow(nn.Module):
    def __init__(self, n_mel_channels: int = 80, n_flows: int = 12, n_group: int = 8, n_early_every: int = 4,
                 n_early_size: int = 2, WN_config: Optional[dict] = None, cond_layers: bool = False):
        super().__init__()
        WN_config = dict(WN_config or {"n_layers": 8, "n_channels": 256, "kernel_size": 3})
        self.upsample = nn.ConvTranspose1d(n_mel_channels, n_mel_channels, 1024, stride=256)
        self.n_flows, self.n_group = n_flows, n_group
        self.n_early_every, self.n_early_size = n_early_every, n_early_size
        self.WN = nn.ModuleList()
        self.convinv = nn.ModuleList()
        n_half = n_group // 2
        n_remaining = n_group
        self.z_split_sizes: List[int] = []
        for k in range(n_flows):
            if k % n_early_every == 0 and k > 0:
                n_half -= n_early_size // 2
                n_remaining -= n_early_size
                self.z_split_sizes.append(n_early_size)
            self.convinv.append(Invertible1x1Conv(n_remaining))
            self.WN.append(WN(n_half, n_mel_channels * n_group, cond_layers=cond_layers, **WN_config))
        self.n_remaining_channels = n_remaining
        self.z_split_sizes.append(n_remaining)

    def conditioning(self, spect: Tensor, T: int) -> Tensor:
        """upsample -> [:T] -> unfold by n_group: (B, n_mel * n_group, T / n_group)."""
        spect = self.upsample(spect)
        assert spect.size(2) >= T
        spect = spect[:, :, :T]
        spect = spect.unfold(2, self.n_group, self.n_group).permute(0, 2, 1, 3)
        return spect.contiguous().view(spect.size(0), spect.size(1), -1).permute(0, 2, 1)

    def forward(self, spect: Tensor, audio: Tensor) -> Tuple[Tensor, Tensor]:
        """(z (B, T) in the package's unsqueezed order, per-item log-det)."""
        cond = self.conditioning(spect, audio.size(1))
        audio = audio.unfold(1, self.n_group, self.n_group).permute(0, 2, 1)
        output_audio = []
        logdet = audio.new_zeros(audio.size(0))
        for k in range(self.n_flows):
            if k % self.n_early_every == 0 and k > 0:
                output_audio.append(audio[:, :self.n_early_size, :])
                audio = audio[:, self.n_early_size:, :]
            audio, log_det_w = self.convinv[k](audio)
            n_half = audio.size(1) // 2
            audio_0, audio_1 = audio[:, :n_half, :], audio[:, n_half:, :]
            output = self.WN[k](audio_0, cond)
            log_s, b = output[:, n_half:, :], output[:, :n_half, :]
            audio_1 = torch.exp(log_s) * audio_1 + b
            logdet = logdet + log_s.sum((1, 2)) + audio.size(2) * log_det_w
            audio = torch.cat([audio_0, audio_1], 1)
        output_audio.append(audio)
        z = torch.cat(output_audio, 1)
        return z.permute(0, 2, 1).reshape(z.size(0), -1), logdet

    def reverse(self, spect: Tensor, z: Tensor, with_logdet: bool = True) -> Tuple[Tensor, Optional[Tensor]]:
        """NVIDIA's infer loop on the noise z (B, T) split as the package splits it; returns (audio, per-item log-det or
        None)."""
        cond = self.conditioning(spect, z.size(1))
        zs = z.unfold(1, self.n_group, self.n_group).permute(0, 2, 1)
        parts = list(zs.split(self.z_split_sizes, 1))
        audio = parts.pop()
        logdet = z.new_zeros(z.size(0))
        for k in reversed(range(self.n_flows)):
            n_half = audio.size(1) // 2
            audio_0, audio_1 = audio[:, :n_half, :], audio[:, n_half:, :]
            output = self.WN[k](audio_0, cond)
            s, b = output[:, n_half:, :], output[:, :n_half, :]
            audio_1 = (audio_1 - b) / torch.exp(s)
            audio = torch.cat([audio_0, audio_1], 1)
            audio = self.convinv[k].reverse(audio)
            if with_logdet:
                logdet = logdet - s.sum((1, 2)) - audio.size(2) * torch.logdet(self.convinv[k].conv.weight.squeeze(-1))
            if k % self.n_early_every == 0 and k > 0:
                audio = torch.cat((parts.pop(), audio), 1)
        return audio.permute(0, 2, 1).reshape(audio.size(0), -1), (logdet if with_logdet else None)

    def infer(self, spect: Tensor, z: Tensor) -> Tensor:
        """``infer``: the upsampled mel loses its last 1024 - 256 samples, so the output has frames * 256 samples."""
        time_cutoff = self.upsample.kernel_size[0] - self.upsample.stride[0]
        T = (spect.size(2) - 1) * self.upsample.stride[0] + self.upsample.kernel_size[0] - time_cutoff
        return self.reverse(spect, z[:, :T], with_logdet=False)[0]


def randomize(model: WaveGlow, seed: int = 0, scale: float = 1.0) -> WaveGlow:
    """Random weights of a trained model's magnitude (NVIDIA's init leaves `end` at zero, which would hide the WN)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("weight_g"):
                p.copy_(0.5 + torch.rand(p.shape, generator=g, dtype=torch.float64).to(p.dtype))
            elif "convinv" in name:
                continue
            else:
                fan = p[0].numel() if p.dim() > 1 else 1
                std = (0.02 if name.endswith("bias") else 1.0 / fan ** 0.5) * scale
                if name.startswith("WN.") and ".end." in name:
                    std *= 0.05
                if name.startswith("upsample."):
                    std = 0.05 if name.endswith("weight") else 0.02
                p.copy_(torch.randn(p.shape, generator=g, dtype=torch.float64).to(p.dtype) * std)
    return model
