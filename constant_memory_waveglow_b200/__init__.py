"""constant_memory_waveglow_b200 -- B200-native (sm_100a) flow hot path of constant-memory-waveglow.

Host side: PyTorch modules / autograd Functions with the reference's names and semantics.
Device side: hand-written CUDA (tcgen05 / TMEM / TMA GEMM engine + fp32 CUDA-core engine +
HBM-bound flow primitives) behind the C ABI of include/cmwg_b200.h, loaded with ctypes.
"""
from .base import FlowBase, Reversible, pad_batch
from .efficient_modules import (AffineCouplingBlock, AffineCouplingFunc, Conv1x1Func, InvAffineCouplingFunc,
                                InvConv1x1Func, InvertibleConv1x1)
from .loss import WaveGlowLoss
from .precision import get_precision, set_precision
from .utils import add_weight_norms, get_instance, remove_weight_norms
from .waveglow import WN, NonCausalLayer, WaveGlow, fused_gate, invalidate_packs
from .waveflow import WN2D, NonCausalLayer2D, WaveFlow
from .wsrglow import WSRGlow
from .mr_waveglow import MRWaveGlow
from .melglow import MelGlow, WN_LVC
from .denoiser import Denoiser

__all__ = ["FlowBase", "Reversible", "AffineCouplingBlock", "InvertibleConv1x1", "AffineCouplingFunc",
           "InvAffineCouplingFunc", "Conv1x1Func", "InvConv1x1Func", "WaveGlowLoss", "WN", "NonCausalLayer",
           "WaveGlow", "WSRGlow", "MRWaveGlow", "MelGlow", "WN_LVC", "WaveFlow", "WN2D", "NonCausalLayer2D", "fused_gate", "add_weight_norms", "remove_weight_norms", "get_instance", "set_precision",
           "get_precision", "invalidate_packs", "pad_batch", "Denoiser"]
