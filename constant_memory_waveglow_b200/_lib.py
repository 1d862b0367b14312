"""ctypes binding of libcmwg_b200.so (the C ABI declared in include/cmwg_b200.h).

There is NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
PyTorch is used only for device memory (tensors), streams and autograd plumbing; every op on the
flow hot path goes through the functions bound here.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcmwg_b200.so")

MAX_DEPTH = 16
PREC_FP32, PREC_BF16, PREC_FP16 = 0, 1, 2
PREC_NAMES = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp16": PREC_FP16}

c_float_p = C.POINTER(C.c_float)


class WnConfig(C.Structure):
    _fields_ = [("in_channels", C.c_int), ("aux_channels", C.c_int), ("dil_channels", C.c_int),
                ("res_channels", C.c_int), ("skip_channels", C.c_int), ("depth", C.c_int),
                ("radix", C.c_int), ("has_bias", C.c_int), ("precision", C.c_int),
                ("height", C.c_int), ("h_dilation", C.c_int * MAX_DEPTH)]


class ConvParam(C.Structure):
    _fields_ = [("g", C.c_void_p), ("v", C.c_void_p), ("bias", C.c_void_p)]


class WnParams(C.Structure):
    _fields_ = [("V", ConvParam), ("start", ConvParam), ("W", ConvParam * MAX_DEPTH),
                ("W_o", ConvParam * MAX_DEPTH), ("end", ConvParam)]


class ConvGrad(C.Structure):
    _fields_ = [("g", C.c_void_p), ("v", C.c_void_p), ("bias", C.c_void_p)]


class WnGrads(C.Structure):
    _fields_ = [("V", ConvGrad), ("start", ConvGrad), ("W", ConvGrad * MAX_DEPTH),
                ("W_o", ConvGrad * MAX_DEPTH), ("end", ConvGrad)]


# name -> (restype, argtypes); must list EVERY function declared in include/cmwg_b200.h
_LL = C.c_longlong
_VP = C.c_void_p
_I = C.c_int
_SZ = C.c_size_t
SIGNATURES = {
    "cmwg_last_error": (C.c_char_p, []),
    "cmwg_version": (_I, []),
    "cmwg_launch_count": (C.c_ulonglong, []),
    "cmwg_reset_launch_count": (None, []),
    "cmwg_small_inverse_logdet": (_I, [_VP, _I, _VP, _VP, _VP]),
    "cmwg_conv1x1_apply": (_I, [_VP, _I, _VP, _LL, _VP, _LL, _I, _I, _I, _VP]),
    "cmwg_conv1x1_wgrad_workspace": (_SZ, [_I, _I, _I]),
    "cmwg_conv1x1_wgrad": (_I, [_VP, _LL, _VP, _LL, _I, _I, _I, _VP, _VP, _VP]),
    "cmwg_conv1x1_dw_finalize": (_I, [_VP, _VP, _VP, _I, _I, _I, _VP, _VP]),
    "cmwg_conv1x1_backward_workspace": (_SZ, [_I, _I, _I]),
    "cmwg_conv1x1_backward": (_I, [_VP, _VP, _I, _VP, _LL, _VP, _LL, _VP, _I, _I, _I, _VP, _LL, _VP, _LL, _VP, _VP, _VP]),
    "cmwg_coupling_apply": (_I, [_VP, _LL, _VP, _VP, _LL, _VP, _I, _I, _I, _I, _VP]),
    "cmwg_coupling_apply_varlen": (_I, [_VP, _LL, _VP, _VP, _LL, _VP, _I, _I, _I, _VP, _I, _VP]),
    "cmwg_coupling_bwd": (_I, [_VP, _LL, _VP, _VP, _LL, _VP, _LL, _VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "cmwg_wn_tc_supported": (_I, [C.POINTER(WnConfig)]),
    "cmwg_wn_aux_padded": (_I, [C.POINTER(WnConfig)]),
    "cmwg_cond_pack": (_I, [C.POINTER(WnConfig), _VP, _LL, _LL, _LL, _I, _I, _VP, _VP]),
    "cmwg_cond_unpack_grad": (_I, [C.POINTER(WnConfig), _VP, _I, _I, _VP, _VP]),
    "cmwg_wn_packed_bytes": (_SZ, [C.POINTER(WnConfig)]),
    "cmwg_wn_pack": (_I, [C.POINTER(WnConfig), C.POINTER(WnParams), _VP, _VP]),
    "cmwg_wn_workspace_bytes": (_SZ, [C.POINTER(WnConfig), _I, _I]),
    "cmwg_wn_saved_bytes": (_SZ, [C.POINTER(WnConfig), _I, _I]),
    "cmwg_wn_forward": (_I, [C.POINTER(WnConfig), _VP, _VP, _LL, _VP, _I, _I, _VP, _VP, _VP, _VP]),
    "cmwg_wn_varlen_workspace_bytes": (_SZ, [C.POINTER(WnConfig), _I, _I]),
    "cmwg_wn_forward_varlen": (_I, [C.POINTER(WnConfig), _VP, _VP, _LL, _VP, _I, _I, C.POINTER(C.c_int), _VP, _VP, _VP,
                                    _VP]),
    "cmwg_wn_line_state_bytes": (_SZ, [C.POINTER(WnConfig), _I, _I]),
    "cmwg_wn_forward_lines": (_I, [C.POINTER(WnConfig), _VP, _VP, _LL, _VP, _I, _I, _I, _I, _VP, _VP, _VP, _VP]),
    "cmwg_waveflow_affine": (_I, [_VP, _I, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, _VP]),
    "cmwg_waveflow_inverse_flow": (_I, [C.POINTER(WnConfig), _VP, _VP, _I, _VP, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "cmwg_waveflow_affine_bwd": (_I, [_VP, _VP, _VP, _I, _VP, _VP, _VP, _I, _I, _I, _VP]),
    "cmwg_upsample_dense_workspace": (_SZ, [_I, _I]),
    "cmwg_upsample_dense_fwd": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, C.c_float, _VP, _VP, _VP]),
    "cmwg_upsample_dense_bwd": (_I, [_VP, _VP, _VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, C.c_float, _VP, _VP, _VP,
                                     _VP, _VP]),
    "cmwg_wn_backward": (_I, [C.POINTER(WnConfig), C.POINTER(WnParams), _VP, _VP, _LL, _VP, _I, _I, _VP, _VP,
                              _VP, _VP, _LL, _VP, C.POINTER(WnGrads), _VP]),
    "cmwg_melspec_frames": (_I, [_I, _I, _I]),
    "cmwg_melspec_fwd": (_I, [_VP, _LL, _I, _I, _VP, _VP, _VP, _VP, _I, _I, _I, _I, C.c_float, _I, _VP, _VP]),
    "cmwg_denoise_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "cmwg_stft_frame_magnitude": (_I, [_VP, _I, _VP, _I, _I, _I, _VP, _VP]),
    "cmwg_denoise": (_I, [_VP, _LL, _I, _I, C.POINTER(C.c_int), _VP, _VP, _VP, C.c_float, _I, _I, _VP, _VP, _VP]),
    "cmwg_wsrglow_cond": (_I, [_VP, _I, _I, _VP, _I, _I, _VP, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "cmwg_lvc_gate_forward": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _I, _VP, _VP]),
    "cmwg_lvc_gate_backward": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP]),
    "cmwg_upsample_fwd": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP]),
    "cmwg_upsample_bwd_workspace": (_SZ, [_I, _I, _I]),
    "cmwg_upsample_bwd": (_I, [_VP, _VP, _VP, _VP, _LL, _LL, _I, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "cmwg_upsample_bwd_input": (_I, [_VP, _VP, _VP, _LL, _LL, _I, _I, _I, _I, _I, _I, _I, _VP, _VP]),
    "cmwg_squeeze": (_I, [_VP, _VP, _I, _I, _I, _I, _VP]),
    "cmwg_nll_loss": (_I, [_VP, _VP, _I, _I, C.c_float, _I, _VP, _VP, _VP, _VP]),
    "cmwg_sum_per_batch": (_I, [_VP, _LL, _I, _I, _VP, _I, C.c_float, _VP]),
    "cmwg_logdet_accumulate": (_I, [_VP, _LL, _I, _I, _VP, _VP, _VP, _VP]),
    "cmwg_logdet_accumulate_varlen": (_I, [_VP, _LL, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "cmwg_profile_enable": (_I, [_I]),
    "cmwg_profile_collect": (_I, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "cmwg_mega_clk_read": (_I, [C.POINTER(C.c_longlong), _I]),
    "cmwg_debug_counter": (C.c_ulonglong, [_I]),
    "cmwg_wgrad_plan_splits": (_I, [_I, _I, _I, _I]),
    "cmwg_mega_task_list": (_I, [_I, _I, _I, _I, C.POINTER(C.c_int), _I, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "cmwg_mega_task_list_varlen": (_I, [_I, _I, _I, C.POINTER(C.c_int), C.POINTER(C.c_int), _I, C.POINTER(C.c_int),
                                        C.POINTER(C.c_int), C.POINTER(C.c_int), _I, C.POINTER(C.c_int)]),
    "cmwg_selftest_tc_gemm": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _I, _VP]),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load (once) and return the ctypes handle; raises RuntimeError when the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"cmwg_b200: native library not found at {LIB_PATH}; build it with "
                "`python -m constant_memory_waveglow_b200.build` (there is no CPU / PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError -> missing export, fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().cmwg_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"cmwg_b200 {what} failed (code {rc}): {msg}")


def stream_ptr(device=None) -> int:
    """Raw cudaStream_t of torch's CURRENT stream (looked up at call time: the autograd engine may
    run backward on a different thread / stream than forward)."""
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def require_cuda(*tensors, op: str = "op") -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                f"cmwg_b200 {op}: expected CUDA tensors; this package has no CPU implementation "
                "(the CPU oracle lives in oracle/ and is test-only)")


def launch_count() -> int:
    return int(load().cmwg_launch_count())


def reset_launch_count() -> None:
    load().cmwg_reset_launch_count()
