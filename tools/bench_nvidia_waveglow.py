"""NVIDIA's WaveGlow on this package: the upsampler GEMM against the CUDA-core kernel, and synthesis rates.

Workload: the published configuration (80 mels, 12 flows, n_group 8, WN 8 x 256, kernel 3), random weights of a trained
model's magnitude (oracle/nvidia_glow.py randomize), sigma 0.6, default precision (fp16 operands), 22.05 kHz.
  upsampler    4 x 10 s of mel (861 frames each): cmwg_nvidia_upsample_slab (operand kernel + tcgen05 GEMM writing the
               fp16 WN slab) against the CUDA-core path to the same slab (cmwg_upsample_dense_fwd, FFMA, fp32 (B, 80, T)
               output, + unfold + cmwg_cond_pack), and against cmwg_upsample_dense_fwd alone; TFLOP/s from 13.1 MFLOP per
               frame (2 x 80 x 80 x 4 taps x 256 samples); share = time / one synthesis call of the same input.
  layered WN   NVIDIA's WN has a bias on every conv, which the single-kernel WN forward does not take, so it runs on the
               layered pipeline.  The same 4 x 10 s call with the biases dropped (same weights otherwise) runs on the task
               kernel; the kernel classes launched (cmwg_profile_collect) show which path each call took.
  synthesis    4 x 10 s in one call; the 64-utterance 1-8 s workload of tools/bench_varlen.py, one utterance per call and
               length-sorted batches of 16 with lengths; NVIDIA's model restated in PyTorch (oracle/nvidia_glow.py, weight
               norm removed as NVIDIA's inference.py does) in fp32 and fp16 on the same GPU, one utterance per call.
Rates count VALID samples only.  CUDA events around each pass, warm-up excluded, L2 flushed by a 256 MB write before every
pass.  Prints one JSON line and writes it to --out.

  python tools/bench_nvidia_waveglow.py [--reps 3] [--out profiles/r05_nvidia_waveglow_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import constant_memory_waveglow_b200 as cm  # noqa: E402
from constant_memory_waveglow_b200 import _lib as L  # noqa: E402
from constant_memory_waveglow_b200 import waveglow as W  # noqa: E402
from constant_memory_waveglow_b200.base import pad_batch  # noqa: E402
from oracle import nvidia_glow as NG  # noqa: E402

SR, HOP, SIGMA = 22050, 256, 0.6
PUBLISHED = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
                 WN_config=dict(n_layers=8, n_channels=256, kernel_size=3))
FLOP_PER_FRAME = 2 * 80 * 80 * 4 * 256


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return name, power
    except Exception as e:  # pragma: no cover
        return torch.cuda.get_device_name(), f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--utterances", type=int, default=64)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_nvidia_waveglow: needs a CUDA device")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    ref = NG.randomize(NG.WaveGlow(**PUBLISHED).double(), seed=0).float()
    model = cm.load_nvidia_waveglow(ref.state_dict())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b) / 1e3)
        return min(ts), sorted(ts)[len(ts) // 2]

    res = {}
    # ---- upsampler: 4 x 10 s ---------------------------------------------------------------------------------------
    g = torch.Generator().manual_seed(1)
    F10 = (10 * SR) // HOP
    h4 = torch.randn(4, 80, F10, generator=g).to(dev)
    z4 = (torch.randn(4, F10 * HOP, generator=g) * SIGMA).to(dev)
    Tq = F10 * HOP // 8
    lib = L.load()
    w = model.upsample.weight.detach().contiguous()
    bias = model.upsample.bias.detach().contiguous()
    Tout = (F10 - 1) * HOP + 1024
    ydense = torch.empty((4, 80, Tout), device=dev)
    wsd = torch.empty(int(lib.cmwg_upsample_dense_workspace(80, 1024)), device=dev, dtype=torch.uint8)

    def dense():
        L.check(lib.cmwg_upsample_dense_fwd(h4.data_ptr(), None, w.data_ptr(), bias.data_ptr(), 4, 80, F10, 1024, HOP, 0, 0,
                                            1.0, ydense.data_ptr(), wsd.data_ptr(), L.stream_ptr(dev)), "dense")

    cfg16 = model.WNs[0].F._config("fp16")

    def dense_to_slab():   # the exact path's conditioning, packed into the same 16-bit slab the GEMM writes
        W._CondCache().get(model._conditioning(h4, Tq, "fp32"), cfg16)

    # the same flow with the WN biases dropped: the WN forward can then run as the single task kernel
    nobias = cm.load_nvidia_waveglow(ref.state_dict())
    for coup in nobias.WNs:
        F = coup.F
        nb = cm.WN(F.in_chs, F.aux_chs, F.dil_chs, F.res_chs, F.skp_chs, len(F.layers), F.rdx, bias=False)
        nb.load_state_dict({k: v for k, v in F.state_dict().items() if not k.endswith("bias")})
        coup.F = nb.to(dev).eval()

    def classes(m):        # kernel classes launched by one 4 x 10 s synthesis call
        lib.cmwg_profile_enable(1)
        m.infer(h4, SIGMA, z=z4)
        ms, n = (C.c_double * 8)(), (C.c_longlong * 8)()
        L.check(lib.cmwg_profile_collect(ms, n), "profile_collect")
        lib.cmwg_profile_enable(0)
        return {"gate": n[0], "resskip": n[1], "fwd_task_kernel": n[6]}

    with torch.no_grad():
        t_gemm = timed(lambda: model._conditioning(h4, Tq, "fp16"), 20)
        t_dense_full = timed(dense_to_slab, 5)
        t_dense = timed(dense, 5)
        t_call = timed(lambda: model.infer(h4, SIGMA, z=z4), args.reps)
        t_nobias = timed(lambda: nobias.infer(h4, SIGMA, z=z4), args.reps)
        launched, launched_nobias = classes(model), classes(nobias)
    flop = FLOP_PER_FRAME * 4 * F10
    res["upsampler_4x10s"] = {
        "frames": 4 * F10, "gflop": flop / 1e9,
        "gemm_ms": t_gemm[0] * 1e3, "gemm_tflops": flop / t_gemm[0] / 1e12,
        "dense_path_to_slab_ms": t_dense_full[0] * 1e3, "dense_upsample_only_ms": t_dense[0] * 1e3,
        "dense_upsample_only_tflops": flop / t_dense[0] / 1e12,
        "speedup_vs_dense_path_to_slab": t_dense_full[0] / t_gemm[0], "speedup_vs_dense_upsample_only": t_dense[0] / t_gemm[0],
        "synthesis_call_ms": t_call[0] * 1e3,
        "gemm_share_of_call": t_gemm[0] / t_call[0], "dense_path_share_of_call": t_dense_full[0] / t_call[0]}
    res["synthesis_4x10s_mhz"] = 4 * F10 * HOP / t_call[0] / 1e6
    res["layered_wn_4x10s"] = {
        "with_bias_ms": t_call[0] * 1e3, "without_bias_ms": t_nobias[0] * 1e3, "ratio": t_call[0] / t_nobias[0],
        "launch_classes_with_bias": launched, "launch_classes_without_bias": launched_nobias}

    # ---- 64 utterances of 1-8 s (tools/bench_varlen.py's workload) --------------------------------------------------
    g = torch.Generator().manual_seed(1234)
    secs = torch.rand(args.utterances, generator=g) * 7 + 1
    frames = [max(1, int(s * SR) // HOP) for s in secs.tolist()]
    mels = [torch.randn(80, f, generator=g).to(dev) for f in frames]
    noise = [torch.randn(f * HOP, generator=g).to(dev) * SIGMA for f in frames]
    order = sorted(range(len(frames)), key=lambda i: frames[i])
    valid = sum(frames) * HOP
    batches = []
    for s0 in range(0, len(order), 16):
        idx = order[s0:s0 + 16]
        hb, fr = pad_batch([mels[i] for i in idx])
        zb, _ = pad_batch([noise[i] for i in idx])
        batches.append((hb, zb, fr))

    def solo():
        for i in range(len(frames)):
            model.infer(mels[i].unsqueeze(0), SIGMA, z=noise[i].unsqueeze(0))

    def varlen16():
        for hb, zb, fr in batches:
            model.infer(hb, SIGMA, z=zb, lengths=fr)

    nv = NG.WaveGlow(**PUBLISHED)
    nv.load_state_dict(ref.state_dict())
    for mod in nv.modules():
        if hasattr(mod, "weight_g"):
            torch.nn.utils.remove_weight_norm(mod)
    nv = nv.to(dev).eval()

    def pytorch_ref(m, dt):
        for i in range(len(frames)):
            m.infer(mels[i].unsqueeze(0).to(dt), noise[i].unsqueeze(0).to(dt))

    with torch.no_grad():
        t_solo = timed(solo, args.reps)
        t_var = timed(varlen16, args.reps)
        t_nv32 = timed(lambda: pytorch_ref(nv, torch.float32), 2)
        nvh = nv.half()
        t_nv16 = timed(lambda: pytorch_ref(nvh, torch.float16), 2)
    res["utterances_1_8s"] = {
        "n": len(frames), "valid_samples": valid,
        "solo_mhz": valid / t_solo[0] / 1e6, "varlen16_mhz": valid / t_var[0] / 1e6,
        "nvidia_pytorch_fp32_solo_mhz": valid / t_nv32[0] / 1e6, "nvidia_pytorch_fp16_solo_mhz": valid / t_nv16[0] / 1e6,
        "varlen16_over_nvidia_fp16": t_nv16[0] / t_var[0], "solo_over_nvidia_fp16": t_nv16[0] / t_solo[0]}
    name, power = gpu_info()
    res.update({"gpu": name, "power_limit": power, "precision": cm.get_precision(), "reps": args.reps,
                "timing": "min over reps of CUDA-event time per pass, L2 flushed before each pass"})
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
