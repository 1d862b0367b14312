#!/usr/bin/env python
"""Benchmark of the flow hot path (BASELINE.json metric: WaveGlow train segments/s at 1/2/4/8 B200,
synthesis kHz/GPU, % of roofline, next to the reference CPU path).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference (baseline/_ref) on the host cores

A "step" = one constant-memory training step (forward + NLL loss + reversible backward + gradient
all-reduce + Adam) of the WaveGlow LJ configuration (256 channels, 12 flows, 8 WN layers, 80 mel) on a
batch of 24 synthetic 16000-sample segments PER GPU (weak scaling; the line's `strong` object holds the
reference's own split, global batch 24 // N per GPU, train.py:51-53).  One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

LJ = dict(flows=12, n_group=8, n_early_every=4, n_early_size=2, hop_size=256, n_mels=80)
LJ_WN = dict(dilation_channels=256, residual_channels=256, skip_channels=256, depth=8, radix=3, bias=False)
SEGMENT = 16000
FRAMES = 63                      # MelSpec frames of a 16000-sample segment (SURVEY 8d)
PER_GPU_BATCH = 24
SIGMA = 0.7
FWD_GFLOP_PER_SEGMENT = 214.023  # algorithmic, counted on the reference (BASELINE.md section 4)
# dram__bytes_read.sum + dram__bytes_write.sum of ONE training-shape gate GEMM launch (B=24, R=48000 rows, the
# forward non-saving variant; 37.8 MB read + 1.1 MB written -- the 24.6 MB gate output is still in L2 when the
# kernel ends), from the `ncu --set full` capture summarised in profiles/r01_v5_ncu_gemm_summary.txt.
# Algorithmic bytes of the same launch: 48000 x (512 hi + 256 y in, 512 g out) = 61.4 MB.
GATE_TRAFFIC_BYTES_PER_LAUNCH = 38.9e6
# dram__bytes_read.sum + dram__bytes_write.sum per wn_fwd_mega_kernel launch at B=24, fp16 operands (ncu --set full,
# profiles/r02_s2_v5_ncu_task_kernels_summary.txt): 656.5 MB for the forward variant (290.5 read + 366.0 written: g per
# layer and the single-stream residual per layer; neither h_0, a `lo` slab nor the fp32 skip sum exists), 901.0 MB for the
# recompute variant that also stores the sigmoid (330.9 + 570.1); a step launches 12 of each.  (Round 2's first session:
# 1118 / 1662 MB; round 1: 1143 / 1760 MB.)
FUSED_TRAFFIC_BYTES_PER_LAUNCH = 0.5 * (656.5e6 + 901.0e6)
TRAIN_GFLOP_PER_SEGMENT = 4 * FWD_GFLOP_PER_SEGMENT
SYNTH_FRAMES = 862               # 10 s at 22.05 kHz -> 220672 samples (model/base.py:47-48)
GLOBAL_BATCH = 24                # configs/waveglow_LJ_speech.json:31; train.py:51-53 divides it by the GPU count
WSR_FWD_GFLOP_PER_SEGMENT = 234.978   # WSRGlow-2x, 8192-sample segment (SURVEY 8d)
WSR_SEGMENT, WSR_BATCH = 8192, 12     # configs/wsrglow_vctk_2x.json
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def workload_config(world: int, per_gpu_batch: int):
    """The `config` object of BOTH arms (the reference arm times a bounded sample of the same workload)."""
    return {"workload": "waveglow_lj_train_fwd+reversible_bwd+adam", "per_gpu_batch": per_gpu_batch, "segment": SEGMENT,
            "n_mels": 80, "channels": 256, "flows": 12, "wn_layers": 8,
            "l2": "256 MiB flush between timed steps; per-step working set >> 126 MB L2", "parallelism": f"dp{world}"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


# ---------------------------------------------------------------------------------------------
# clocks sampling
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML is polled in-process from a thread that is
    started before the warm-up (nvmlInit and an `nvidia-smi` start-up both take driver locks for 100+ ms, which
    must not land inside a timed step); samples are kept only while `active` is set.  `nvidia-smi -lms` is the
    fallback when pynvml cannot be used."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    MASKS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index = index
        self.rows = []          # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.active = False
        self.busy = False
        self.alive = False
        self.proc = None
        self.nvml = None
        self.handle = None
        self.thread = None

    def _open_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        self.nvml, self.handle = pynvml, h

    def start(self):
        """Open the sampler (call before the warm-up); sampling is recorded only between begin() and end()."""
        try:
            self._open_nvml()
            self.alive = True
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def begin(self):
        self.active = True

    def end(self):
        """Stop recording and wait for a query that is still in flight (on some boxes an NVML query takes tens of
        milliseconds and holds a driver lock the launch path needs: it must not reach into the next timed leg)."""
        self.active = False
        t0 = time.time()
        while self.busy and time.time() - t0 < 1.0:
            time.sleep(0.001)

    def sample_once(self):
        """One synchronous sample from the calling thread (used to top up a leg that got fewer than three)."""
        n = self.nvml
        if n is None:
            return
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        try:
            mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                bits = int(get_reasons(self.handle))
            except Exception:
                bits = 0
            self.rows.append((mhz, bits))
        except Exception:
            pass

    def _poll_nvml(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while self.alive:
            if self.active:
                self.busy = True
                try:
                    mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                    try:
                        bits = int(get_reasons(self.handle))
                    except Exception:
                        bits = 0
                    self.rows.append((mhz, bits))
                except Exception:
                    pass
                self.busy = False
                time.sleep(0.060)   # a query takes 1 ms on most boxes but 20-40 ms on some, holding a driver lock the
                                    # launch path needs: a few samples per timed leg are enough for the median   # NVML queries take a driver lock the launch path shares: keep them sparse
            else:
                time.sleep(0.001)

    def _read_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            if not self.active:
                continue
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) < 6:
                continue
            try:
                mhz = float(parts[0])
                self.max_mhz = float(parts[1])
            except ValueError:
                continue
            bits = 0
            for nme, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    bits |= self.MASKS[nme]
            self.rows.append((mhz, bits))

    def stop(self):
        self.active = False
        self.alive = False
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.nvml is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}
        if self.thread is not None and self.nvml is not None:
            self.thread.join(timeout=1)
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        reasons = sorted(k for k, m in self.MASKS.items() if bits & m)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_oracle_train(batch: int, steps: int, warmup: int):
    from oracle import flow_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    spec = O.WaveGlowSpec(**LJ)
    sd = O.random_state(spec, 256, 8, seed=0)
    g = torch.Generator().manual_seed(0)
    x = torch.rand(batch, SEGMENT, generator=g) * 2 - 1
    h = torch.randn(batch, LJ["n_mels"], FRAMES, generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.waveglow_train_step(sd, spec, x, h, SIGMA)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return batch / (sum(times) / len(times)), times


def cpu_oracle_synth(frames: int):
    """Oracle port of WaveGlow.infer on `frames` mel frames (one utterance), host cores; returns kHz."""
    from oracle import flow_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    spec = O.WaveGlowSpec(**LJ)
    sd = O.random_state(spec, 256, 8, seed=0)
    g = torch.Generator().manual_seed(0)
    h = torch.randn(1, LJ["n_mels"], frames, generator=g)
    z = torch.randn(1, frames * LJ["hop_size"], generator=g) * 0.6
    with torch.no_grad():
        O.waveglow_infer(sd, spec, h[..., :8], z[:, :8 * LJ["hop_size"]])   # warm-up
        t0 = time.perf_counter()
        O.waveglow_infer(sd, spec, h, z)
        dt = time.perf_counter() - t0
    return frames * LJ["hop_size"] / dt / 1e3, dt


WAVEFLOW = dict(flows=8, n_group=64, n_mels=80, use_conv1x1=False)       # configs/waveflow_LJ_speech.json:6-15
WAVEFLOW_WN = dict(dilation_channels=64, residual_channels=64, skip_channels=64, bias=False)
WAVEFLOW_BATCH = 12                                                       # configs/waveflow_LJ_speech.json:31
WAVEFLOW_FWD_GFLOP_PER_SEGMENT = 164.502                                  # SURVEY.md section 8d


def waveflow_leg(dev, cpu_baseline: bool):
    """Config 4 (WaveFlow, 64 residual channels, h = 64): training step (forward + loss + plain backward) in
    segments/s and synthesis of one 10 s utterance in kHz, on one GPU."""
    import constant_memory_waveglow_b200 as cm
    torch.manual_seed(0)
    m = cm.WaveFlow(memory_efficient=False, zero_init=False, **WAVEFLOW, **WAVEFLOW_WN).to(dev).train()
    loss_fn = cm.WaveGlowLoss(SIGMA)
    B = WAVEFLOW_BATCH
    x = torch.rand(B, SEGMENT, device=dev) * 2 - 1
    h = torch.randn(B, 80, FRAMES, device=dev)

    def step():
        m.zero_grad(set_to_none=True)
        z, ld = m(x, h)
        loss = loss_fn(z, ld)
        loss.backward()
        return loss

    def timed(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    for _ in range(3):
        step()
    ms_train = timed(step, 5)
    m.eval()
    hs = torch.randn(1, 80, SYNTH_FRAMES, device=dev)
    zs = torch.randn(1, SYNTH_FRAMES * 256, device=dev) * 0.6
    with torch.no_grad():
        for _ in range(2):
            m.infer(hs, 0.6, z=zs)
        ms_synth = timed(lambda: m.infer(hs, 0.6, z=zs), 3)
    out = {"config": {"workload": "waveflow_lj (8 flows, n_group 64, 64 channels)", "train_batch": B, "segment": SEGMENT,
                      "synth_batch": 1, "utterance_samples": SYNTH_FRAMES * 256},
           "train_segments_per_s": B / (ms_train * 1e-3), "train_ms_per_step": ms_train,
           "train_tflops": 3 * B * WAVEFLOW_FWD_GFLOP_PER_SEGMENT / ms_train,
           "synth_khz": SYNTH_FRAMES * 256 / ms_synth, "synth_ms": ms_synth,
           "synth_note": "row-recurrent (63 sequential rows x 8 flows), replayed as one CUDA graph"}
    if cpu_baseline:
        from oracle import flow_oracle as O
        spec = O.WaveFlowSpec(8, 64, 80)
        sd = O.waveflow_random_state(spec, 64, seed=0)
        g = torch.Generator().manual_seed(0)
        xc = torch.rand(1, SEGMENT, generator=g) * 2 - 1
        hc = torch.randn(1, 80, FRAMES, generator=g)
        O.waveflow_train_step(sd, spec, xc[:, :4096], hc[..., :16], SIGMA)
        t0 = time.perf_counter()
        O.waveflow_train_step(sd, spec, xc, hc, SIGMA)
        t_train = time.perf_counter() - t0
        with torch.no_grad():
            t0 = time.perf_counter()
            O.waveflow_reverse(sd, spec, xc * 0.6, hc)
            t_syn = time.perf_counter() - t0
        out["cpu_baseline"] = {"train_segments_per_s": 1.0 / t_train, "synth_khz": SEGMENT / t_syn / 1e3,
                               "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"oracle port, 1 training step of 1 x 16000 samples ({t_train:.1f} s) and the "
                                         f"row-recurrent reverse of 16000 samples ({t_syn:.1f} s)"}
    return out


CPU_SAMPLE_BATCH = 2   # segments per CPU step: ~2 s per step on 16 host cores, so K+W steps stay within minutes


def import_reference():
    """The UNMODIFIED reference tree (baseline/_ref, a copy of /root/reference made by __graft_entry__.build()) as the
    top-level packages `model` / `utils` / `datasets` it expects to be; nothing of this repository is on that path.
    Only `pytorch_lightning`, which this image does not have, is replaced by an in-memory stub (model/lightning.py:5
    needs the name at import time; the benchmark never touches Lightning).  Returns the `model` package or None."""
    if not os.path.exists(os.path.join(REF_DIR, "model", "efficient_modules.py")):
        return None
    import types
    import warnings
    warnings.filterwarnings("ignore")
    if "pytorch_lightning" not in sys.modules:
        try:
            import importlib.util
            have = importlib.util.find_spec("pytorch_lightning") is not None and \
                not os.path.abspath(importlib.util.find_spec("pytorch_lightning").origin).startswith(ROOT)
        except Exception:
            have = False
        if not have:
            pl = types.ModuleType("pytorch_lightning")

            class _LM(torch.nn.Module):
                def save_hyperparameters(self, *a, **k):
                    pass

            pl.LightningModule, pl.Callback, pl.Trainer = _LM, object, object
            sys.modules["pytorch_lightning"] = pl
    for name in list(sys.modules):
        if name in ("model", "utils", "datasets") or name.startswith(("model.", "datasets.")):
            del sys.modules[name]
    sys.path[:] = [REF_DIR] + [q for q in sys.path if os.path.abspath(q or ".") != ROOT]
    import model as ref_model
    assert os.path.abspath(ref_model.__file__).startswith(REF_DIR), ref_model.__file__
    return ref_model


def ref_waveglow(ref_model, seed=0):
    torch.manual_seed(seed)
    m = ref_model.WaveGlow(memory_efficient=True, zero_init=False, **LJ, **LJ_WN)
    from model.loss import WaveGlowLoss
    return m, WaveGlowLoss(SIGMA)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    task = args.ref_task
    ref = import_reference()
    kind = "reference" if ref is not None else "port"
    if ref is None:
        sys.path.insert(0, ROOT)
    g = torch.Generator().manual_seed(0)

    if task == "train":
        batch = CPU_SAMPLE_BATCH
        x = torch.rand(batch, SEGMENT, generator=g) * 2 - 1
        h = torch.randn(batch, LJ["n_mels"], FRAMES, generator=g)
        if ref is not None:
            m, loss_fn = ref_waveglow(ref)
            m.train()
            opt = torch.optim.Adam(m.parameters(), lr=1e-4)
            times = []
            for i in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                opt.zero_grad(set_to_none=True)
                z, logdet = m(x.clone(), h)
                loss = loss_fn(z, logdet)
                loss.backward()
                opt.step()
                dt = time.perf_counter() - t0
                if i >= args.warmup:
                    times.append(dt)
            value = batch / (sum(times) / len(times))
            what = ("baseline/_ref (the unmodified reference): model.WaveGlow(memory_efficient=True) + WaveGlowLoss + "
                    "torch.optim.Adam on CPU fp32")
        else:
            value, times = cpu_oracle_train(batch, args.steps, args.warmup)
            what = "oracle port of the reference (baseline/_ref missing), autograd over the naive flow, no optimizer"
        line = {
            "impl": "reference", "metric": "waveglow_lj_train_segments_per_s", "value": value, "unit": "segments/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, PER_GPU_BATCH), "sample_batch": batch,
            "cpu_baseline": {"value": value, "unit": "segments/s", "cores": cores, "kind": kind,
                             "sample": f"{what}; each step = {batch} of the workload's {PER_GPU_BATCH} segments x {SEGMENT} "
                                       f"samples: forward + loss + reversible backward + Adam, {sum(times):.1f} s timed"},
            "e2e": {"value": value, "unit": "segments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line), flush=True)
        return

    if task == "synth":      # one 10 s utterance through the reference's inverse (inference.py:50-56 times exactly this)
        frames = SYNTH_FRAMES
        h = torch.randn(1, LJ["n_mels"], frames, generator=g)
        if ref is not None:
            m, _ = ref_waveglow(ref)
            import utils as ref_utils
            m.apply(ref_utils.remove_weight_norms)   # inference.py:17
            m.eval()
            with torch.no_grad():
                m.infer(h[..., :32], 0.6)
                t0 = time.perf_counter()
                m.infer(h, 0.6)
                dt = time.perf_counter() - t0
            khz = frames * LJ["hop_size"] / dt / 1e3
        else:
            khz, dt = cpu_oracle_synth(frames)
        print(json.dumps({"khz": khz, "seconds": dt, "cores": cores, "kind": kind, "frames": frames}), flush=True)
        return

    if task == "parity":     # seeded weights / inputs and the reference's own outputs, for the B200 arm to compare with
        if ref is None:
            print(json.dumps({"unavailable": "baseline/_ref missing"}), flush=True)
            return
        m, loss_fn = ref_waveglow(ref, seed=0)
        m.train()
        B = 2
        x = torch.rand(B, SEGMENT, generator=g) * 2 - 1
        h = torch.randn(B, LJ["n_mels"], FRAMES, generator=g)
        zs = torch.randn(B, FRAMES * LJ["hop_size"], generator=g) * 0.6
        state = {k: v.clone() for k, v in m.state_dict().items()}
        z, logdet = m(x.clone(), h)
        loss = loss_fn(z, logdet)
        loss.backward()
        grads = {n: p.grad.clone() for n, p in m.named_parameters()}
        with torch.no_grad():
            m.eval()
            audio, _ = m.reverse(zs.clone(), h)
            xr, _ = m.reverse(z.detach().clone(), h)
        torch.save({"state": state, "x": x, "h": h, "zs": zs, "z": z.detach(), "logdet": logdet.detach(),
                    "loss": loss.detach(), "grads": grads, "audio": audio, "ref_roundtrip_rel_l2":
                    ((xr - x).norm() / x.norm()).item()}, args.out)
        print(json.dumps({"ok": True, "kind": kind}), flush=True)
        return

    if task == "wsrglow":    # config 5: one training step and one inverse of a single 8192-sample segment
        x = torch.rand(1, WSR_SEGMENT, generator=g) * 2 - 1
        c = torch.rand(1, WSR_SEGMENT // 2, generator=g) * 2 - 1
        if ref is not None:
            torch.manual_seed(0)
            m = ref.WSRGlow(upsample_rate=2, memory_efficient=True, zero_init=False)
            from model.loss import WaveGlowLoss
            loss_fn = WaveGlowLoss(1.0)
            m.train()
            ts = []
            for _ in range(2):
                t0 = time.perf_counter()
                m.zero_grad(set_to_none=True)
                z, logdet = m(x.clone(), c.clone())
                loss_fn(z, logdet).backward()
                ts.append(time.perf_counter() - t0)
            with torch.no_grad():
                m.eval()
                t0 = time.perf_counter()
                m.reverse(z.detach().clone(), c.clone())
                t_inv = time.perf_counter() - t0
            t_train = min(ts)
        else:
            from oracle import flow_oracle as O
            spec = O.wsrglow_spec(2)
            sd = O.wsrglow_random_state(2, 256, 8, seed=0)
            t0 = time.perf_counter()
            z, _, _, _ = O.wsrglow_train_step(sd, spec, x, c, 1.0)
            t_train = time.perf_counter() - t0
            with torch.no_grad():
                t0 = time.perf_counter()
                O.wsrglow_reverse(sd, spec, z.detach(), c)
                t_inv = time.perf_counter() - t0
        print(json.dumps({"train_segments_per_s": 1.0 / t_train, "inverse_khz": WSR_SEGMENT / t_inv / 1e3, "cores": cores,
                          "kind": kind, "train_seconds": t_train, "inverse_seconds": t_inv}), flush=True)
        return


def reference_subprocess(task: str, extra=(), timeout=600):
    """Run one reference-arm task in its own interpreter (the reference's `model` / `utils` / `datasets` packages share
    their names with this repository's drop-in shims, so they never live in one process) and parse its JSON line."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-task", task, *extra]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (r.stderr or r.stdout)[-400:]}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200(args):
    import torch.distributed as dist
    import constant_memory_waveglow_b200 as cm
    from constant_memory_waveglow_b200 import _lib, precision
    from constant_memory_waveglow_b200.parallel import FlowGradSync, flow_buckets

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    precision.set_precision(args.precision)
    lib = _lib.load()

    torch.manual_seed(0)
    model = cm.WaveGlow(memory_efficient=True, zero_init=False, **LJ, **LJ_WN).to(dev).train()
    loss_fn = cm.WaveGlowLoss(SIGMA)
    sync = FlowGradSync(flow_buckets(model))
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True, capturable=True)
    from constant_memory_waveglow_b200.graphs import GraphedTrainStep
    # the whole step as one CUDA graph per batch shape (constant_memory_waveglow_b200/graphs.py): same kernels, same order,
    # one launch; --no-graph times the eager step (Python issuing every launch through autograd)
    gstep = None if args.no_graph else GraphedTrainStep(model, lambda x_, h_: loss_fn(*model(x_, h_)), opt, sync)

    B = args.batch
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = (torch.rand(B, SEGMENT, generator=g) * 2 - 1).pin_memory()
    h_host = torch.randn(B, LJ["n_mels"], FRAMES, generator=g).pin_memory()
    x_dev, h_dev = x_host.to(dev), h_host.to(dev)
    Bs = max(1, GLOBAL_BATCH // world)                     # the reference's split (train.py:51-53)
    xs_dev, hs_dev = x_dev[:Bs].clone(), h_dev[:Bs].clone()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    phase_ms = []

    def trace(msg):
        if os.environ.get("CMWG_BENCH_TRACE") == "1":
            torch.cuda.synchronize()
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    def step(x, h, eager=False):
        if gstep is not None and not eager:
            return gstep(x, h)
        x, h = x.to(dev, non_blocking=True), h.to(dev, non_blocking=True)
        if os.environ.get("CMWG_BENCH_DEBUG") == "1":
            t = [time.perf_counter()]
            sync.zero_grad(); t.append(time.perf_counter())
            z, logdet = model(x, h); t.append(time.perf_counter())
            loss = loss_fn(z, logdet); t.append(time.perf_counter())
            loss.backward(); t.append(time.perf_counter())
            sync.finish(); t.append(time.perf_counter())
            opt.step(); t.append(time.perf_counter())
            ms_ = torch.cuda.memory_stats()
            phase_ms.append([round((b - a) * 1e3, 1) for a, b in zip(t[:-1], t[1:])] +
                            [ms_["num_device_alloc"], ms_["num_device_free"], ms_["num_alloc_retries"],
                             ms_["reserved_bytes.all.current"] >> 20, int(lib.cmwg_debug_counter(0)), int(lib.cmwg_debug_counter(1))])
            return loss
        sync.zero_grad()
        z, logdet = model(x, h)
        loss = loss_fn(z, logdet)
        loss.backward()
        sync.finish()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_ms = {False: [], True: []}
    dbg_host = []

    def timed(nsteps, e2e):
        total_ms = 0.0
        last = None
        for _ in range(nsteps):
            flush.zero_()                                  # evict L2 between timed iterations
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a.record()
            if e2e and os.environ.get("CMWG_BENCH_DEBUG") == "1":
                t0 = time.perf_counter()
                t1 = time.perf_counter()
                lt = step(x_host, h_host)
                t2 = time.perf_counter()
                last = lt.item()
                t3 = time.perf_counter()
                dbg_host.append([round((t1 - t0) * 1e3, 2), round((t2 - t1) * 1e3, 2), round((t3 - t2) * 1e3, 2)])
            elif e2e:
                # the inputs are temporaries, as in the warm-up: keeping last step's tensors bound while the next ones
                # are created asks the caching allocator for one more 2 MB segment in the second step, and a cudaMalloc
                # issued while the device is busy stalled that step's backward by 60-200 ms
                last = step(x_host, h_host).item()  # H2D from pinned memory inside step(), + D2H read of the loss
            else:
                last = step(x_dev, h_dev)
            b.record()
            barrier()
            total_ms += a.elapsed_time(b)
            step_ms[e2e].append(round(a.elapsed_time(b), 3))
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), last

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                    # opened before the warm-up, records only while active
    for _ in range(args.warmup):
        step(x_dev, h_dev)
    for _ in range(min(args.warmup, 2)):                   # warm the pinned-host -> device path of the e2e leg too
        step(x_host, h_host).item()
    barrier()

    import gc
    gc.collect()
    gc.disable()                                           # no collector pauses inside a timed step
    trace("warm-up done")
    sampler.begin()
    lib.cmwg_reset_launch_count()
    ms, loss = timed(args.steps, e2e=False)
    launches = int(lib.cmwg_launch_count())
    if gstep is not None:
        launches = gstep.launches_per_step * args.steps    # counted while the step was captured; every replay runs them all
    if os.environ.get("CMWG_BENCH_SAMPLE_E2E", "0") != "1":
        sampler.end()      # clocks are sampled over the device-resident leg (the timed region of `value`): an NVML query
                           # holds a driver lock, and the e2e leg -- whose host thread cannot run ahead of the device
                           # because it reads the loss back every step -- showed 60-100 ms stalls with the sampler on
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, loss)       # now: every later leg steps the model again
    # the e2e leg allocates its inputs per step, which shifts where the caching allocator places everything after them:
    # let it reach its steady state (two alternating layouts) before timing
    for _ in range(min(args.warmup, 3)):
        step(x_host, h_host).item()
    trace("device-resident leg done")
    ms_e2e, loss_e2e = timed(args.steps, e2e=True)
    trace("e2e leg done")
    sampler.end()
    if rank == 0 and sampler.nvml is not None and len(sampler.rows) < 3:
        # slow NVML on this box: top the clock samples up under the same load (untimed steps in flight)
        for _ in range(3):
            step(x_dev, h_dev, eager=True)
        for _ in range(3):
            sampler.sample_once()
            time.sleep(0.01)
        torch.cuda.synchronize()
    gc.enable()
    clocks = sampler.stop() if rank == 0 else None

    # ---- reference-semantics split: global batch 24 divided over the GPUs (24 // N segments per GPU), same timing rules
    strong = None
    if world > 1 and not args.no_strong:
        for _ in range(args.warmup):
            step(xs_dev, hs_dev)
        barrier()
        tot = 0.0
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a.record()
            step(xs_dev, hs_dev)
            b.record()
            barrier()
            tot += a.elapsed_time(b)
        t = torch.tensor([tot], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong = {"value": world * Bs * args.steps / (t.item() * 1e-3), "unit": "segments/s", "scaling": "strong",
                  "global_batch": world * Bs, "per_gpu_batch": Bs, "ms_per_step": t.item() / args.steps,
                  "note": "train.py:51-53 semantics: batch_size //= gpus; row tiles per GPU = per_gpu_batch * 8 for 74 CTA pairs"}

    trace("strong leg done")
    # ---- roofline leg: device time of every GEMM class over one more step (events on the launching stream)
    import ctypes as C
    # eager steps (the per-class CUDA events sit between the launches); two untimed ones first -- the legs above replay
    # graphs, and the first eager step after them pays for re-encoded tensor maps and a clock ramp -- then the mean of three
    ROOF_STEPS = 3
    for _ in range(2):
        step(x_dev, h_dev, eager=True)
    torch.cuda.synchronize()
    lib.cmwg_profile_enable(1)
    for _ in range(ROOF_STEPS):
        step(x_dev, h_dev, eager=True)
    torch.cuda.synchronize()
    kms = (C.c_double * 8)()
    kn = (C.c_longlong * 8)()
    _lib.check(lib.cmwg_profile_collect(kms, kn), "profile_collect")
    lib.cmwg_profile_enable(0)
    names = ["gate", "resskip", "dgate", "dx", "dcond", "wgrad", "fwdfused", "bwdfused"]
    kern = {n: {"ms": kms[i] / ROOF_STEPS, "launches": int(kn[i]) // ROOF_STEPS} for i, n in enumerate(names)}

    trace("roofline leg done")
    # ---- synthesis (config 3): sigma 0.6, 10 s utterances, utterance-sharded, no collective
    synth = None
    if not args.no_synth:
        model.eval()
        sb = args.synth_batch
        hs_host = torch.randn(sb, LJ["n_mels"], SYNTH_FRAMES).pin_memory()
        audio_host = torch.empty(sb, SYNTH_FRAMES * LJ["hop_size"]).pin_memory()
        hs = hs_host.to(dev)
        zs = torch.randn(sb, SYNTH_FRAMES * LJ["hop_size"], device=dev) * 0.6
        samples = sb * SYNTH_FRAMES * LJ["hop_size"]
        pk = peaks()

        def timed_synth(fn, reps=3):
            with torch.no_grad():
                for _ in range(2):
                    fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                barrier()
                a.record()
                for _ in range(reps):
                    fn()
                b.record()
                barrier()
            t = torch.tensor([a.elapsed_time(b) / reps], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()

        ms_dev = timed_synth(lambda: model.infer(hs, 0.6, z=zs))

        def synth_e2e():
            # the call a user makes (inference.py:50-56): mel from pinned host memory, noise drawn on the device by infer(),
            # audio back to the host
            audio_host.copy_(model.infer(hs_host.to(dev, non_blocking=True), 0.6).view(sb, -1), non_blocking=True)

        ms_e2e_s = timed_synth(synth_e2e)
        # roofline of the synthesis path's dominant kernel: the non-saving forward task kernel, 12 launches per call
        lib.cmwg_profile_enable(1)
        with torch.no_grad():
            model.infer(hs, 0.6, z=zs)
        torch.cuda.synchronize()
        sms, sn = (C.c_double * 8)(), (C.c_longlong * 8)()
        _lib.check(lib.cmwg_profile_collect(sms, sn), "profile_collect")
        lib.cmwg_profile_enable(0)
        srows = sb * SYNTH_FRAMES * LJ["hop_size"] // LJ["n_group"]
        sflops = srows * (8 * 2.0 * 512 * (3 * 256 + 80) + 7 * 2.0 * 256 * 256 + 8 * 2.0 * 256 * 256)
        s_ms = sms[6] / max(int(sn[6]), 1)
        s_ach = sflops / (s_ms * 1e-3) / 1e12 if s_ms > 0 else 0.0
        khz = world * samples / (ms_dev * 1e-3) / 1e3
        synth = {"metric": "waveglow_lj_synth_khz", "value": khz, "unit": "kHz (all GPUs)", "per_gpu_khz": khz / world,
                 "batch_per_gpu": sb, "utterance_samples": SYNTH_FRAMES * LJ["hop_size"], "sigma": 0.6, "ms": ms_dev,
                 "operand_dtype": precision.resolve(True, False),
                 "e2e": {"value": world * samples / (ms_e2e_s * 1e-3) / 1e3, "unit": "kHz (all GPUs)", "ms": ms_e2e_s,
                         "h2d_bytes_per_step": int(hs_host.numel() * 4), "d2h_bytes_per_step": int(audio_host.numel() * 4)},
                 "tflops_per_gpu": samples * 13.3764e6 / (ms_dev * 1e-3) / 1e12,
                 "frac_of_bf16_peak": samples * 13.3764e6 / (ms_dev * 1e-3) / 1e12 / pk["tflops_sustained"],
                 "roofline": {"bound": "tensor", "kernel": "wn_fwd_mega_kernel<no saves>", "achieved": s_ach,
                              "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": s_ach / pk["tflops_sustained"],
                              "flops_per_launch": sflops, "ms_per_launch": s_ms, "launches_per_call": int(sn[6]),
                              "traffic": None}}
        # batch sweep of config 3 (10 s utterances, batch 1-64 per GPU): kHz per GPU at each batch size
        if not args.no_synth_sweep:
            sweep = {}
            for sbb in (1, 4, 16, 64):
                hb = torch.randn(sbb, LJ["n_mels"], SYNTH_FRAMES, device=dev)
                zb = torch.randn(sbb, SYNTH_FRAMES * LJ["hop_size"], device=dev) * 0.6
                with torch.no_grad():
                    model.infer(hb, 0.6, z=zb)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    a.record()
                    for _ in range(2):
                        model.infer(hb, 0.6, z=zb)
                    b.record()
                    torch.cuda.synchronize()
                sweep[str(sbb)] = round(sbb * SYNTH_FRAMES * LJ["hop_size"] / (a.elapsed_time(b) / 2 * 1e-3) / 1e3, 1)
                del hb, zb
            synth["per_gpu_khz_by_batch"] = sweep
            torch.cuda.empty_cache()
        model.train()

    if rank != 0:
        finish_ranks(world)
        return

    pk = peaks()
    segs = world * B * args.steps
    value = segs / (ms * 1e-3)
    value_e2e = segs / (ms_e2e * 1e-3)
    rows = B * (SEGMENT // LJ["n_group"])
    gate_flops = 2.0 * rows * 512 * (3 * 256 + 80)          # algorithmic: 80 mel rows, not the padded 128
    gate = kern["gate"]
    roof_kernel = "tc_gemm_kernel<gate epilogue> (dilated conv + conditioning GEMM)"
    roof_traffic = GATE_TRAFFIC_BYTES_PER_LAUNCH
    if kern["fwdfused"]["launches"] > 0:
        # single-kernel WN forward: per launch all 8 gate GEMMs, 7 residual and 8 skip contractions of one WN
        gate = kern["fwdfused"]
        gate_flops = rows * (8 * 2.0 * 512 * (3 * 256 + 80) + 7 * 2.0 * 256 * 256 + 8 * 2.0 * 256 * 256)
        roof_kernel = "wn_fwd_mega_kernel (all gate / residual / skip GEMM tiles of one WN forward)"
        roof_traffic = FUSED_TRAFFIC_BYTES_PER_LAUNCH
    gate_ms = gate["ms"] / max(gate["launches"], 1)
    achieved = gate_flops / (gate_ms * 1e-3) / 1e12 if gate_ms > 0 else 0.0
    total_kernel_ms = sum(v["ms"] for v in kern.values())
    mode = precision.resolve(True, True)
    line = {
        "metric": "waveglow_lj_train_segments_per_s", "value": value, "unit": "segments/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": {"bf16": "bf16", "fp32": "f32", "fp16": "fp16"}[mode],
        "operand_precision": {"fp16": "fp16 operands (10 mantissa bits = TF32's), fp32 accumulate in TMEM, power-of-two "
                                      "gradient scale chosen on the device", "bf16": "bf16 operands, fp32 accumulate",
                              "fp32": "fp32 FFMA engine"}[mode],
        "data": "synthetic",
        "config": workload_config(world, B), "loss": float(loss.detach()),
        "e2e": {"value": value_e2e, "unit": "segments/s", "h2d_bytes_per_step": int(x_host.numel() * 4 + h_host.numel() * 4),
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "launch_mode": "eager (one Python-issued launch per kernel)" if gstep is None else
                       f"one CUDA graph per step ({gstep.launches_per_step} kernels of libcmwg_b200.so per replay, + optimizer / torch glue)",
        "ms_per_timed_step": {"device_resident": step_ms[False], "e2e": step_ms[True]},
        **({"debug_e2e_host_ms_copy_enqueue_wait": dbg_host, "debug_phase_ms_zero_fwd_loss_bwd_finish_opt": phase_ms[-2 * args.steps - 1:]} if dbg_host else {}),
        "train_tflops_per_gpu": B * TRAIN_GFLOP_PER_SEGMENT / (ms / args.steps),
        "roofline": {"bound": "tensor", "kernel": roof_kernel,
                     "achieved": achieved, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / pk["tflops_sustained"], "traffic": roof_traffic,
                     "peak_source": pk["source"],
                     "flops_per_launch": gate_flops, "ms_per_launch": gate_ms, "launches_per_step": gate["launches"],
                     "share_of_gemm_time": gate["ms"] / total_kernel_ms if total_kernel_ms else None,
                     "kernel_classes_ms_per_step": {k: round(v["ms"], 3) for k, v in kern.items()}},
        "clocks": clocks,
        "synth": synth,
    }
    if strong is not None:
        line["strong"] = strong
    want_cpu = not args.no_cpu_baseline and world == 1
    # ---- parity of THIS arm's precision mode against the unmodified reference on the same weights and inputs
    if want_cpu and not args.no_parity:
        line["parity"] = parity_leg(model, loss_fn, dev, args)
    del opt, sync, gstep
    if not args.no_wsrglow and world == 1:
        del model
        model = None
        torch.cuda.empty_cache()
        line["wsrglow"] = wsrglow_leg(dev, flush, want_cpu)
    if not args.no_waveflow and world == 1:
        model = None
        torch.cuda.empty_cache()
        line["waveflow"] = waveflow_leg(dev, not args.no_cpu_baseline)
    if want_cpu and synth is not None:
        r = reference_subprocess("synth")                     # the same 10 s utterance, a few seconds of CPU work
        if "khz" in r:
            synth["cpu_baseline"] = {"value": r["khz"], "unit": "kHz", "cores": r["cores"], "kind": r["kind"],
                                     "sample": f"one utterance of {SYNTH_FRAMES} frames = {SYNTH_FRAMES * 256} samples through "
                                               f"the reference's infer() after remove_weight_norms, {r['seconds']:.1f} s"}
            synth["x_cpu_per_gpu"] = synth["per_gpu_khz"] / r["khz"]
        else:
            synth["cpu_baseline"] = r
    if want_cpu:
        r = reference_subprocess("train", ["--steps", "6", "--warmup", "1"])   # ~15-25 s of CPU work
        line["cpu_baseline"] = r.get("cpu_baseline", r)
    print(json.dumps(line), flush=True)
    finish_ranks(world)


def finish_ranks(world):
    """End of a multi-rank run: the ranks meet once more, then tear the process group down -- under a watchdog.  One N = 2
    run of this round printed its line and then sat in `destroy_process_group()` until the box's time limit (one rank had
    left, the other waited inside NCCL's teardown); the measurement is complete by then, so a teardown that does not return
    within 20 s ends the process instead of the run."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    wd = threading.Timer(20.0, lambda: os._exit(0))
    wd.daemon = True
    wd.start()
    try:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    finally:
        wd.cancel()


DUMP_SAMPLE_PER_TENSOR = 4096
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, model, loss):
    """What the last timed training step hands its caller, as .npy files in `out_dir`, so that two builds can be compared
    output for output: `loss.npy` (float64 scalar), and `grad_sample.npy` / `param_sample.npy` (float32), every parameter's
    gradient and updated value at up to DUMP_SAMPLE_PER_TENSOR positions per tensor, concatenated in `named_parameters()`
    order.  The positions come from a fixed seed and the parameter shapes alone, so they are the same in every run; at the
    LJ configuration the three files hold 8 MB; more than DUMP_MAX_BYTES is refused before anything is written.  Everything
    is copied to the host first: no device memory is allocated between the timed legs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    gen = torch.Generator().manual_seed(0)
    grads, params = [], []
    for name, p in model.named_parameters():
        assert p.grad is not None, f"no gradient for {name}"
        n = p.numel()
        idx = torch.randperm(n, generator=gen)[:DUMP_SAMPLE_PER_TENSOR].sort().values if n > DUMP_SAMPLE_PER_TENSOR \
            else torch.arange(n)
        params.append(p.detach().cpu().reshape(-1)[idx])
        grads.append(p.grad.detach().cpu().reshape(-1)[idx])
    arrays = {"loss": np.array(loss.detach().item(), dtype=np.float64), "grad_sample": torch.cat(grads).float().numpy(),
              "param_sample": torch.cat(params).float().numpy()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def parity_leg(model, loss_fn, dev, args):
    """z / log-det / loss / every parameter gradient / synthesis audio / round trip of the CUDA path in the precision mode
    being benchmarked, against the UNMODIFIED reference (baseline/_ref, CPU fp32) on the same random-init weights and inputs
    (LJ config, 2 segments): the reference process writes its state dict and results, this one loads the state dict."""
    from constant_memory_waveglow_b200 import precision
    with tempfile.TemporaryDirectory(prefix="cmwg_parity_") as tmp:      # the benchmarked tree may be read-only
        out = os.path.join(tmp, "ref_parity.pt")
        r = reference_subprocess("parity", ["--out", out])
        if not r.get("ok"):
            return {"unavailable": r}
        fx = torch.load(out, map_location="cpu", weights_only=False)
    keep = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model.load_state_dict(fx["state"])
    model.train()
    for p_ in model.parameters():
        p_.grad = None

    def rel(a, b):
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()

    z, logdet = model(fx["x"].to(dev), fx["h"].to(dev))
    loss = loss_fn(z, logdet)
    loss.backward()
    num = den = 0.0
    worst = ("", 0.0)
    for n, p_ in model.named_parameters():
        gr = fx["grads"][n].double()
        e2 = (p_.grad.double().cpu() - gr).pow(2).sum().item()
        d2 = gr.pow(2).sum().item()
        num += e2
        den += d2
        e = (e2 / max(d2, 1e-300)) ** 0.5
        if e > worst[1]:
            worst = (n, e)
    with torch.no_grad():
        model.eval()
        xr, _ = model.reverse(z.detach().clone(), fx["h"].to(dev))
        audio, _ = model.reverse(fx["zs"].to(dev), fx["h"].to(dev))
    out = {"against": "baseline/_ref (unmodified reference, CPU fp32), LJ config, 2 x 16000 samples, same state dict",
           "mode": precision.resolve(True, True), "z_rel_l2": rel(z, fx["z"]), "logdet_rel_l2": rel(logdet, fx["logdet"]),
           "loss_rel": abs(loss.item() - fx["loss"].item()) / abs(fx["loss"].item()),
           "grad_rel_l2_aggregate": (num / max(den, 1e-300)) ** 0.5,
           "grad_rel_l2_worst": {"tensor": worst[0], "rel_l2": worst[1]},
           "audio_rel_l2": rel(audio, fx["audio"]), "roundtrip_rel_l2": rel(xr, fx["x"]),
           "reference_roundtrip_rel_l2": fx["ref_roundtrip_rel_l2"],
           "tolerance": "north_star: rel-L2 <= 1e-3 (tensor-core operands), <= 1e-5 (fp32)"}
    model.load_state_dict(keep)
    model.train()
    for p_ in model.parameters():
        p_.grad = None
    return out


def wsrglow_leg(dev, flush, cpu_baseline: bool):
    """Config 5 (WSRGlow 2x super-resolution, VCTK shape: 12 segments of 8192 samples, 4096-sample low-rate input,
    configs/wsrglow_vctk_2x.json): training step (forward + loss + reversible backward + Adam) and the inverse."""
    import constant_memory_waveglow_b200 as cm
    from constant_memory_waveglow_b200 import _lib, precision
    lib = _lib.load()
    torch.manual_seed(0)
    m = cm.WSRGlow(upsample_rate=2, memory_efficient=True, zero_init=False).to(dev).train()
    loss_fn = cm.WaveGlowLoss(1.0)
    opt = torch.optim.Adam(m.parameters(), lr=1e-4, fused=True)
    B = WSR_BATCH
    x = torch.rand(B, WSR_SEGMENT, device=dev) * 2 - 1
    c = torch.rand(B, WSR_SEGMENT // 2, device=dev) * 2 - 1

    def step():
        opt.zero_grad(set_to_none=True)
        z, logdet = m(x.clone(), c.clone())
        loss = loss_fn(z, logdet)
        loss.backward()
        opt.step()
        return z

    def timed(fn, n):
        tot = 0.0
        for _ in range(n):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        return tot / n

    for _ in range(3):
        z = step()
    lib.cmwg_reset_launch_count()
    ms_train = timed(step, 3)
    launches = int(lib.cmwg_launch_count()) // 3
    z = z.detach()
    m.eval()
    with torch.no_grad():
        for _ in range(2):
            m.reverse(z.clone(), c.clone())
        ms_inv = timed(lambda: m.reverse(z.clone(), c.clone()), 3)
    pk = peaks()
    tf_train = 4 * B * WSR_FWD_GFLOP_PER_SEGMENT / ms_train
    tf_inv = B * WSR_FWD_GFLOP_PER_SEGMENT / ms_inv
    out = {"config": {"workload": "wsrglow_2x_vctk (12 flows, n_group 16, 256 channels, 8 WN layers, 3659 conditioning rows)",
                      "batch": B, "segment": WSR_SEGMENT, "low_rate_samples": WSR_SEGMENT // 2},
           "operand_dtype": precision.resolve(True, True),
           "train_segments_per_s": B / (ms_train * 1e-3), "train_ms_per_step": ms_train, "gpu_launches_per_step": launches,
           "train_tflops": tf_train, "train_frac_of_peak": tf_train / pk["tflops_sustained"],
           "inverse_khz": B * WSR_SEGMENT / ms_inv, "inverse_ms": ms_inv, "inverse_tflops": tf_inv,
           "inverse_frac_of_peak": tf_inv / pk["tflops_sustained"],
           "flops": "234.978 GFLOP per 8192-sample segment forward (SURVEY 8d), training = 4x"}
    del m, opt
    torch.cuda.empty_cache()
    if cpu_baseline:
        r = reference_subprocess("wsrglow")
        if "train_segments_per_s" in r:
            out["cpu_baseline"] = {"train_segments_per_s": r["train_segments_per_s"], "inverse_khz": r["inverse_khz"],
                                   "cores": r["cores"], "kind": r["kind"],
                                   "sample": f"one 8192-sample segment: forward + loss + reversible backward "
                                             f"({r['train_seconds']:.1f} s) and the inverse ({r['inverse_seconds']:.1f} s)"}
            out["train_x_cpu"] = out["train_segments_per_s"] / r["train_segments_per_s"]
            out["inverse_x_cpu"] = out["inverse_khz"] / r["inverse_khz"]
        else:
            out["cpu_baseline"] = r
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="auto", choices=["bf16", "fp32", "fp16", "auto"],
                    help="auto = fp16 operands (TF32's mantissa) with fp32 accumulation, gradients scaled on the device")
    ap.add_argument("--ref-task", default="train", choices=["train", "synth", "parity", "wsrglow"],
                    help="--impl reference only: which bounded sample of the reference to time")
    ap.add_argument("--out", help="--ref-task parity only: the file the reference's outputs are written to")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/*.npy (see dump_outputs)")
    ap.add_argument("--no-graph", action="store_true", help="eager training step instead of one CUDA graph per step")
    ap.add_argument("--no-strong", action="store_true", help="skip the reference-semantics (24 // N per GPU) leg at N > 1")
    ap.add_argument("--no-wsrglow", action="store_true", help="skip the WSRGlow (config 5) leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity check against baseline/_ref")
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH)
    ap.add_argument("--synth-batch", type=int, default=4)
    ap.add_argument("--no-synth", action="store_true")
    ap.add_argument("--no-synth-sweep", action="store_true", help="skip the synthesis batch sweep (1, 4, 16, 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-waveflow", action="store_true", help="skip the WaveFlow (config 4) leg")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.ref_task == "parity" and not args.out:
        ap.error("--ref-task parity needs --out")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
