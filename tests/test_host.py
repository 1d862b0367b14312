"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares, the host
modules keep the reference's structure (state-dict keys, parameter order, channel schedule) and the
product path fails loudly without a GPU."""
import os
import re

import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import _lib, precision
from tests._util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "cmwg_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cmwg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    syms = declared_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(lib, s), s
        assert s in _lib.SIGNATURES, f"{s} declared in the header but not bound in _lib.SIGNATURES"
    for s in _lib.SIGNATURES:
        assert s in syms, f"{s} bound in _lib but not declared in include/cmwg_b200.h"
    assert lib.cmwg_version() >= 100
    assert lib.cmwg_launch_count() >= 0


def test_size_queries_need_no_gpu():
    import ctypes as C
    lib = _lib.load()
    cfg = _lib.WnConfig(4, 80, 256, 256, 256, 8, 3, 0, _lib.PREC_BF16)
    assert lib.cmwg_wn_tc_supported(C.byref(cfg)) == 1
    assert lib.cmwg_wn_aux_padded(C.byref(cfg)) == 128
    assert lib.cmwg_wn_packed_bytes(C.byref(cfg)) > 0
    assert lib.cmwg_wn_saved_bytes(C.byref(cfg), 2, 2000) > lib.cmwg_wn_saved_bytes(C.byref(cfg), 1, 2000)
    small = _lib.WnConfig(8, 20, 32, 32, 32, 2, 3, 0, _lib.PREC_FP32)
    assert lib.cmwg_wn_tc_supported(C.byref(small)) == 0
    assert lib.cmwg_wn_aux_padded(C.byref(small)) == 32
    bad = _lib.WnConfig(8, 20, 32, 32, 32, 2, 3, 0, _lib.PREC_BF16)  # tensor cores need multiples of 64
    assert lib.cmwg_wn_packed_bytes(C.byref(bad)) == 0
    assert b"multiples of 64" in lib.cmwg_last_error()


def test_state_dict_layout_matches_reference_fixture():
    fx = load_golden("waveglow_tiny.pt")
    m = cm.WaveGlow(memory_efficient=True, **fx["arch"], **fx["wn_kwargs"])
    sd = m.state_dict()
    assert list(sd.keys()) == list(fx["state"].keys())
    for k in sd:
        assert sd[k].shape == fx["state"][k].shape, k
    m.load_state_dict(fx["state"])
    assert m.z_split_sizes == [2, 6]
    fc = load_golden("coupling_a.pt")
    blk = cm.AffineCouplingBlock(cm.WN, True, **fc["kwargs"])
    assert [n for n, _ in blk.F.named_parameters()] == fc["param_order"]
    blk.load_state_dict(fc["state"])
    # remove_weight_norms collapses g/v pairs to .weight (inference.py:17)
    blk.apply(cm.remove_weight_norms)
    names = [n for n, _ in blk.F.named_parameters()]
    assert "V.weight" in names and not any(n.endswith("weight_g") for n in names)


def test_lj_channel_schedule():
    m = cm.WaveGlow(12, 8, 4, 2, 256, 80, True, dilation_channels=64, residual_channels=64, skip_channels=64, depth=1)
    assert [c.in_channels for c in m.invconv1x1] == [8] * 4 + [6] * 4 + [4] * 4
    assert m.z_split_sizes == [2, 2, 4]
    assert m.upsampler.weight_v.shape == (80, 1, 65) and m.upsampler.bias.shape == (80,)
    w = m.invconv1x1[0].weight.squeeze(-1)
    assert torch.det(w) > 0
    assert torch.allclose(w @ w.t(), torch.eye(8), atol=1e-5)


def test_product_path_fails_loudly_on_cpu():
    conv = cm.InvertibleConv1x1(4, True)
    with pytest.raises(RuntimeError, match="no CPU"):
        conv(torch.randn(1, 4, 16))
    blk = cm.AffineCouplingBlock(cm.WN, True, in_channels=2, aux_channels=4, dilation_channels=8,
                                 residual_channels=8, skip_channels=8, depth=1)
    with pytest.raises(RuntimeError, match="no CPU"):
        blk(torch.randn(1, 4, 16), torch.randn(1, 4, 16))
    with pytest.raises(RuntimeError, match="no CPU"):
        cm.WaveGlowLoss()(torch.randn(2, 8), torch.zeros(2))


def test_precision_resolution():
    old = precision.get_precision()
    flag = torch.backends.cudnn.allow_tf32
    try:
        precision.set_precision("auto")
        torch.backends.cudnn.allow_tf32 = False
        assert precision.resolve(True, False) == "fp32"
        torch.backends.cudnn.allow_tf32 = True
        assert precision.resolve(True, True) == "fp16"       # training: fp16 operands + device-side gradient scale
        assert precision.resolve(True, False) == "fp16"      # synthesis: TF32's mantissa at bf16's tensor-core rate
        assert precision.resolve(False, True) == "fp32"
        precision.set_precision("bf16")
        assert precision.resolve(True, True) == "bf16" and precision.resolve(True, False) == "bf16"   # opt-in only
        precision.set_precision("fp16")
        assert precision.resolve(True, False) == "fp16"
        assert precision.resolve(True, True) == "fp16"
        with pytest.raises(ValueError):
            precision.set_precision("int8")
    finally:
        precision.set_precision(old)
        torch.backends.cudnn.allow_tf32 = flag


def test_fused_optimizer_step_invalidates_weight_packs():
    """torch's fused optimizers update parameters without touching their version counters (checked here), so the weight-pack
    key carries a generation number that every optimizer step bumps."""
    from constant_memory_waveglow_b200 import waveglow as W
    p = torch.nn.Parameter(torch.randn(16))
    opt = torch.optim.Adam([p], lr=1e-3, fused=True)
    p.grad = torch.randn(16)
    g0, v0 = W.pack_generation(), p._version
    opt.step()
    assert W.pack_generation() > g0
    if p._version == v0:           # the behaviour that makes the generation number necessary
        assert True
    g1 = W.pack_generation()
    wn = cm.WN(2, 4, dilation_channels=8, residual_channels=8, skip_channels=8, depth=1)
    wn.load_state_dict(wn.state_dict())
    assert W.pack_generation() > g1
    g2 = W.pack_generation()
    cm.invalidate_packs()
    assert W.pack_generation() == g2 + 1


def test_every_native_switch_is_documented():
    """Every CMWG_* environment variable the native library reads (getenv, or engine_tc.cu's dbg_flag) is described in
    INTEGRATION.md, so a switch cannot be added without saying what it selects."""
    csrc = os.path.join(ROOT, "constant_memory_waveglow_b200", "csrc")
    names = set()
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh")):
            names |= set(re.findall(r'\b(?:getenv|dbg_flag)\("(CMWG_[A-Z0-9_]+)"\)', open(os.path.join(csrc, f)).read()))
    assert "CMWG_MEGA" in names and "CMWG_DEBUG_NOCACHE" in names
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    missing = sorted(n for n in names if not re.search(r"`" + n + r"\b", doc))
    assert not missing, f"switches read in csrc/ but not documented in INTEGRATION.md: {missing}"


def test_no_product_import_of_oracle():
    pkg = os.path.join(ROOT, "constant_memory_waveglow_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


@pytest.mark.parametrize("tag", ["a", "b"])
def test_waveflow_state_dict_layout_matches_reference_fixture(tag):
    fx = load_golden(f"waveflow_tiny_{tag}.pt")
    m = cm.WaveFlow(memory_efficient=False, **fx["arch"], **fx["wn_kwargs"])
    sd = m.state_dict()
    assert list(sd.keys()) == list(fx["state"].keys())
    for k in sd:
        assert sd[k].shape == fx["state"][k].shape, k
    m.load_state_dict(fx["state"])
    ref_order = list(fx["grads"].keys())
    assert [n for n, _ in m.named_parameters()] == ref_order
    with pytest.raises(RuntimeError, match="no CPU"):
        m(fx["x"], fx["h"])
    import model
    assert model.WaveFlow is cm.WaveFlow


def test_line_state_size_query():
    import ctypes as C
    lib = _lib.load()
    hd = (C.c_int * _lib.MAX_DEPTH)(1, 2, 4, 8, 16, 1, 2, 4)
    cfg = _lib.WnConfig(1, 80, 64, 64, 64, 8, 3, 0, _lib.PREC_BF16, 63, hd)
    n = lib.cmwg_wn_line_state_bytes(C.byref(cfg), 2, 100)
    assert n >= 8 * 2 * 63 * 100 * 64 * 2
    assert lib.cmwg_upsample_dense_workspace(80, 9) >= (80 * 80 * 9 + 80) * 4


# ---- task lists of the single-kernel WN forward / backward chain (csrc/engine_mega.cuh) --------------------------------
def _task_list(backward, depth, B, T):
    import ctypes as C
    lib = _lib.load()
    cap = 1 << 17
    out = (C.c_int * (4 * cap))()
    total, lag = C.c_int(0), C.c_int(0)
    assert lib.cmwg_mega_task_list(int(backward), depth, B, T, out, cap, C.byref(total), C.byref(lag)) == 0
    assert total.value <= cap
    rows = [tuple(out[4 * i:4 * i + 4]) for i in range(total.value)]
    return rows, lag.value


@pytest.mark.parametrize("depth,B,T", [(8, 24, 2000), (8, 1, 100), (8, 2, 300), (1, 2, 700), (3, 5, 2000), (8, 4, 27584),
                                       (2, 1, 513), (8, 3, 256)])
def test_task_lists_are_in_dependency_order(depth, B, T):
    """The kernels' own decode functions, run on the host: every task appears exactly once and AFTER everything it waits
    for -- the property that makes `pair p runs entries p, p + P, ...` deadlock free (the lowest unfinished entry is always
    runnable) -- for one row tile, ragged tiles, a single layer, the LJ training shape and a 10 s utterance."""
    tpb = -(-T // 256)
    RT = B * tpb

    def neighbours(rt):
        b, tb = divmod(rt, tpb)
        return [b * tpb + t for t in (tb - 1, tb, tb + 1) if 0 <= t < tpb]

    # forward: 0 gate G(layer, rt, nt), 1 residual R(layer, rt), 2 skip S(rt)
    rows, lag = _task_list(False, depth, B, T)
    assert 0 <= lag <= max(0, RT - 2)
    pos = {}
    for i, (typ, layer, rt, nt) in enumerate(rows):
        if typ == 3:
            continue
        key = (typ, layer, rt, nt) if typ == 0 else (typ, layer if typ == 1 else 0, rt, 0)
        assert key not in pos, key
        pos[key] = i
    assert sum(1 for k in pos if k[0] == 0) == depth * RT * 2
    assert sum(1 for k in pos if k[0] == 1) == (depth - 1) * RT
    assert sum(1 for k in pos if k[0] == 2) == RT
    dist = []
    for (typ, layer, rt, nt), i in pos.items():
        if typ == 0 and layer > 0:
            deps = [(1, layer - 1, r, 0) for r in neighbours(rt)]
        elif typ == 1:
            deps = [(0, layer, rt, n) for n in (0, 1)]
        elif typ == 2:
            deps = [(0, depth - 1, rt, n) for n in (0, 1)]
        else:
            deps = []
        for d in deps:
            assert d in pos and pos[d] < i, ((typ, layer, rt, nt), d)
            dist.append(i - pos[d])
    if (depth, B, T) == (8, 24, 2000):
        assert lag == 64 and min(dist) >= 190      # 2.6 rounds of 74 pairs between a task and what it waits for

    # backward chain: 0 dgate DG(layer, rt), 1 dx DX(layer, rt)
    rows, lag = _task_list(True, depth, B, T)
    assert 0 <= lag <= max(0, RT - 2)
    pos = {}
    for i, (typ, layer, rt, _) in enumerate(rows):
        if typ == 3:
            continue
        assert (typ, layer, rt) not in pos
        pos[(typ, layer, rt)] = i
    assert len(pos) == 2 * depth * RT
    for (typ, layer, rt), i in pos.items():
        if typ == 0:
            deps = [(1, layer + 1, rt)] if layer < depth - 1 else []
        else:
            deps = [(0, layer, r) for r in neighbours(rt)]
        for d in deps:
            assert d in pos and pos[d] < i, ((typ, layer, rt), d)


# ---- split-K plan of the batched weight-gradient launch (csrc/engine_tc.cu: wgrad_group_splits) -------------------------
def test_weight_gradient_split_plan_minimises_rounds_times_k():
    """74 CTA pairs take ceil(tiles * s / 74) rounds of ceil(units / s) k-blocks.  The LJ training shape has 24 x 32 = 768
    time units; 49 tiles (the batched launch with both folds) are ONE round of the full K with s = 1 and two rounds of a
    third with s = 3; 63 tiles (no folds) gain too little from any split to pay for its partial tiles at s <= 6."""
    lib = _lib.load()
    units = 24 * 32

    def rounds_times_k(tiles, s):
        return -(-tiles * s // 74) * -(-units // s)

    s49 = lib.cmwg_wgrad_plan_splits(49, 256, 24, 2000)
    assert s49 == 3 and rounds_times_k(49, s49) * 3 <= rounds_times_k(49, 1) * 2 + 3
    for tiles in (1, 8, 24, 37, 49, 57, 63, 74, 100):
        s = lib.cmwg_wgrad_plan_splits(tiles, 256, 24, 2000)
        assert 1 <= s <= 80
        assert rounds_times_k(tiles, s) <= rounds_times_k(tiles, 1)          # never worse than no split
    assert lib.cmwg_wgrad_plan_splits(24, 128, 24, 2000) == 3                 # the N = 128 group: one round of a third of K
    assert lib.cmwg_wgrad_plan_splits(2, 256, 1, 64) == 1                     # a single time unit cannot be split
    assert lib.cmwg_wgrad_plan_splits(0, 256, 1, 64) == -1 and lib.cmwg_wgrad_plan_splits(4, 64, 1, 64) == -1
