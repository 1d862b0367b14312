"""Host side of variable-length batched inference (no device needed): the compacted task list of the single-kernel WN
forward (cmwg_mega_task_list_varlen, the kernel's own decode function run on the host) and the argument checks of the
Python API."""
import ctypes as C

import pytest
import torch

import constant_memory_waveglow_b200 as cm
from constant_memory_waveglow_b200 import _lib
from constant_memory_waveglow_b200.base import pad_batch


def _varlen_list(depth, T, lengths):
    lib = _lib.load()
    B = len(lengths)
    cap = 1 << 17
    out = (C.c_int * (4 * cap))()
    tcap = B * -(-T // 256)
    tiles = (C.c_int * (3 * tcap))()
    total, lag, rts = C.c_int(0), C.c_int(0), C.c_int(0)
    rc = lib.cmwg_mega_task_list_varlen(depth, B, T, (C.c_int * B)(*lengths), out, cap, C.byref(total), C.byref(lag),
                                        tiles, tcap, C.byref(rts))
    assert rc == 0
    assert total.value <= cap
    rows = [tuple(out[4 * i:4 * i + 4]) for i in range(total.value)]
    tab = [tuple(tiles[3 * r:3 * r + 3]) for r in range(rts.value)]
    return rows, lag.value, tab


def _dense_list(depth, B, T):
    lib = _lib.load()
    cap = 1 << 17
    out = (C.c_int * (4 * cap))()
    total, lag = C.c_int(0), C.c_int(0)
    assert lib.cmwg_mega_task_list(0, depth, B, T, out, cap, C.byref(total), C.byref(lag)) == 0
    return [tuple(out[4 * i:4 * i + 4]) for i in range(total.value)], lag.value


CASES = [
    (8, 2000, [2000] * 3),                   # every item full length: the dense list
    (8, 27584, [27584, 300, 257, 100, 1]),   # one long item and many short ones
    (8, 2000, [200, 1, 255, 17]),            # every item shorter than one row tile
    (8, 2048, [512, 256, 2048, 768]),        # exact multiples of the 256-row tile
    (3, 700, [700, 1]),
    (1, 300, [300, 12]),
]


@pytest.mark.parametrize("depth,T,lengths", CASES)
def test_varlen_task_lists_are_in_dependency_order(depth, T, lengths):
    rows, lag, tab = _varlen_list(depth, T, lengths)
    RT = sum(-(-n // 256) for n in lengths)
    assert len(tab) == RT
    assert 0 <= lag <= max(0, RT - 2)
    # the table: item order, consecutive tiles per item, tile counts of the items
    assert [t[0] for t in tab] == sorted(t[0] for t in tab)
    for b, n in enumerate(lengths):
        mine = [t for t in tab if t[0] == b]
        assert [t[1] for t in mine] == list(range(-(-n // 256))) and all(t[2] == -(-n // 256) for t in mine)

    def neighbours(rt):
        b, tb, ntb = tab[rt]
        return [rt + d for d in (-1, 0, 1) if 0 <= tb + d < ntb]   # within the item only

    pos = {}
    for i, (typ, layer, rt, nt) in enumerate(rows):
        if typ == 3:
            continue
        key = (typ, layer, rt, nt) if typ == 0 else (typ, layer if typ == 1 else 0, rt, 0)
        assert key not in pos, key
        assert 0 <= rt < RT
        pos[key] = i
    assert sum(1 for k in pos if k[0] == 0) == depth * RT * 2
    assert sum(1 for k in pos if k[0] == 1) == (depth - 1) * RT
    assert sum(1 for k in pos if k[0] == 2) == RT
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
    if all(n == T for n in lengths):
        assert (rows, lag) == _dense_list(depth, len(lengths), T)


def test_varlen_task_list_rejects_bad_lengths():
    lib = _lib.load()
    out = (C.c_int * 64)()
    tiles = (C.c_int * 64)()
    a, b, c = C.c_int(0), C.c_int(0), C.c_int(0)
    for bad in ([0, 10], [10, 301]):
        assert lib.cmwg_mega_task_list_varlen(8, 2, 300, (C.c_int * 2)(*bad), out, 16, C.byref(a), C.byref(b), tiles, 16,
                                              C.byref(c)) == -1
        assert b"outside" in lib.cmwg_last_error()


def _small_waveglow(**kw):
    return cm.WaveGlow(4, 8, 2, 2, 256, 80, True, dilation_channels=64, residual_channels=64, skip_channels=64, depth=1,
                       **kw)


@pytest.mark.parametrize("lengths,exc,match", [
    ([1024, 12], ValueError, "multiple of n_group"),        # not a multiple of n_group
    ([1024, 2048], ValueError, r"in \[1, 1024\]"),           # longer than the batch
    ([1024, 0], ValueError, r"in \[1, 1024\]"),
    ([4, 2], ValueError, "multiple of n_group"),            # mel frames passed where samples are expected
    ([1024], ValueError, "1 lengths for a batch of 2"),
    ([1024.0, 512.0], TypeError, "integers"),
    (torch.tensor([1024.0, 512.0]), TypeError, "integer tensor"),
])
def test_model_lengths_validation(lengths, exc, match):
    m = _small_waveglow()
    x, h = torch.zeros(2, 1024), torch.zeros(2, 80, 4)
    with torch.no_grad(), pytest.raises(exc, match=match):
        m(x, h, lengths=lengths)
    with torch.no_grad(), pytest.raises(exc, match=match):
        m.reverse(x, h, lengths=lengths)


def test_model_lengths_need_inference_mode():
    m = _small_waveglow()
    x, h = torch.zeros(2, 1024), torch.zeros(2, 80, 4)
    with pytest.raises(NotImplementedError, match="inference only"):
        m(x, h, lengths=[1024, 512])
    with pytest.raises(NotImplementedError, match="inference only"):
        m.reverse(x, h, lengths=torch.tensor([1024, 512]))
    m2 = _small_waveglow(reverse_mode=True)     # direction dispatch: forward() runs the synthesis direction
    with pytest.raises(NotImplementedError, match="inference only"):
        m2(x, h, lengths=[1024, 512])


def test_infer_lengths_are_frames():
    m = _small_waveglow()
    h = torch.zeros(2, 80, 4)
    with pytest.raises(ValueError, match="mel frames"):
        m.infer(h, 0.5, lengths=[4, 5])
    with pytest.raises(ValueError, match="mel frames"):
        m.infer(h, 0.5, lengths=[4, 0])


def test_other_families_reject_lengths():
    x, h = torch.zeros(1, 1024), torch.zeros(1, 80, 4)
    wsr = cm.WSRGlow(upsample_rate=2, memory_efficient=True, dilation_channels=64, residual_channels=64, skip_channels=64,
                     depth=1)
    for m in (wsr,):
        with torch.no_grad(), pytest.raises(NotImplementedError, match="WaveGlow only"):
            m(x, h, lengths=[1024])
        with torch.no_grad(), pytest.raises(NotImplementedError, match="WaveGlow only"):
            m.reverse(x, h, lengths=[1024])
        with pytest.raises(NotImplementedError, match="WaveGlow only"):
            m.infer(h, 0.5, lengths=[4])
    for cls in (cm.MRWaveGlow, cm.WaveFlow, cm.MelGlow):
        assert cls._supports_lengths is False
        assert cls.forward is cm.FlowBase.forward and cls.reverse is cm.FlowBase.reverse


def test_pad_batch():
    mels = [torch.ones(80, 3), torch.full((80, 5), 2.0), torch.full((80, 1), 3.0)]
    h, frames = pad_batch(mels)
    assert frames == [3, 5, 1] and h.shape == (3, 80, 5)
    assert torch.equal(h[0, :, :3], mels[0]) and (h[0, :, 3:] == 0).all() and (h[2, :, 1:] == 0).all()
    w, n = pad_batch([torch.ones(7), torch.ones(2)])
    assert n == [7, 2] and w.shape == (2, 7) and w[1, 2:].abs().sum() == 0
    with pytest.raises(ValueError):
        pad_batch([torch.ones(80, 3), torch.ones(40, 3)])
