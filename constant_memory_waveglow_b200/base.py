"""Direction dispatch and the flow-model contract: the surface of the reference's ``model/base.py``
(``Reversible`` :7-28, ``FlowBase`` :31-55) -- same names, methods and argument meaning.

A ``Reversible`` owns two computations, one the inverse of the other; ``reverse_mode=True`` swaps which of them ``forward()``
runs, so that a flow can be trained in the synthesis direction.  ``FlowBase`` adds the model contract
``forward(x, h) -> (z, logdet)``, ``reverse(z, h) -> (x, logdet)`` and ``infer(h, sigma) -> audio``.
"""
from typing import Callable, List, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor, nn

FlowOut = Tuple[Tensor, Tensor]


class Reversible(nn.Module):
    _reverse_mode: bool

    def __init__(self, reverse_mode, **kwargs) -> None:
        super().__init__(**kwargs)
        self._reverse_mode = reverse_mode

    # the two directions a subclass provides
    def forward_computation(self, x: Tensor, *args, **kwargs) -> FlowOut:
        raise NotImplementedError(f"{type(self).__name__} defines no forward computation")

    def reverse_computation(self, z: Tensor, *args, **kwargs) -> FlowOut:
        raise NotImplementedError(f"{type(self).__name__} defines no reverse computation")

    def _direction(self, inverse: bool) -> Callable[..., FlowOut]:
        """The computation that realises the requested direction under this module's mode (XOR of the two switches)."""
        return self.reverse_computation if inverse != bool(self._reverse_mode) else self.forward_computation

    def forward(self, x: Tensor, *args, **kwargs) -> FlowOut:
        return self._direction(False)(x, *args, **kwargs)

    def reverse(self, z: Tensor, *args, **kwargs) -> FlowOut:
        return self._direction(True)(z, *args, **kwargs)


Lengths = Union[Sequence[int], Tensor]


def pad_batch(items: Sequence[Tensor]) -> Tuple[Tensor, List[int]]:
    """Stack tensors that differ only in their last dimension -- mel spectrograms (n_mels, frames) or waveforms (samples,)
    -- into one zero-padded batch (B, ..., max_len).  Returns (batch, lengths), lengths in the unit of that last dimension:
    mel frames for ``infer(h, lengths=...)``, samples for ``forward`` / ``reverse``."""
    if len(items) == 0:
        raise ValueError("pad_batch: no items")
    lead = tuple(items[0].shape[:-1])
    for t in items:
        if tuple(t.shape[:-1]) != lead:
            raise ValueError(f"pad_batch: items differ in more than their last dimension: {tuple(t.shape)} vs {lead + (-1,)}")
    lengths = [int(t.shape[-1]) for t in items]
    out = items[0].new_zeros((len(items),) + lead + (max(lengths),))
    for i, t in enumerate(items):
        out[i, ..., :lengths[i]] = t
    return out, lengths


class FlowBase(Reversible):
    # forward / reverse / infer accept per-item `lengths` (inference on a padded batch).  Only WaveGlow implements them.
    _supports_lengths = False

    def __init__(self, condition_hop_length: int, reverse_mode=False) -> None:
        super().__init__(reverse_mode=reverse_mode)
        self._hop_length = condition_hop_length

    def _require_lengths(self) -> None:
        if not self._supports_lengths:
            raise NotImplementedError(f"{type(self).__name__}: per-item `lengths` are implemented for WaveGlow only; "
                                      "call this model once per utterance instead")

    def forward(self, x: Tensor, *args, lengths: Optional[Lengths] = None, **kwargs) -> FlowOut:
        if lengths is None:
            return super().forward(x, *args, **kwargs)
        self._require_lengths()
        return super().forward(x, *args, lengths=lengths, **kwargs)

    def reverse(self, z: Tensor, *args, lengths: Optional[Lengths] = None, **kwargs) -> FlowOut:
        if lengths is None:
            return super().reverse(z, *args, **kwargs)
        self._require_lengths()
        return super().reverse(z, *args, lengths=lengths, **kwargs)

    def forward_computation(self, x: Tensor, h: Tensor) -> FlowOut:
        raise NotImplementedError(f"{type(self).__name__} defines no forward computation")

    def reverse_computation(self, z: Tensor, h: Tensor) -> FlowOut:
        raise NotImplementedError(f"{type(self).__name__} defines no reverse computation")

    @torch.no_grad()
    def infer(self, h: Tensor, sigma: float = 1., z: Optional[Tensor] = None, lengths: Optional[Lengths] = None) -> Tensor:
        """Synthesis (``model/base.py:42-55``): z ~ N(0, sigma^2) with ``frames * hop`` samples per item, pushed through the
        direction that maps noise to audio.  ``z`` may be supplied (already scaled) so that parity tests feed the oracle and
        this path identical noise.

        ``lengths``: valid MEL FRAMES per item of a zero-padded batch ``h`` (B, n_mels, F_max) (see ``pad_batch``).  Item b
        is then synthesised from its first ``lengths[b]`` frames exactly as a call on that item alone, and the result is
        (B, F_max * hop) with zeros after ``lengths[b] * hop`` samples."""
        cond = h if h.dim() == 3 else h.unsqueeze(0)
        if lengths is not None:
            self._require_lengths()
            frames = lengths_list(lengths, cond.shape[0], "infer", "mel frames")
            for f in frames:
                if not 1 <= f <= cond.shape[2]:
                    raise ValueError(f"infer: frame length {f} outside [1, {cond.shape[2]}] (lengths are in mel frames)")
            if z is None:
                z = cond.new_empty((cond.shape[0], cond.shape[2] * self._hop_length)).normal_(std=sigma)
            audio, _ = self._direction(True)(z, cond, lengths=[f * self._hop_length for f in frames])
            return audio
        if z is None:
            n_items, frames = cond.shape[0], cond.shape[2]
            z = cond.new_empty((n_items, frames * self._hop_length)).normal_(std=sigma)
        audio, _ = self._direction(True)(z, cond)
        return audio.squeeze()


def lengths_list(lengths: Lengths, batch: int, what: str, unit: str) -> List[int]:
    """`lengths` (a sequence of ints or a CPU integer tensor, one per batch item) as a list of Python ints."""
    if isinstance(lengths, Tensor):
        if lengths.is_cuda or lengths.is_floating_point() or lengths.is_complex() or lengths.dim() != 1:
            raise TypeError(f"{what}: lengths must be a 1-D CPU integer tensor or a sequence of ints ({unit})")
        lengths = lengths.tolist()
    out = []
    for v in lengths:
        if isinstance(v, bool) or not isinstance(v, int):
            if isinstance(v, Tensor) and v.dim() == 0 and not v.is_floating_point():
                v = int(v)
            else:
                raise TypeError(f"{what}: lengths must be integers ({unit}), got {v!r}")
        out.append(int(v))
    if len(out) != batch:
        raise ValueError(f"{what}: {len(out)} lengths for a batch of {batch}")
    return out
