"""The conv weight packs: how each conv's weight is laid out for the conv kernels, and one cache of them per model.

The conv kernels read packs, not the fp32 OIHW parameters: `wf` [Cout,3,3,Cin] for the forward, `wd` [Cin,3,3,Cout]
for the data gradient and, for a stride-2 conv with Cin in {32, 64}, `ws`, the parity-stacked data-gradient pack of
`ops.conv_dgrad_s2` (made from `wd`).  A `Layout` says how the weight sits in them; its kind is one of

    stem  the first conv's <= 8 input channels zero-padded to 32 (the tensor-core stem reads 64 B per pixel)
    conv  a plain 3x3 pack
    k1    a 1x1 weight as the centre tap of a zero 3x3 kernel (the CLIP fusion conv), over its first `cin` inputs
    head  a 3x3 head with its output channels zero-padded: to 32 for the bf16 tensor-core kernels, to 8 for fp32

`PackStore` (`model._packs`) caches them and holds the packs that FusedSGD / FusedAdam(model=) write in their step.
"""
from __future__ import annotations

from typing import Dict, NamedTuple, Optional, Tuple

import torch
import torch.nn as nn

from . import ops

BF16 = torch.bfloat16


class Layout(NamedTuple):
    kind: str
    cout: int
    cin: int  # input channels read from the weight
    cout_pad: int
    cin_pad: int
    ksize: int  # 1: the weight is the centre tap
    dtype: torch.dtype


def layout(conv: nn.Conv2d, kind: str, dtype=BF16, cin_used: Optional[int] = None) -> Layout:
    cout = conv.out_channels
    cin = conv.in_channels if cin_used is None else cin_used
    cout_pad = (32 if dtype == BF16 else 8) if kind == "head" else cout
    cin_pad = 32 if kind == "stem" else cin
    return Layout(kind, cout, cin, cout_pad, cin_pad, 1 if kind == "k1" else 3, dtype)


def build(w: torch.Tensor, lay: Layout, need_dgrad: bool):
    """(wf, wd) of weight w in layout lay; wd is None unless need_dgrad."""
    w = w.detach()
    if lay.ksize == 1 or lay.cout_pad != lay.cout or lay.cin_pad != lay.cin:
        wp = torch.zeros((lay.cout_pad, lay.cin_pad, 3, 3), dtype=torch.float32, device=w.device)
        if lay.ksize == 1:
            wp[:lay.cout, :lay.cin, 1, 1] = w[:, :lay.cin, 0, 0]
        else:
            wp[:lay.cout, :lay.cin] = w
        w = wp
    return ops.pack_conv_weights(w, need_dgrad=need_dgrad, dtype=lay.dtype)


class Pack:
    """The packs of one weight in one layout, and the state of the weight they hold."""
    __slots__ = ("layout", "wf", "wd", "ws", "version", "ptr")

    def __init__(self, lay: Layout, w: torch.Tensor, wf, wd, ws=None):
        self.layout, self.wf, self.wd, self.ws = lay, wf, wd, ws
        self.stamp(w)

    def stamp(self, w: torch.Tensor) -> None:
        self.version, self.ptr = w._version, w.data_ptr()

    def valid(self, w: torch.Tensor, need_dgrad: bool) -> bool:
        return self.version == w._version and self.ptr == w.data_ptr() and self.wf.device == w.device \
            and (self.wd is not None or not need_dgrad)


class PackStore:
    def __init__(self):
        self.cache: Dict[Tuple[int, Layout], Pack] = {}
        self.emitted: Dict[int, Pack] = {}  # id(weight) -> the packs a flat optimizer step writes
        self._s2: Dict[int, Tuple[torch.Tensor, Optional[torch.Tensor]]] = {}  # id(weight) -> (wd, ws made from it)

    def get(self, conv: nn.Conv2d, kind: str, dtype, need_dgrad: bool, cin_used: Optional[int] = None):
        """(wf, wd) of conv's weight in layout(conv, kind, dtype, cin_used): the emitted packs if they have exactly
        that layout and are current, else a cached pack, rebuilt when the weight has changed."""
        w = conv.weight
        lay = layout(conv, kind, dtype, cin_used)
        p = self.emitted.get(id(w))
        if p is None or p.layout != lay or not p.valid(w, need_dgrad):
            p = self.cache.get((id(w), lay))
            if p is None or not p.valid(w, need_dgrad):
                p = self.cache[(id(w), lay)] = Pack(lay, w, *build(w, lay, need_dgrad))
        return p.wf, p.wd

    def s2(self, conv: nn.Conv2d, wd: torch.Tensor) -> Optional[torch.Tensor]:
        """The stride-2 pack made from wd (a dgrad pack get() returned for conv), or None where there is none."""
        p = self.emitted.get(id(conv.weight))
        if p is not None and p.wd is wd:
            return p.ws
        hit = self._s2.get(id(conv.weight))
        if hit is None or hit[0] is not wd:
            hit = self._s2[id(conv.weight)] = (wd, ops.pack_s2_dgrad_weights(wd))
        return hit[1]

    def emit(self, conv: nn.Conv2d, kind: str) -> Pack:
        """The bf16 packs of conv that a flat optimizer step writes, made from the current weight on first use.  They
        are never reallocated: the step's descriptor table and captured CUDA graphs hold their addresses."""
        p = self.emitted.get(id(conv.weight))
        if p is None:
            w, lay = conv.weight, layout(conv, kind)
            wf, wd = build(w, lay, need_dgrad=kind != "stem")  # the stem's data gradient is never computed
            ws = ops.pack_s2_dgrad_weights(wd) if conv.stride[0] == 2 else None
            p = self.emitted[id(w)] = Pack(lay, w, wf, wd, ws)
        return p

    def stamp(self, params) -> None:
        """A flat step has written the emitted packs of these parameters from their current values."""
        for w in params:
            p = self.emitted.get(id(w))
            if p is not None:
                p.stamp(w)
