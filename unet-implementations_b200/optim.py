"""Fused optimizer step for the reference's trainer: `torch.optim.SGD(lr, momentum, nesterov=True, weight_decay)`
(Our_UNet/src/train.py:431-451, stepped at :650 / :664) -- SURVEY.md section 8f, row 1.

`FusedSGD` is a `torch.optim.Optimizer`: `param_groups[i]["lr"]` is what `LambdaLR` (train.py:454-477) drives, the
per-parameter state is `momentum_buffer` as in torch, so `state_dict()` is interchangeable with `torch.optim.SGD`.
The arithmetic mirrors torch's foreach implementation on CUDA operation by operation (bit-exact, tests/test_gpu_aux.py).

Two modes:

* `FusedSGD(model.parameters(), ...)` -- one multi-tensor launch over the parameters where they are
  (b200unet_sgd_nesterov_step).  The parameters' version counters are bumped after the launch, so the bf16 operand
  packs `UNet` caches per weight version are rebuilt on the next forward.
* `FusedSGD(model.parameters(), ..., model=model)` -- the flat form: the parameters are re-pointed into ONE flat
  fp32 master buffer laid out like the model's flat gradient buffer (flat.FlatGradSink; the data-parallel reducer of
  ddp.py IS such a sink, so the step runs straight on the all-reduced buffer), momentum lives in a third buffer at the
  same offsets, and ONE launch (b200unet_sgd_flat_step) scales the gradient, updates master + momentum and EMITS
  the bf16 [Cout,3,3,Cin] / [Cin,3,3,Cout] / stride-2 packs the conv kernels read, which `UNet` then uses directly:
  no repack kernels between the optimizer and the next forward, and packs that cannot go stale.

`FusedAdam(model.parameters(), ..., model=model)` is the autoencoder trainer's `torch.optim.Adam`
(AE_pretrained/reconstruction/src/train.py:390-394; AdamW with `decoupled_weight_decay=True`) in the same flat form:
exp_avg / exp_avg_sq at the flat offsets, the per-parameter step counts in device memory, ONE prologue + ONE flat launch
(b200unet_adam_flat_step) that emits the packs like FusedSGD's.  Bit-identical to torch.optim.Adam on CUDA
(tests/test_gpu_adam.py), and its state_dict() has torch.optim.Adam's layout, so either optimizer resumes the other.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import _lib
from .flat import FlatGradSink, sink_of

BF16 = torch.bfloat16


def _bump_versions(params) -> None:
    """The kernels write parameters through raw pointers, which autograd cannot see: bump the version counters so that
    everything keyed on `Tensor._version` (UNet's pack cache, saved-tensor checks) notices the update."""
    torch.autograd.graph.increment_version(list(params))


def _sync_lr(opt, dtype) -> None:
    """The device copy of param_groups[0]["lr"] that a capturable flat optimizer's kernel reads (`opt._lr_dev`)."""
    if not opt.capturable or opt._flat is None:
        return
    dev = opt._flat.master.device
    if opt._lr_dev is None:
        opt._lr_dev = torch.zeros(1, dtype=dtype, device=dev)
        opt._lr_host = torch.zeros(1, dtype=dtype).pin_memory()
        opt._lr_last = None
    lr = float(opt.param_groups[0]["lr"])
    if lr != opt._lr_last:
        torch.cuda.current_stream().synchronize()  # the pinned scalar may still be in flight from the last change
        opt._lr_host[0] = lr
        opt._lr_dev.copy_(opt._lr_host, non_blocking=True)
        opt._lr_last = lr


class FusedSGD(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, momentum=0.0, dampening=0.0, weight_decay=0.0, nesterov=False, model=None,
                 grad_scale: float = 1.0, capturable: bool = False):
        if dampening != 0.0:
            raise ValueError("FusedSGD: dampening is not supported (the trainer uses 0)")
        if nesterov and momentum <= 0:
            raise ValueError("Nesterov momentum requires a momentum")
        super().__init__(params, dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay,
                                      nesterov=nesterov))
        self.grad_scale = float(grad_scale)  # multiplies every gradient inside the flat step (e.g. 1 / loss scale)
        # capturable (flat mode): the learning rate is read from a device scalar, so that `step()` can sit inside a CUDA
        # graph (graph.GraphedStep(..., optimizer=opt)); `sync_lr()` copies param_groups[0]["lr"] there before a replay
        self.capturable = bool(capturable)
        self._lr_dev: Optional[torch.Tensor] = None
        self._lr_host: Optional[torch.Tensor] = None
        self._flat: Optional[_FlatState] = None
        if model is not None:
            if len(self.param_groups) != 1:
                raise ValueError("FusedSGD(model=...): the flat step supports one parameter group (the trainer has one)")
            self._flat = _FlatState(model, self.param_groups[0]["params"], "FusedSGD")

    # ------------------------------------------------------------------------------------------------ step
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self._flat is not None:
            self._flat_step()
            return loss
        for group in self.param_groups:
            ps = [p for p in group["params"] if p.grad is not None]
            if not ps:
                continue
            mom = float(group["momentum"])
            # parameters seen for the first time get buf = g (torch: clone of the decayed gradient); they go in their own launch
            if mom != 0:
                batches = [(True, [p for p in ps if "momentum_buffer" not in self.state[p]]),
                           (False, [p for p in ps if "momentum_buffer" in self.state[p]])]
            else:
                batches = [(True, ps)]
            for first, sel in batches:
                if not sel:
                    continue
                for p in sel:
                    if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and p.grad.is_contiguous()
                            and p.grad.dtype == torch.float32 and not p.grad.is_sparse):
                        raise RuntimeError("FusedSGD: parameters and gradients must be contiguous fp32 CUDA tensors")
                    if mom != 0 and first:
                        self.state[p]["momentum_buffer"] = torch.empty_like(p)
                n = len(sel)
                PT = ctypes.c_void_p * n
                params = PT(*[p.data_ptr() for p in sel])
                grads = PT(*[p.grad.data_ptr() for p in sel])
                bufs = PT(*[self.state[p]["momentum_buffer"].data_ptr() for p in sel]) if mom != 0 else None
                numels = (ctypes.c_int64 * n)(*[p.numel() for p in sel])
                with torch.cuda.device(sel[0].device):
                    _lib.call("b200unet_sgd_nesterov_step", params, grads, bufs, numels, n, float(group["lr"]), mom,
                              float(group["weight_decay"]), int(bool(group["nesterov"])), int(first and mom != 0),
                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                _bump_versions(sel)
        return loss

    def sync_lr(self):
        """capturable mode: copy the current learning rate (what LambdaLR wrote into param_groups) to the device scalar
        the captured optimizer kernel reads.  Called by step() when eager, and by GraphedStep.replay() before a replay."""
        _sync_lr(self, torch.float32)

    def _flat_step(self):
        group = self.param_groups[0]
        fs = self._flat
        mom = float(group["momentum"])
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            fs.sync(self.state, mom != 0)
            self.sync_lr()
        elif not self.capturable or self._lr_dev is None or any(f < 0 or (f & 2) for f in fs.flags):
            raise RuntimeError("FusedSGD: capture step() with capturable=True and after two eager steps (the first one "
                               "initialises the momentum buffers, the second uploads the steady-state tensor table)")
        with torch.cuda.device(fs.master.device):
            _lib.call("b200unet_sgd_flat_step", ctypes.c_void_p(fs.table_dev.data_ptr()), fs.count, fs.total_blocks,
                      ctypes.c_void_p(fs.master.data_ptr()), ctypes.c_void_p(fs.sink.flat.data_ptr()),
                      ctypes.c_void_p(fs.bufs["momentum_buffer"].data_ptr()) if mom != 0 else None, float(group["lr"]), mom,
                      float(group["weight_decay"]), int(bool(group["nesterov"])), float(self.grad_scale),
                      ctypes.c_void_p(self._lr_dev.data_ptr()) if self._lr_dev is not None else None,
                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        if not capturing:
            fs.after_step(self.state, mom != 0)


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam (AdamW with decoupled_weight_decay=True) as one flat step over the model's buffers.

    Only the flat form exists: `model=` is required and the parameters become views of one fp32 master buffer, exactly
    as with FusedSGD(model=...).  Each step is two launches (b200unet_adam_flat_step): a one-block prologue that
    advances the step counts and forms torch's bias corrections in double, and the flat kernel that updates
    parameters, exp_avg and exp_avg_sq and emits the bf16 conv weight packs.  The result is bit-identical to
    torch.optim.Adam (foreach, CUDA) for grad_scale 1, and state_dict() / load_state_dict() interchange with it.

    grad_scale multiplies every gradient inside the step (the 1 / world size of ddp.BucketedGradAllReduce).
    capturable: the learning rate is read from a float64 device scalar, so that step() can sit inside a CUDA graph
    (graph.GraphedStep(..., optimizer=opt) refreshes it before each replay); betas, eps and weight_decay are fixed at
    capture.  Not implemented (ValueError): amsgrad, maximize, differentiable, fused, more than one parameter group.
    """

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, *,
                 decoupled_weight_decay: bool = False, model=None, grad_scale: float = 1.0, capturable: bool = False,
                 amsgrad: bool = False, maximize: bool = False, foreach=None, differentiable: bool = False, fused=None):
        for name, on in (("amsgrad", amsgrad), ("maximize", maximize), ("differentiable", differentiable),
                         ("fused", fused)):
            if on:
                raise ValueError(f"FusedAdam: {name}=True is not implemented")
        if model is None:
            raise ValueError("FusedAdam needs model=...: it steps the model's flat parameter and gradient buffers")
        if not 0.0 <= float(lr):
            raise ValueError(f"Invalid learning rate: {lr}")
        if not 0.0 <= float(eps):
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not (0.0 <= float(betas[0]) < 1.0 and 0.0 <= float(betas[1]) < 1.0):
            raise ValueError(f"Invalid beta parameters: {betas}")
        if not 0.0 <= float(weight_decay):
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        # the group has torch.optim.Adam's keys, so that a state_dict of either optimizer loads into the other
        # ("capturable" is left out: it means device-side step counts and different arithmetic to torch)
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, amsgrad=False,
                                      maximize=False, foreach=foreach, differentiable=False, fused=None,
                                      decoupled_weight_decay=bool(decoupled_weight_decay)))
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdam: the flat step supports one parameter group")
        self.grad_scale = float(grad_scale)
        self.capturable = bool(capturable)
        self._lr_dev: Optional[torch.Tensor] = None
        self._lr_host: Optional[torch.Tensor] = None
        self._flat = _FlatState(model, self.param_groups[0]["params"], "FusedAdam", buffers=("exp_avg", "exp_avg_sq"),
                                step_counters=True)
        self._scalars = torch.empty(4 * self._flat.count, dtype=torch.float32, device=self._flat.master.device)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        group = self.param_groups[0]
        for name in ("amsgrad", "maximize", "differentiable", "fused"):  # a loaded state_dict may ask for them
            if group.get(name):
                raise ValueError(f"FusedAdam: {name}=True is not implemented")
        fs = self._flat
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            fs.sync(self.state, True)
            self.sync_lr()
        elif not self.capturable or self._lr_dev is None or any(f < 0 for f in fs.flags):
            raise RuntimeError("FusedAdam: capture step() with capturable=True and after one eager step (it creates the "
                               "optimizer state and uploads the tensor table)")
        beta1, beta2 = group["betas"]
        with torch.cuda.device(fs.master.device):
            _lib.call("b200unet_adam_flat_step", ctypes.c_void_p(fs.table_dev.data_ptr()), fs.count, fs.total_blocks,
                      ctypes.c_void_p(fs.master.data_ptr()), ctypes.c_void_p(fs.sink.flat.data_ptr()),
                      ctypes.c_void_p(fs.bufs["exp_avg"].data_ptr()), ctypes.c_void_p(fs.bufs["exp_avg_sq"].data_ptr()),
                      ctypes.c_void_p(fs.steps.data_ptr()), ctypes.c_void_p(self._scalars.data_ptr()),
                      float(group["lr"]), ctypes.c_void_p(self._lr_dev.data_ptr()) if self._lr_dev is not None else None,
                      float(beta1), float(beta2), float(group["eps"]), float(group["weight_decay"]),
                      int(bool(group["decoupled_weight_decay"])), float(self.grad_scale),
                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        if not capturing:
            fs.after_step(self.state, True)
        return loss

    def sync_lr(self):
        """capturable mode: copy the current learning rate (what a scheduler wrote into param_groups) to the float64
        device scalar the captured prologue reads.  Called by step() when eager, and by GraphedStep.replay()."""
        _sync_lr(self, torch.float64)

    def state_dict(self):
        """torch.optim.Adam's layout: per parameter `step` (fp32 scalar tensor on the CPU), `exp_avg`, `exp_avg_sq`.
        The step counts live on the device and are read back here (one synchronising copy)."""
        sd = super().state_dict()
        fs = self._flat
        host = fs.steps.cpu()
        where = {v.data_ptr(): i for i, v in enumerate(fs.step_views)}
        out = {}
        for k, st in sd["state"].items():
            st = dict(st)
            s = st.get("step")
            if s is not None and s.is_cuda and s.data_ptr() in where:
                st["step"] = host[where[s.data_ptr()]].clone()
            out[k] = st
        sd["state"] = out
        return sd


class _FlatState:
    """Flat master and optimizer-state buffers in the layout of the model's flat gradient sink, the bf16 pack arena and
    the device descriptor table of the flat step entry points (b200unet_sgd_flat_step, b200unet_adam_flat_step).

    `buffers` names the per-parameter state tensors the optimizer keeps (torch's names: "momentum_buffer" for SGD,
    "exp_avg" and "exp_avg_sq" for Adam); each is one flat buffer at the gradient offsets, and `state[p][name]` is a
    view of it.  `step_counters`: an fp32 step count per parameter in device memory (Adam's state["step"]), also held
    in `state[p]` as a view."""

    def __init__(self, model, params: List[nn.Parameter], owner: str, buffers=("momentum_buffer",),
                 step_counters: bool = False):
        sink = sink_of(model)
        if sink is None:
            sink = FlatGradSink(model)
        self.sink = sink
        self.model = model
        wanted = {id(p) for p in params}
        self.params = [p for p in sink.params if id(p) in wanted]
        missing = wanted - {id(p) for p in self.params}
        if missing:
            raise ValueError(f"{owner}(model=...): every optimised parameter must be a trainable parameter of the model")
        for p in self.params:
            if not (p.is_cuda and p.dtype == torch.float32):
                raise RuntimeError(f"{owner}(model=...): move the model to its CUDA device first (fp32 parameters)")
        dev = sink.flat.device
        self.master = torch.zeros(sink.numel, dtype=torch.float32, device=dev)
        self.bufs = {name: torch.zeros(sink.numel, dtype=torch.float32, device=dev) for name in buffers}
        self.mviews: Dict[int, torch.Tensor] = {}
        self.views: Dict[str, Dict[int, torch.Tensor]] = {name: {} for name in buffers}
        for p in self.params:
            off = sink.offsets[id(p)]
            self.mviews[id(p)] = self.master[off:off + p.numel()].view(p.shape)
            for name, buf in self.bufs.items():
                self.views[name][id(p)] = buf[off:off + p.numel()].view(p.shape)
        self._fresh: List[nn.Parameter] = []
        self.steps = torch.zeros(len(self.params), dtype=torch.float32, device=dev) if step_counters else None
        self.step_views = [self.steps[i] for i in range(len(self.params))] if step_counters else None
        # (state name, id(p) -> view) in the order torch creates the state entries
        self._entries = [(name, self.views[name]) for name in buffers]
        if step_counters:
            self._entries.insert(0, ("step", {id(p): v for p, v in zip(self.params, self.step_views)}))
        self._adopt_parameters()
        self._build_packs()
        self.block = _lib.call("b200unet_sgd_flat_block_elems")
        self.count = len(self.params)
        self.flags: List[int] = [-1] * self.count
        self.table_host = (_lib.FlatTensor * self.count)()
        blocks = 0
        for i, p in enumerate(self.params):
            t = self.table_host[i]
            t.offset = sink.offsets[id(p)]
            t.numel = p.numel()
            t.first_block = blocks
            blocks += (p.numel() + self.block - 1) // self.block
            spec = self.packs.get(id(p))
            if spec is not None:
                t.cout, t.cin, t.ksize = spec["cout"], spec["cin"], spec["ksize"]
                t.cout_pad, t.cin_pad = spec["cout_pad"], spec["cin_pad"]
                t.wf = spec["wf"].data_ptr()
                t.wd = spec["wd"].data_ptr() if spec["wd"] is not None else None
                t.ws = spec["ws"].data_ptr() if spec["ws"] is not None else None
        self.total_blocks = blocks
        nbytes = ctypes.sizeof(self.table_host)
        self.table_dev = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.table_pinned = torch.empty(nbytes, dtype=torch.uint8).pin_memory()

    # the parameters become views of the flat master buffer (values preserved); called again if something re-pointed
    # them (model.to(), .float(), a loader that assigns .data)
    def _adopt_parameters(self):
        with torch.no_grad():
            for p in self.params:
                v = self.mviews[id(p)]
                if p.data_ptr() != v.data_ptr():
                    v.copy_(p.detach())
                    p.data = v

    def _build_packs(self):
        """bf16 packs for every conv weight the tensor-core path reads, filled once from the current weights with the
        library's pack kernels and from then on by the optimizer kernel itself; registered with the model."""
        from . import ops
        model = self.model
        self.packs: Dict[int, dict] = {}
        ext = {}
        mine = {id(p) for p in self.params}
        layers = model._layers()
        fusion = model._fusion_unit() if hasattr(model, "_fusion_unit") else None
        units = [(L["unit"][0], "conv") for L in layers]
        if fusion is not None:
            units.append((fusion[0], "fusion"))
        head = model._head_conv()
        if getattr(model, "head_kind", "seg1x1") != "seg1x1":
            units.append((head, "head3x3"))
        first_conv = layers[0]["unit"][0]
        with torch.no_grad():
            for conv, kind in units:
                w = conv.weight
                if id(w) not in mine or id(w) in self.packs:
                    continue
                cout, cin = conv.out_channels, conv.in_channels
                spec = None
                if kind == "conv" and conv is first_conv and cin <= 8 and cout == 32 and conv.stride[0] == 1:
                    wf = ops.pack_stem_weights(w)  # [Cout,3,3,32], input channels zero-padded
                    spec = dict(cout=cout, cin=cin, ksize=3, cout_pad=cout, cin_pad=32, wf=wf, wd=None, ws=None, key="stem")
                elif kind == "conv" and cin % 32 == 0 and cout % 32 == 0 and tuple(conv.kernel_size) == (3, 3):
                    wf, wd = ops.pack_conv_weights(w, need_dgrad=True)
                    ws = ops.pack_s2_dgrad_weights(wd) if conv.stride[0] == 2 else None
                    spec = dict(cout=cout, cin=cin, ksize=3, cout_pad=cout, cin_pad=cin, wf=wf, wd=wd, ws=ws, key="conv")
                elif kind == "fusion" and tuple(conv.kernel_size) == (1, 1) and cin % 32 == 0 and cout % 32 == 0:
                    w3 = torch.zeros((cout, cin, 3, 3), dtype=torch.float32, device=w.device)
                    w3[:, :, 1, 1] = w.detach()[:, :, 0, 0]
                    wf, wd = ops.pack_conv_weights(w3, need_dgrad=True)
                    spec = dict(cout=cout, cin=cin, ksize=1, cout_pad=cout, cin_pad=cin, wf=wf, wd=wd, ws=None, key="k1")
                elif kind == "head3x3" and cin % 32 == 0 and cout <= 4:
                    wp = torch.zeros((32, cin, 3, 3), dtype=torch.float32, device=w.device)
                    wp[:cout] = w.detach()
                    wf, wd = ops.pack_conv_weights(wp, need_dgrad=True)
                    spec = dict(cout=cout, cin=cin, ksize=3, cout_pad=32, cin_pad=cin, wf=wf, wd=wd, ws=None, key="head")
                if spec is None:
                    continue
                spec["version"] = w._version
                self.packs[id(w)] = spec
                ext[id(w)] = spec
        model._ext_packs = ext

    def sync(self, state, stateful: bool):
        """Host-side bookkeeping before the launch: parameters / state buffers re-pointed by someone else are adopted
        again, gradients that autograd did not leave in the flat buffer are copied there, and the per-tensor flags
        (has a gradient / first momentum step) are uploaded when they changed."""
        self._adopt_parameters()
        sink = self.sink
        changed = False
        entries = self._entries
        self._fresh = []  # parameters whose state entries after_step() creates
        for i, p in enumerate(self.params):
            g = p.grad
            flag = 0
            if g is not None:
                flag = 1
                key = id(p)
                gv = sink._views.get(key)
                if gv is None:
                    off = sink.offsets[id(p)]
                    gv = sink._views[id(p)] = sink.flat[off:off + p.numel()].view(p.shape)
                if g.data_ptr() != gv.data_ptr():
                    gv.copy_(g)  # a cloned / accumulated / externally produced gradient: bring it into the flat buffer
                if stateful:
                    st = state[p]
                    missing = None
                    for name, views in entries:  # state loaded by load_state_dict is adopted into the flat buffers
                        t = st.get(name)
                        if t is None:
                            missing = (missing or []) + [name]
                        else:
                            v = views[key]
                            if t.data_ptr() != v.data_ptr():
                                v.copy_(t)
                                st[name] = v
                    if missing:
                        self._fresh.append(p)
                        if self.steps is None:
                            flag |= 2  # SGD: the kernel initialises the momentum buffer with the gradient, as torch does
                        else:
                            for name in missing:  # Adam starts from zero moments and step 0
                                (self.step_views[i] if name == "step" else self.views[name][id(p)]).zero_()
            if flag != self.flags[i]:
                self.flags[i] = flag
                self.table_host[i].flags = flag
                changed = True
        if changed:
            nbytes = ctypes.sizeof(self.table_host)
            ctypes.memmove(self.table_pinned.data_ptr(), ctypes.addressof(self.table_host), nbytes)
            self.table_dev.copy_(self.table_pinned, non_blocking=True)
            # the pinned staging buffer must not be rewritten before this copy has run
            torch.cuda.current_stream().synchronize()

    def after_step(self, state, stateful: bool):
        upd = [p for i, p in enumerate(self.params) if self.flags[i] & 1]
        if not upd:
            return
        _bump_versions(upd)
        for p in upd:
            spec = self.packs.get(id(p))
            if spec is not None:
                spec["version"] = p._version  # the packs were emitted from exactly these values
        if stateful:
            for p in self._fresh:  # first step of p: its state entries are views of the flat buffers
                st = state[p]
                for name, views in self._entries:
                    if name not in st:
                        st[name] = views[id(p)]
