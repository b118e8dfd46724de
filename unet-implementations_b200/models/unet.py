"""B200-native drop-in for the reference's `models.unet` (Ulixes-8/UNet-Implementations, Our_UNet/models/unet.py).

Same classes, constructor arguments, attribute tree and `state_dict` as the reference (`SpatialDropout2d`
unet.py:13-35, `ConvBlock` :37-141, `UpBlock` :143-231, `UNet` :233-432), so `src/train.py` / `src/evaluate.py`
construct, checkpoint and call it unchanged.  What differs is everything below the module surface:
`UNet.forward` runs as ONE `torch.autograd.Function` whose forward and backward enqueue the hand-written sm_100a
kernels of libb200unet.so (include/b200unet.h) on torch's current stream:

    conv 3x3 (tcgen05 implicit GEMM, raw bf16 output + InstanceNorm partial sums in the epilogue)
      -> finalize (per-(n,c) mean/rstd folded with gamma, beta and the SpatialDropout scale)
      -> apply (normalise + LeakyReLU + channel dropout in one pass, written straight into its consumer's buffer:
                the next conv's input or the skip half of a decoder concat buffer -- torch.cat never runs)
    bilinear 2x upsample written into the other half of the concat buffer; 1x1 head -> fp32 NCHW logits.

Activations live as NHWC bf16; parameters stay fp32 OIHW `nn.Parameter`s and receive fp32 `.grad`s.
There is no torch/cuDNN/CPU fallback on this path: without the CUDA library or an sm_100 device it raises.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple, Type, Union

import os

import torch
import torch.nn as nn
import torch.nn.functional as F

try:  # package import (unet_implementations_b200.models.unet)
    from .. import ops, packs
except ImportError:  # imported as top-level `models.unet` through the drop-in shim directory
    from unet_implementations_b200 import ops, packs

BF16 = torch.bfloat16


def _lib_call(name, *args):
    return ops._lib.call(name, *args)


class SpatialDropout2d(nn.Module):
    """Channel dropout of the reference (unet.py:13-35): one Bernoulli(1-p) draw per (sample, channel), kept
    channels scaled by 1/(1-p).  Inside `UNet.forward` the draw below is made with the reference's exact call
    (`draw`), and the resulting [N,C] scale is folded into the fused normalise kernel."""

    def __init__(self, drop_prob):
        super().__init__()
        self.drop_prob = drop_prob

    def draw(self, like: torch.Tensor, batch: int, channels: int) -> torch.Tensor:
        # the reference's call, verbatim in shape/dtype/device so that the same seed gives the same mask (unet.py:30-31)
        mask = like.new_empty(batch, channels, 1, 1).bernoulli_(1 - self.drop_prob)
        return mask.div_(1 - self.drop_prob)

    def forward(self, x):
        if not self.training or self.drop_prob == 0:
            return x
        mask = self.draw(x, x.size(0), x.size(1))
        return x * mask.expand_as(x)


class ConvBlock(nn.Module):
    """[Conv2d 3x3 (stride on the first conv only) -> InstanceNorm2d -> LeakyReLU -> SpatialDropout2d] x n_convs in
    one `nn.Sequential` called `.block`, built in the reference's order (unet.py:97-134) so that parameter
    names, shapes and the RNG consumed by construction are identical."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: Union[int, Tuple[int, int]],
                 stride: Union[int, Tuple[int, int]], n_convs: int = 2, padding: Optional[int] = None,
                 norm_op: Type[nn.Module] = nn.InstanceNorm2d, norm_op_kwargs: Dict = None,
                 dropout_op: Optional[Type[nn.Module]] = None, dropout_op_kwargs: Dict = None,
                 nonlin: Type[nn.Module] = nn.LeakyReLU, nonlin_kwargs: Dict = None, conv_bias: bool = True,
                 spatial_dropout_rate: float = 0.0):
        super().__init__()
        norm_op_kwargs = {"eps": 1e-5, "affine": True} if norm_op_kwargs is None else norm_op_kwargs
        nonlin_kwargs = {"inplace": True} if nonlin_kwargs is None else nonlin_kwargs
        dropout_op_kwargs = {} if dropout_op_kwargs is None else dropout_op_kwargs
        if padding is None:
            padding = kernel_size // 2 if isinstance(kernel_size, int) else (kernel_size[0] // 2, kernel_size[1] // 2)
        layers: List[nn.Module] = []
        ch = in_channels
        for i in range(n_convs):
            layers.append(nn.Conv2d(ch, out_channels, kernel_size, stride if i == 0 else 1, padding, bias=conv_bias))
            if norm_op is not None:
                layers.append(norm_op(out_channels, **norm_op_kwargs))
            if nonlin is not None:
                layers.append(nonlin(**nonlin_kwargs))
            if spatial_dropout_rate > 0:
                layers.append(SpatialDropout2d(spatial_dropout_rate))
            if dropout_op is not None:
                layers.append(dropout_op(**dropout_op_kwargs))
            ch = out_channels
        self.block = nn.Sequential(*layers)

    def units(self):
        """The block parsed into fused units: [(conv, norm, nonlin, spatial_dropout or None), ...].  Raises for a
        composition the kernels do not implement (anything but the trainer's, train.py:776-795)."""
        mods = list(self.block)
        out, i = [], 0
        while i < len(mods):
            conv = mods[i]
            norm = mods[i + 1] if i + 1 < len(mods) else None
            act = mods[i + 2] if i + 2 < len(mods) else None
            if not (isinstance(conv, nn.Conv2d) and isinstance(norm, nn.InstanceNorm2d) and isinstance(act, nn.LeakyReLU)):
                raise NotImplementedError(
                    "b200unet implements ConvBlock = [Conv2d 3x3 -> InstanceNorm2d(affine) -> LeakyReLU -> "
                    f"SpatialDropout2d]; got {[type(m).__name__ for m in mods]}")
            i += 3
            drop = None
            if i < len(mods) and isinstance(mods[i], SpatialDropout2d):
                drop = mods[i]
                i += 1
            if tuple(conv.kernel_size) != (3, 3) or tuple(conv.padding) != (1, 1) or conv.stride[0] != conv.stride[1] \
                    or conv.stride[0] not in (1, 2) or conv.groups != 1 or tuple(conv.dilation) != (1, 1):
                raise NotImplementedError(f"b200unet: unsupported conv {conv}")
            if not norm.affine or norm.track_running_stats:
                raise NotImplementedError("b200unet: InstanceNorm2d must be affine without running stats")
            out.append((conv, norm, act, drop))
        return out

    def forward(self, x):
        """Stand-alone use (NCHW fp32 in and out); `UNet.forward` does not go through here."""
        return _run_block_standalone(self, x)


class UpBlock(nn.Module):
    """Bilinear upsample to the skip's size, cat([x, skip], 1), ConvBlock (unet.py:143-231)."""

    def __init__(self, in_channels: int, skip_channels: int, out_channels: int,
                 kernel_size: Union[int, Tuple[int, int]], n_convs: int = 2,
                 norm_op: Type[nn.Module] = nn.InstanceNorm2d, norm_op_kwargs: Dict = None,
                 dropout_op: Optional[Type[nn.Module]] = None, dropout_op_kwargs: Dict = None,
                 nonlin: Type[nn.Module] = nn.LeakyReLU, nonlin_kwargs: Dict = None, conv_bias: bool = True,
                 spatial_dropout_rate: float = 0.0):
        super().__init__()
        self.conv_block = ConvBlock(in_channels + skip_channels, out_channels, kernel_size, stride=1, n_convs=n_convs,
                                    padding=None, norm_op=norm_op, norm_op_kwargs=norm_op_kwargs,
                                    dropout_op=dropout_op, dropout_op_kwargs=dropout_op_kwargs, nonlin=nonlin,
                                    nonlin_kwargs=nonlin_kwargs, conv_bias=conv_bias,
                                    spatial_dropout_rate=spatial_dropout_rate)

    def forward(self, x, skip):
        """Stand-alone use (NCHW fp32 in and out, unet.py:203-231): bilinear 2x upsample written into the concat buffer
        next to the skip, then the ConvBlock.  `UNet.forward` does not go through here (it keeps everything NHWC)."""
        if not (x.is_cuda and skip.is_cuda):
            raise RuntimeError("b200unet: UpBlock needs CUDA tensors on an sm_100 device; there is no CPU path")
        return self.conv_block(_UpsampleCatFunction.apply(x, skip))


class UNet(nn.Module):
    """The reference's 6-stage encoder-decoder (unet.py:233-432) with its constructor, attributes and state_dict."""

    def __init__(self, in_channels: int = 3, num_classes: int = 3, n_stages: int = 6,
                 features_per_stage: List[int] = None, kernel_sizes: List[Tuple[int, int]] = None,
                 strides: List[Tuple[int, int]] = None, n_conv_per_stage: List[int] = None,
                 n_conv_per_stage_decoder: List[int] = None, conv_bias: bool = True,
                 norm_op: Type[nn.Module] = nn.InstanceNorm2d, norm_op_kwargs: Dict = None,
                 dropout_op: Optional[Type[nn.Module]] = None, dropout_op_kwargs: Dict = None,
                 nonlin: Type[nn.Module] = nn.LeakyReLU, nonlin_kwargs: Dict = None,
                 encoder_dropout_rates: List[float] = None, decoder_dropout_rates: List[float] = None):
        super().__init__()
        if features_per_stage is None:
            features_per_stage = [32, 64, 128, 256, 512, 512]
        if kernel_sizes is None:
            kernel_sizes = [[3, 3]] * n_stages
        if strides is None:
            strides = [[1, 1]] + [[2, 2]] * (n_stages - 1)
        if n_conv_per_stage is None:
            n_conv_per_stage = [2] * n_stages
        if n_conv_per_stage_decoder is None:
            n_conv_per_stage_decoder = [2] * (n_stages - 1)
        if norm_op_kwargs is None:
            norm_op_kwargs = {"eps": 1e-5, "affine": True}
        if nonlin_kwargs is None:
            nonlin_kwargs = {"inplace": True}
        if encoder_dropout_rates is None:
            encoder_dropout_rates = [0.0, 0.0, 0.1, 0.2, 0.3, 0.3]
        if decoder_dropout_rates is None:
            decoder_dropout_rates = [0.3, 0.2, 0.2, 0.1, 0.0]
        self.in_channels = in_channels
        self.num_classes = num_classes
        self.n_stages = n_stages
        self.features_per_stage = features_per_stage

        common = dict(norm_op=norm_op, norm_op_kwargs=norm_op_kwargs, dropout_op=dropout_op,
                      dropout_op_kwargs=dropout_op_kwargs, nonlin=nonlin, nonlin_kwargs=nonlin_kwargs,
                      conv_bias=conv_bias)
        self.encoder_stages = nn.ModuleList()
        ch = in_channels
        for s in range(n_stages):
            self.encoder_stages.append(ConvBlock(ch, features_per_stage[s], kernel_sizes[s], strides[s],
                                                 n_convs=n_conv_per_stage[s],
                                                 spatial_dropout_rate=encoder_dropout_rates[s], **common))
            ch = features_per_stage[s]
        # variant hook: modules the reference creates between the encoder and the decoder (CLIP fusion layer)
        self._build_bottleneck(features_per_stage[-1], conv_bias, norm_op, norm_op_kwargs, nonlin, nonlin_kwargs)
        self.decoder_stages = nn.ModuleList()
        for j in range(n_stages - 1):
            d = n_stages - 2 - j
            self.decoder_stages.append(UpBlock(features_per_stage[d + 1], features_per_stage[d], features_per_stage[d],
                                               kernel_sizes[d], n_convs=n_conv_per_stage_decoder[d],
                                               spatial_dropout_rate=decoder_dropout_rates[j], **common))
        self._build_head(features_per_stage[0], num_classes)
        self.initialize_weights()
        # test/DDP hooks (not part of the reference surface)
        self._mask_override: Optional[List[torch.Tensor]] = None  # inject dropout masks instead of drawing them
        self.last_dropout_masks: List[torch.Tensor] = []          # [N,C] scales used by the last training forward
        self._trace = None                                        # debug: list collecting (raw conv out, activation) per unit
        self._trace_bwd = None                                    # debug: list collecting the backward tensors per unit
        self._trace_fwd = None                                    # debug: forward tensors per unit WITHOUT changing the path
        self._grad_sink = None                                    # callable(param, grad) fired as backward produces grads
        # backward runs each weight-gradient kernel (tensor-bound) on a side stream, concurrently with the NEXT layer's
        # InstanceNorm backward (HBM-bound) on the main stream; B200UNET_OVERLAP=0 or this flag = False serialises
        self.overlap_wgrad = os.environ.get("B200UNET_OVERLAP", "1") != "0"
        # kernels that write a gradient dz also reduce the norm-backward sums of the unit that consumes it (A/B knob)
        self.producer_sums = os.environ.get("B200UNET_PRODUCER_SUMS", "1") != "0"          # the head backward (a gain)
        self.split_concat_grad = os.environ.get("B200UNET_SPLIT_DCAT", "1") != "0"  # A/B knob (models/unet.py backward)
        # fusion variant: extra features that are constant over each (sample, channel) plane cancel in the InstanceNorm
        self.skip_constant_features = True
        self.producer_sums_dgrad = os.environ.get("B200UNET_PRODUCER_SUMS_DGRAD", "0") == "1"  # dgrad epilogues (a loss)
        self._side_streams: Dict[int, torch.cuda.Stream] = {}
        self._packs = packs.PackStore()  # the conv weight packs the kernels read (packs.py)
        # "bf16": production path (tcgen05 convs, NHWC bf16 arena).  "fp32": verification mode -- the same fused
        # forward/backward with an fp32 arena, the storage-type templates of the norm/resample/head kernels and the
        # direct fp32 convs; agrees with the reference to 1e-4 on loss and every gradient (tests/test_gpu_model.py)
        self.precision = "bf16"

    # which output layer follows the decoder: "seg1x1" = Conv2d(32 -> classes, 1x1) (unet.py:374-381);
    # "recon3x3" = Conv2d(32 -> 3, 3x3) + Sigmoid (the autoencoder variant, models/autoencoder.py)
    head_kind = "seg1x1"

    def _build_head(self, features: int, out_channels: int):
        self.segmentation_output = nn.Conv2d(features, out_channels, kernel_size=1, stride=1, padding=0, bias=True)

    def _head_conv(self) -> nn.Conv2d:
        return self.segmentation_output

    def _build_bottleneck(self, features, conv_bias, norm_op, norm_op_kwargs, nonlin, nonlin_kwargs):
        return None

    def _fusion_unit(self):
        """(conv1x1, norm, act, None) applied to cat([bottleneck, extra features]) before the decoder, or None."""
        return None

    def initialize_weights(self):
        """kaiming_normal_(fan_out, leaky_relu) on conv weights, zero conv biases, IN weight 1 / bias 0 (unet.py:386-397)."""
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="leaky_relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.InstanceNorm2d):
                if m.weight is not None:
                    nn.init.constant_(m.weight, 1)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)

    @property
    def _ext_packs(self):  # read-only view of _packs.emitted: id(weight) -> {"key", "version", "wf", "wd", "ws"}
        return {k: dict(key=p.layout.kind, version=p.version, wf=p.wf, wd=p.wd, ws=p.ws)
                for k, p in self._packs.emitted.items()}

    # ------------------------------------------------------------------------------------------------ plan
    def _layers(self):
        """Flat list of fused units in forward order with their role in the graph."""
        layers = []
        for s, stage in enumerate(self.encoder_stages):
            us = stage.units()
            if len(us) < 1:
                raise NotImplementedError("b200unet: a stage needs at least one conv")
            for i, u in enumerate(us):
                layers.append(dict(kind="enc", stage=s, idx=i, last=(i == len(us) - 1), unit=u))
        for j, up in enumerate(self.decoder_stages):
            us = up.conv_block.units()
            for i, u in enumerate(us):
                layers.append(dict(kind="dec", stage=j, idx=i, last=(i == len(us) - 1), unit=u))
        return layers

    # normalisation applied to uint8 HWC input batches (the dataset's, train.py:303-308)
    input_mean = (0.485, 0.456, 0.406)
    input_std = (0.229, 0.224, 0.225)

    def forward(self, x):
        """x: fp32 NCHW [B,C,H,W] as the trainer feeds it (train.py:630), or -- SURVEY.md 8f row 2 -- the batch as the
        dataset stores it: uint8 HWC [B,H,W,3], normalised on the device inside the stem's layout kernel."""
        if x.dtype == torch.uint8:
            if x.dim() != 4 or x.size(3) != self.in_channels or self.in_channels != 3:
                raise ValueError(f"UNet.forward expects uint8 [B,H,W,3] images, got {tuple(x.shape)}")
        elif x.dim() != 4 or x.size(1) != self.in_channels:
            raise ValueError(f"UNet.forward expects [B,{self.in_channels},H,W], got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("b200unet: UNet.forward needs a CUDA tensor on an sm_100 device; there is no CPU path")
        if x.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError("b200unet: the gradient with respect to the input image is not computed by the fused "
                                      "backward (the stem's data gradient is skipped, SURVEY.md A.1); detach the input")
        params = [p for p in self.parameters()]
        return _UNetFunction.apply(self, x, *params)


# ====================================================================================================================
# The fused forward/backward
# ====================================================================================================================
# ====================================================================================================================
# Hooks on inner Conv2d modules (Grad-CAM: Our_UNet/utils/visualize.py:391-402 registers a forward and a backward hook on
# `decoder_stages[0].conv_block.block[0]`).  Inside the fused node no nn.Module.__call__ runs, so the hooks are fired
# by hand with what a stock module would have shown them: (input,), output = conv(input) + bias in NCHW fp32, and in
# backward grad_output = d loss / d output.  Only observation is supported (a hook that returns a replacement raises).
# ====================================================================================================================
def _to_nchw_f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype == BF16 and t.stride(3) == 1:
        return ops.nhwc_to_nchw(t)
    return t.permute(0, 3, 1, 2).float().contiguous()


def _fire_forward_hooks(conv: nn.Conv2d, x_nchw_or_nhwc, y_nhwc, is_nchw_input: bool):
    out = _to_nchw_f32(y_nhwc)
    if conv.bias is not None:
        out = out + conv.bias.detach().view(1, -1, 1, 1)
    inp = x_nchw_or_nhwc if is_nchw_input else _to_nchw_f32(x_nchw_or_nhwc)
    for hook in list(conv._forward_hooks.values()):
        if hook(conv, (inp,), out) is not None:
            raise NotImplementedError("b200unet: a forward hook on an inner Conv2d may observe its output, not replace it")


def _fire_backward_hooks(conv: nn.Conv2d, dx_nhwc, dy_nhwc):
    go = (_to_nchw_f32(dy_nhwc),)
    gi = (_to_nchw_f32(dx_nhwc),)
    for hook in list(conv._backward_hooks.values()):
        if hook(conv, gi, go) is not None:
            raise NotImplementedError("b200unet: a backward hook on an inner Conv2d may observe gradients, not replace them")


def _use_tc(cin: int, cout: int) -> bool:
    return cin % 32 == 0 and cout % 32 == 0


def _conv_fwd(x, wf, stride, out=None):
    cout, cin = wf.shape[0], wf.shape[3]
    return ops.conv_fprop(x, wf, stride, out=out, want_stats=True, simt=not _use_tc(cin, cout))


class _UNetFunction(torch.autograd.Function):
    """forward(model, image, *parameters) -> fp32 NCHW logits.  One autograd node for the whole network: the saved
    state is the NHWC bf16 arena (raw conv outputs, post-activation tensors, concat buffers) plus [N,C] statistics."""

    @staticmethod
    def forward(ctx, model: UNet, x: torch.Tensor, *params):
        ops.require_device()
        with torch.cuda.device(x.device):
            return _forward_impl(ctx, model, x, params)

    @staticmethod
    def backward(ctx, dlogits):
        # a data-parallel reducer asks the conv grids of backward to leave a few SMs to its NCCL kernels (ddp.py)
        sink = getattr(getattr(ctx, "model", None), "_grad_sink", None)
        reserve = int(getattr(sink, "reserve_sms", 0) or 0)
        prev = _lib_call("b200unet_set_reserved_sms", reserve) if reserve else 0
        try:
            with torch.cuda.device(dlogits.device):
                grads = _backward_impl(ctx, dlogits)
        finally:
            if reserve:
                _lib_call("b200unet_set_reserved_sms", prev)
        return (None, None) + tuple(grads)


def _forward_impl(ctx, model: UNet, x: torch.Tensor, params):
    x = x.detach()
    x_u8 = None
    if x.dtype == torch.uint8:
        x_u8 = x.contiguous()
        B, H, W, _ = x_u8.shape
        x = None  # the fp32 NCHW image is only materialised for the paths that need it (_image())
    else:
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        B, _, H, W = x.shape

    def _image():
        nonlocal x
        if x is None:
            from ..data import preprocess_batch
            x = preprocess_batch(x_u8, None, model.input_mean, model.input_std)[0]
        return x
    n = model.n_stages
    feats = list(model.features_per_stage)
    layers = model._layers()
    training = model.training
    if model.precision not in ("bf16", "fp32"):
        raise ValueError(f"b200unet: precision must be 'bf16' or 'fp32', got {model.precision!r}")
    adt = torch.float32 if model.precision == "fp32" else BF16  # activation storage type of the arena
    need_grad = any(ctx.needs_input_grad[2:])  # grad mode is off inside Function.forward; this is the autograd truth
    dev = x_u8.device if x_u8 is not None else x.device

    # spatial size per encoder level
    sizes = []
    h, w = H, W
    for s in range(n):
        st = model.encoder_stages[s].block[0].stride[0]
        h, w = ops.conv_out_hw(h, w, st)
        sizes.append((h, w))
    for d in range(n - 1):
        if sizes[d] != (2 * sizes[d + 1][0], 2 * sizes[d + 1][1]):
            raise NotImplementedError(
                f"b200unet: the upsample kernel is the exact 2x case of F.interpolate (unet.py:220-225); level {d} is "
                f"{sizes[d]} over {sizes[d + 1]} -- use an input size divisible by {2 ** (n - 1)}")

    # decoder concat buffers: cat[d] = [upsampled level d+1 (feats[d+1]) | skip of level d (feats[d])]
    cat = [torch.empty((B, sizes[d][0], sizes[d][1], feats[d + 1] + feats[d]), dtype=adt, device=dev)
           for d in range(n - 1)]

    # dropout scales, drawn in the reference's order with the reference's call (SURVEY.md A.3)
    _f32_like = x if x is not None else torch.empty(0, dtype=torch.float32, device=dev)
    override = list(model._mask_override) if model._mask_override is not None else None
    used_masks = []

    def draw(drop: Optional[SpatialDropout2d], c: int):
        if drop is None or not training or drop.drop_prob == 0:
            return None
        if override is not None:
            m = override.pop(0).to(device=dev, dtype=torch.float32)
        else:
            m = drop.draw(_f32_like, B, c)
        m = m.reshape(B, c).contiguous()
        used_masks.append(m)
        return m

    # optional fusion of extra features at the bottleneck (CLIP_UNet/models/unet.py:441-478): cat([x, features], 1)
    # -> 1x1 conv -> norm -> act.  The last encoder unit writes its activation straight into the concat buffer.
    extra = getattr(model, "_extra_features", None)
    fusion = model._fusion_unit() if extra is not None else None
    catf = None
    const_extra = False
    if fusion is not None:
        fh, fw = sizes[-1]
        # A pooled embedding broadcast over the grid -- what the reference's ClipPatchExtractor produces
        # (`features.view(B, D, 1, 1).expand(-1, -1, 16, 16)`, CLIP_UNet/models/unet.py:611-612: spatial strides 0) -- is
        # constant over each (sample, channel) plane.  Its half of the 1x1 fusion conv is then a per-(sample, channel)
        # constant added to the conv output, which the InstanceNorm that follows subtracts again with the plane mean:
        # like the conv biases (SURVEY.md 8a) it cancels exactly, and its weight gradient is exactly zero.  The fusion
        # conv then runs over the bottleneck's channels only (half the K, no concat buffer, no feature re-layout).
        const_extra = model.skip_constant_features and extra.dim() == 4 and (
            tuple(extra.shape[2:]) == (1, 1) or (extra.stride(2) == 0 and extra.stride(3) == 0))
        if not const_extra:
            if extra.shape[2:] != (fh, fw):
                extra = F.interpolate(extra.float(), size=(fh, fw), mode="bilinear", align_corners=False)  # unet.py:444-451
            catf = torch.empty((B, fh, fw, feats[-1] + extra.shape[1]), dtype=adt, device=dev)
            ops.nchw_to_nhwc(extra.detach().float().contiguous(), out=catf[..., feats[-1]:])
        layers = [L for L in layers if L["kind"] == "enc"] + [dict(kind="fusion", stage=0, idx=0, last=True, unit=fusion)] + \
                 [L for L in layers if L["kind"] == "dec"]

    saved = []  # per layer dict
    cur = None  # current NHWC bf16 activation
    # (a, b, slope) when `cur` is a RAW conv output whose apply pass is fused into its single consumer -- the 2x
    # upsample of the next decoder stage or the 1x1 head -- instead of being run (and written) on its own
    cur_norm = None
    for li_f, L in enumerate(layers):
        conv, norm, act, drop = L["unit"]
        cin, cout = conv.in_channels, conv.out_channels
        stride = conv.stride[0]
        rec = dict(L=L, stride=stride)
        if L["kind"] == "dec" and L["idx"] == 0:
            d = n - 2 - L["stage"]
            c_low = feats[d + 1]
            ops.upsample2x(cur, cat[d][..., :c_low], norm=cur_norm)
            if model._trace_fwd is not None:
                model._trace_fwd.append(dict(kind="up", src=cur, norm=cur_norm, out=cat[d][..., :c_low]))
            rec["low"] = cur  # only its shape matters in backward
            cur = cat[d]
            cur_norm = None
        first = L["kind"] == "enc" and L["stage"] == 0 and L["idx"] == 0
        if first:
            if cin <= 8 and cout == 32 and stride == 1 and adt == BF16 and W >= 64:
                # stem on the tensor-core path: image -> bf16 NHWC zero-padded to 32 channels (64 B per pixel), then
                # the narrow-output 32 -> 32 kernels; the padded copy is also the X operand of the weight gradient.
                # A uint8 HWC batch is normalised inside that one layout kernel (no fp32 image in HBM at all).
                if x_u8 is not None:
                    xin32 = ops.preprocess_u8_nhwc32(x_u8, model.input_mean, model.input_std)
                else:
                    xin32 = ops.image_to_nhwc32(x)
                y, stats = ops.conv_fprop(xin32, model._packs.get(conv, "stem", BF16, False)[0], 1, want_stats=True)
                rec["stem"] = True
                rec["xin32"] = xin32 if need_grad else None
            elif cin == 3 and cout == 32 and stride == 1 and adt == BF16:
                y, stats = ops.stem_fprop(_image(), conv.weight)
                rec["stem"] = True
            else:
                xin = ops.nchw_to_nhwc(_image(), out=_padded_nhwc(B, H, W, cin, dev, adt))
                wf, wd = model._packs.get(conv, "conv", adt, False)
                y, stats = _conv_fwd(xin, wf, stride)
                rec["xin"] = xin
                rec["stem"] = False
        else:
            if L["kind"] == "fusion":
                if conv.kernel_size != (1, 1) or conv.in_channels != feats[-1] + extra.shape[1]:
                    raise NotImplementedError("b200unet: the fusion layer must be a 1x1 conv over cat([bottleneck, features])")
                if const_extra:
                    wf, wd = model._packs.get(conv, "k1", adt, need_grad, cin_used=feats[-1])
                    rec["cin_used"] = feats[-1]
                else:
                    cur = catf
                    wf, wd = model._packs.get(conv, "k1", adt, need_grad)
            else:
                wf, wd = model._packs.get(conv, "conv", adt, need_grad)
            y, stats = _conv_fwd(cur, wf, stride)
            rec["xin"] = cur
            rec["wd"] = wd
        if conv._forward_hooks:
            _fire_forward_hooks(conv, _image() if first else cur, y, first)
        scale = draw(drop, cout)
        oh, ow = y.shape[1], y.shape[2]
        mean, rstd, a, b = ops.in_finalize(stats, norm.weight, norm.bias, scale, norm.eps, oh * ow)
        # destination of the activated tensor: the skip half of a concat buffer for the last unit of an encoder stage
        dst = None
        if L["kind"] == "enc" and L["last"] and L["stage"] < n - 1:
            d = L["stage"]
            dst = cat[d][..., feats[d + 1]:]
        elif L["kind"] == "enc" and L["last"] and catf is not None:
            dst = catf[..., :feats[-1]]
        nxt = layers[li_f + 1] if li_f + 1 < len(layers) else None
        fuse_into_consumer = model._trace is None and dst is None and (
            (nxt is not None and nxt["kind"] == "dec" and nxt["idx"] == 0) or (nxt is None and model.head_kind == "seg1x1"))
        if fuse_into_consumer:
            z, cur_norm = y, (a, b, act.negative_slope)
        else:
            z, cur_norm = ops.in_apply(y, a, b, act.negative_slope, out=dst), None
        rec.update(y=y, mean=mean, rstd=rstd, a=a, b=b, scale=scale, slope=act.negative_slope, conv=conv, norm=norm)
        if model._trace_fwd is not None:
            model._trace_fwd.append(dict(kind="unit", li=li_f, L=L, conv=conv, norm=norm, stride=stride, slope=act.negative_slope,
                                         xin=rec.get("xin32") if rec.get("xin32") is not None else rec.get("xin"),
                                         y=y, mean=mean, rstd=rstd, a=a, b=b, scale=scale,
                                         z=None if fuse_into_consumer else z))
        saved.append(rec)
        cur = z
        if model._trace is not None:
            model._trace.append((y, z))
    head = model._head_conv()
    if model.head_kind == "seg1x1":
        if head.in_channels != 32 or head.out_channels != 3 or head.bias is None:
            raise NotImplementedError("b200unet: the head kernel is built for Conv2d(32 -> 3, 1x1, bias) (unet.py:374-381)")
        logits = ops.head_forward(cur, head.weight, head.bias, norm=cur_norm)
        if model._trace_fwd is not None:
            model._trace_fwd.append(dict(kind="head", z=cur, norm=cur_norm, logits=logits))
        if need_grad:
            ctx.head_norm = cur_norm
    else:
        # reconstruction head (autoencoder.py:374-387): 3x3 conv 32 -> K on the conv kernels with the output channels
        # zero-padded (bf16: to the tensor-core kernels' 32; fp32: to the 8-channel vector width), then bias + sigmoid
        if head.out_channels > 4 or head.bias is None or head.in_channels % 32 != 0:
            raise NotImplementedError("b200unet: the reconstruction head is built for Conv2d(32k -> <=4, 3x3, bias) + Sigmoid")
        wfh, wdh = model._packs.get(head, "head", adt, need_grad)
        yh, _ = ops.conv_fprop(cur, wfh, 1, want_stats=False, simt=not _use_tc(head.in_channels, wfh.shape[0]))
        logits = ops.recon_head_forward(yh[..., :head.out_channels], head.bias)
        if need_grad:
            ctx.head_out = logits
            ctx.head_wd = wdh
    model.last_dropout_masks = used_masks
    if need_grad:
        ctx.model = model
        ctx.saved = saved
        ctx.image = x  # None for a uint8 batch on the tensor-core stem (its weight gradient reads the padded bf16 copy)
        ctx.image_u8 = x_u8
        ctx.z_last = cur
        ctx.cat = cat
        ctx.sizes = sizes
        ctx.param_ids = {id(p): i for i, p in enumerate(params)}
        ctx.param_req = [p.requires_grad for p in params]
        ctx.n_params = len(params)
    else:
        ctx.saved = None
    return logits


def _padded_nhwc(B, H, W, C, dev, dtype=BF16):
    pitch = (C + 7) // 8 * 8
    buf = torch.zeros((B, H, W, pitch), dtype=dtype, device=dev)
    return buf[..., :C]


def _backward_impl(ctx, dlogits):
    if ctx.saved is None:
        raise RuntimeError("b200unet: backward called on a forward that ran without grad")
    model: UNet = ctx.model
    saved = ctx.saved
    n = model.n_stages
    feats = list(model.features_per_stage)
    grads: List[Optional[torch.Tensor]] = [None] * ctx.n_params
    ids = ctx.param_ids
    req = ctx.param_req
    sink = model._grad_sink

    in_place = sink is not None and hasattr(sink, "dest")

    def wants(p: Optional[nn.Parameter]) -> bool:
        return p is not None and req[ids[id(p)]]

    def dest(p: Optional[nn.Parameter]):
        """Slot of p's gradient in the sink's flat buffer (the producing kernel writes there), or None."""
        if sink is None or not wants(p) or not hasattr(sink, "dest"):
            return None
        return sink.dest(p)

    def put(p: Optional[nn.Parameter], g_fn):
        """Store the gradient of parameter p (computed lazily, only if it requires grad)."""
        if not wants(p):
            return
        g = g_fn()
        if sink is not None:
            g = sink(p, g)
            if in_place and p.grad is None:
                # the gradient lives in the sink's flat buffer: make it p.grad directly and hand autograd nothing --
                # AccumulateGrad would otherwise CLONE the view (it only adopts tensors that are not views), an
                # extra 78.6 MB copy per step, and p.grad would no longer be the memory the fused optimizer reads
                p.grad = g
                return
        grads[ids[id(p)]] = g

    # the 22 conv biases that feed an InstanceNorm have an exactly-zero gradient (SURVEY.md 8a).  With a flat sink their
    # slots were zeroed at construction and are never written; otherwise ONE zero buffer per backward is sliced
    # (each bias its own memory: autograd may adopt the slice as .grad) instead of one zeros_like launch per layer
    dead_bias = [rec["conv"].bias for rec in saved if wants(rec["conv"].bias)]
    zero_pool, zero_off = None, [0]
    if dead_bias and (sink is None or not hasattr(sink, "dest")):
        zero_pool = torch.zeros(sum((b.numel() + 3) // 4 * 4 for b in dead_bias), dtype=torch.float32, device=dlogits.device)

    def zero_grad_of(b: nn.Parameter):
        d = dest(b)
        if d is not None:
            return d
        if zero_pool is None:
            return torch.zeros_like(b)
        v = zero_pool[zero_off[0]:zero_off[0] + b.numel()].view(b.shape)
        zero_off[0] += (b.numel() + 3) // 4 * 4
        return v

    btrace = model._trace_bwd  # debug/test: per-layer backward tensors (tests/test_gpu_layerwise.py)

    # the earliest layer (forward order) that still has a trainable parameter: backward stops there
    first_needed = len(saved)
    for li, rec in enumerate(saved):
        ps = [rec["conv"].weight, rec["conv"].bias, rec["norm"].weight, rec["norm"].bias]
        if any(p is not None and req[ids[id(p)]] for p in ps):
            first_needed = li
            break

    head = model._head_conv()
    if dlogits.dtype != torch.float32:
        dlogits = dlogits.float()
    ext_part = None  # norm-backward partial sums of the NEXT unit to process, produced by the kernel that wrote its dz
    if model.head_kind == "seg1x1":
        if ctx.head_norm is not None and model.producer_sums:
            # the head backward reads the last unit's raw output anyway (it recomputes z for dW): it also reduces that
            # unit's norm-backward sums, whose own reduction pass over (dz, y) -- 1.07 GB at 512^2 x 32 -- disappears
            dz, dwh, dbh, ext_part = ops.head_backward(dlogits, ctx.z_last, head.weight, norm=ctx.head_norm,
                                                       out_dw=dest(head.weight), out_db=dest(head.bias), want_bwd_part=True)
        else:
            dz, dwh, dbh = ops.head_backward(dlogits, ctx.z_last, head.weight, norm=ctx.head_norm, out_dw=dest(head.weight),
                                             out_db=dest(head.bias))
    else:
        z_last, wdh = ctx.z_last, ctx.head_wd
        cpad = wdh.shape[3]
        dpre, dbh = ops.recon_head_backward(dlogits, ctx.head_out, cpad, z_last.dtype)
        simt_h = not _use_tc(head.in_channels, cpad)
        dz = ops.conv_dgrad(dpre, wdh, (z_last.shape[1], z_last.shape[2]), 1, simt=simt_h)
        dwh = ops.conv_wgrad(z_last, dpre, 1, simt=simt_h)[:head.out_channels].contiguous()
        ctx.head_out = None
    if btrace is not None:
        btrace.append(dict(kind="head", dlogits=dlogits, dz=dz, dw=dwh, db=dbh))
    put(head.weight, lambda: dwh)
    put(head.bias, lambda: dbh)

    # Weight gradients off the critical path.  The chain  norm-backward(k) -> dgrad(k) -> norm-backward(k-1) -> ...  is
    # the critical path of backward; wgrad(k) only needs dy(k).  It is launched on a side stream once dgrad(k) has
    # finished, so that it (tensor-bound) runs concurrently with norm-backward(k-1) (HBM-bound) on the main stream; the
    # main stream picks the gradient up one layer later (wait on its event, then hand it to the sink / autograd).
    main = torch.cuda.current_stream()
    overlap = bool(model.overlap_wgrad)
    side = None
    if overlap:
        side = model._side_streams.get(main.device.index)
        if side is None:
            side = model._side_streams[main.device.index] = torch.cuda.Stream(device=main.device)
    pending = []  # [(param, gradient tensor, event recorded on the side stream, tensors the side stream reads)]

    def collect():
        while pending:
            p, g, ev, _inputs = pending.pop(0)
            main.wait_event(ev)
            g.record_stream(main)
            put(p, lambda: g)
            # _inputs (main-stream tensors the side stream was reading) are released only here, after the main stream
            # has been ordered behind the side-stream work: no record_stream on the big activations, whose deferred
            # reuse made the caching allocator grow and stall now and then (100 ms steps in bench.py)

    def wgrad_async(p: Optional[nn.Parameter], fn, inputs, trec=None):
        """Run fn() (a weight-gradient launch) for parameter p: on the side stream after everything enqueued on the
        main stream so far, or inline when overlap is off."""
        if not wants(p):
            return
        if not overlap:
            g = fn()
            if trec is not None:
                trec["dw"] = g
            put(p, lambda: g)
            return
        side.wait_stream(main)
        with torch.cuda.stream(side):
            g = fn()
            ev = torch.cuda.Event()
            ev.record(side)
        if trec is not None:
            trec["dw"] = g
        pending.append((p, g, ev, list(inputs)))

    dskip: Dict[int, torch.Tensor] = {}  # encoder level -> gradient view of the skip half of dcat
    dz2 = None
    for li in range(len(saved) - 1, -1, -1):
        if li < first_needed:
            break
        rec = saved[li]
        L = rec["L"]
        conv, norm = rec["conv"], rec["norm"]
        if L["kind"] == "enc" and L["last"] and L["stage"] < n - 1:
            dz2 = dskip.pop(L["stage"])
        else:
            dz2 = None
        dgd, dbd = dest(norm.weight), dest(norm.bias)
        if dgd is None or dbd is None:
            dgd = dbd = None
        # dgamma / dbeta (a 6 us reduction over the batch that dy does not depend on) leave the critical path: with the
        # side stream on, the norm backward stops after dy and the parameter sums run on the side stream
        defer = overlap and (wants(norm.weight) or wants(norm.bias))
        res = ops.in_backward(dz, dz2, rec["y"], rec["a"], rec["b"], rec["mean"], rec["rstd"], rec["scale"],
                              norm.weight, rec["slope"], out_dgamma=dgd, out_dbeta=dbd,
                              ext_part=ext_part if dz2 is None else None, defer_params=defer)
        ext_part = None
        rec_y = rec["y"]
        rec["y"] = None
        collect()  # the previous layer's weight gradient ran beside this norm backward
        if defer:
            dy, finish_params = res
            side.wait_stream(main)
            with torch.cuda.stream(side):
                dgamma, dbeta = finish_params()
                ev_p = torch.cuda.Event()
                ev_p.record(side)
            pending.append((norm.weight, dgamma, ev_p, [finish_params.keep]))
            pending.append((norm.bias, dbeta, ev_p, [finish_params.keep]))
        else:
            dy, dgamma, dbeta = res
            put(norm.weight, lambda: dgamma)
            put(norm.bias, lambda: dbeta)
        trec = None
        if btrace is not None:
            trec = dict(kind="unit", li=li, dz=dz, dz2=dz2, y=rec_y, dy=dy, dgamma=dgamma, dbeta=dbeta, xin=rec.get("xin"),
                        xin32=rec.get("xin32"))
            btrace.append(trec)
        # the conv bias feeds an InstanceNorm: its exact gradient is zero (SURVEY.md 8a)
        put(conv.bias, lambda: zero_grad_of(conv.bias))
        stride = rec["stride"]
        cin, cout = conv.in_channels, conv.out_channels
        simt = not _use_tc(cin, cout)
        if rec.get("stem") is True:
            if conv._backward_hooks:
                _fire_backward_hooks(conv, None, dy)
            xin32 = rec.get("xin32")
            if xin32 is None and ctx.image is None:  # uint8 batch on the narrow-image stem path
                from ..data import preprocess_batch
                ctx.image = preprocess_batch(ctx.image_u8, None, model.input_mean, model.input_std)[0]
            wgrad_async(conv.weight, lambda: ops.stem_wgrad_tc(ctx.image, dy, xin32, out=dest(conv.weight), channels=cin),
                        [ctx.image, dy, xin32], trec)
            break
        xin = rec["xin"]
        last = li == first_needed or rec.get("stem") is False
        dx = None
        if not last:
            wd = rec["wd"]
            ws2 = model._packs.s2(conv, wd) if (stride == 2 and not simt and wd.dtype == BF16) else None
            split_out = None
            if (L["kind"] == "dec" and L["idx"] == 0 and not simt and stride == 1 and dy.dtype == BF16
                    and cin == 96 and feats[n - 1 - L["stage"]] == 64 and model.split_concat_grad):
                # the gradient of a concat buffer whose pixel pitch is not a multiple of 128 bytes (level 0: 64 + 32
                # channels = 192 B) goes to two dense tensors: its consumers then read whole lines (see conv_dgrad_split)
                split_out = feats[n - 1 - L["stage"]]
            if ws2 is not None:
                dx = ops.conv_dgrad_s2(dy, ws2, (xin.shape[1], xin.shape[2]))
            elif split_out is not None:
                dx = ops.conv_dgrad_split(dy, wd, (xin.shape[1], xin.shape[2]), split_out)
            elif model.producer_sums_dgrad and L["idx"] > 0 and L["kind"] != "fusion" and li - 1 >= first_needed \
                    and saved[li - 1]["y"] is not None:
                # dx is the dz of the previous unit of the same block (no skip operand): the data gradient's epilogue can
                # reduce that unit's norm-backward sums where its kernel supports it (the 512^2 / 256^2 levels).  OFF by
                # default: measured a net loss there (DESIGN.md section 3, "tried and dropped") -- the narrow-output
                # kernels have no spare issue slots for ~8 instructions per element on a few epilogue warps
                prev = saved[li - 1]
                dx, ext_part = ops.conv_dgrad(dy, wd, (xin.shape[1], xin.shape[2]), stride, simt=simt,
                                              bwd_sums=(prev["y"], prev["a"], prev["b"], prev["slope"]))
            else:
                dx = ops.conv_dgrad(dy, wd, (xin.shape[1], xin.shape[2]), stride, simt=simt)
        if L["kind"] == "fusion":  # 1x1 weight = centre tap of the 3x3 gradient
            def fusion_dw():
                g = ops.conv_wgrad(xin, dy, stride, simt=simt)[:, :, 1:2, 1:2]
                if rec.get("cin_used") is None:
                    return g.contiguous()
                full = torch.zeros_like(conv.weight)  # the constant-feature half: exactly zero (cancelled by the norm)
                full[:, :rec["cin_used"]] = g
                return full
            wgrad_async(conv.weight, fusion_dw, [xin, dy], trec)
        else:
            wgrad_async(conv.weight, lambda: ops.conv_wgrad(xin, dy, stride, simt=simt, out=dest(conv.weight)), [xin, dy], trec)
        if trec is not None:
            trec["dx"] = torch.cat(dx, dim=-1) if isinstance(dx, tuple) else dx
        if conv._backward_hooks:
            _fire_backward_hooks(conv, torch.cat(dx, dim=-1) if isinstance(dx, tuple) else dx, dy)
        if last:
            break
        rec["xin"] = None
        if L["kind"] == "dec" and L["idx"] == 0:
            d = n - 2 - L["stage"]
            c_low = feats[d + 1]
            dup, dsk = dx if isinstance(dx, tuple) else (dx[..., :c_low], dx[..., c_low:])
            dskip[d] = dsk
            dz = ops.upsample2x_backward(dup)
            if btrace is not None:
                btrace.append(dict(kind="up", d=d, dout=dup, dx=dz))
        elif L["kind"] == "fusion":
            dz = dx[..., :feats[-1]]  # the extra features are inputs: their half of the gradient is dropped (if computed)
        else:
            dz = dx
    collect()
    if sink is not None and hasattr(sink, "finish"):
        sink.finish()
    ctx.saved = None
    ctx.cat = None
    ctx.z_last = None
    return grads


# ====================================================================================================================
# Stand-alone ConvBlock (NCHW fp32 boundary) -- used when a block is called outside UNet.forward
# ====================================================================================================================
class _BlockFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, block: ConvBlock, x, *params):
        ops.require_device()
        units = block.units()
        xin = ops.nchw_to_nhwc(x.detach().float().contiguous(),
                               out=_padded_nhwc(x.size(0), x.size(2), x.size(3), x.size(1), x.device))
        cur = xin
        recs = []
        need_grad = any(ctx.needs_input_grad)
        for conv, norm, act, drop in units:
            wf, wd = packs.build(conv.weight, packs.layout(conv, "conv"), need_grad)  # no pack store here
            y, stats = _conv_fwd(cur, wf, conv.stride[0])
            scale = None
            if drop is not None and block.training and drop.drop_prob > 0:
                scale = drop.draw(x, x.size(0), conv.out_channels).reshape(x.size(0), -1).float().contiguous()
            mean, rstd, a, b = ops.in_finalize(stats, norm.weight, norm.bias, scale, norm.eps, y.shape[1] * y.shape[2])
            z = ops.in_apply(y, a, b, act.negative_slope)
            recs.append(dict(xin=cur, y=y, wd=wd, mean=mean, rstd=rstd, a=a, b=b, scale=scale, conv=conv, norm=norm,
                             slope=act.negative_slope))
            cur = z
        ctx.recs = recs if need_grad else None
        ctx.x_needs = x.requires_grad
        ctx.params = params
        return ops.nhwc_to_nchw(cur)

    @staticmethod
    def backward(ctx, dout):
        recs = ctx.recs
        dz = ops.nchw_to_nhwc(dout.float().contiguous())
        pg = {}
        for i in range(len(recs) - 1, -1, -1):
            r = recs[i]
            conv, norm = r["conv"], r["norm"]
            dy, dg, db = ops.in_backward(dz, None, r["y"], r["a"], r["b"], r["mean"], r["rstd"], r["scale"], norm.weight,
                                         r["slope"])
            simt = not _use_tc(conv.in_channels, conv.out_channels)
            pg[id(norm.weight)], pg[id(norm.bias)] = dg, db
            pg[id(conv.weight)] = ops.conv_wgrad(r["xin"], dy, conv.stride[0], simt=simt)
            if conv.bias is not None:
                pg[id(conv.bias)] = torch.zeros_like(conv.bias)
            if i > 0 or ctx.x_needs:
                xin = r["xin"]
                dxp = _padded_nhwc(xin.shape[0], xin.shape[1], xin.shape[2], xin.shape[3], xin.device)
                dz = ops.conv_dgrad(dy, r["wd"], (xin.shape[1], xin.shape[2]), conv.stride[0], out=dxp, simt=simt)
        dx = ops.nhwc_to_nchw(dz) if ctx.x_needs else None
        return (None, dx) + tuple(pg.get(id(p)) if p.requires_grad else None for p in ctx.params)


class _UpsampleCatFunction(torch.autograd.Function):
    """cat([bilinear_2x(x), skip], 1) on NCHW fp32 tensors through the NHWC kernels (stand-alone UpBlock only)."""

    @staticmethod
    def forward(ctx, x, skip):
        ops.require_device()
        B, c_low, h, w = x.shape
        c_skip = skip.shape[1]
        if tuple(skip.shape[2:]) != (2 * h, 2 * w):
            raise NotImplementedError("b200unet: UpBlock implements the exact 2x case of F.interpolate (unet.py:220-225); "
                                      f"got {tuple(x.shape[2:])} -> {tuple(skip.shape[2:])}")
        if c_low % 8 or c_skip % 8:
            raise NotImplementedError("b200unet: UpBlock needs channel counts that are multiples of 8")
        with torch.cuda.device(x.device):
            cat = torch.empty((B, 2 * h, 2 * w, c_low + c_skip), dtype=BF16, device=x.device)
            xl = ops.nchw_to_nhwc(x.detach().float().contiguous())
            ops.upsample2x(xl, cat[..., :c_low])
            ops.nchw_to_nhwc(skip.detach().float().contiguous(), out=cat[..., c_low:])
            out = ops.nhwc_to_nchw(cat)
        ctx.c_low = c_low
        return out

    @staticmethod
    def backward(ctx, dout):
        c_low = ctx.c_low
        with torch.cuda.device(dout.device):
            d = ops.nchw_to_nhwc(dout.float().contiguous())
            dx = ops.nhwc_to_nchw(ops.upsample2x_backward(d[..., :c_low])) if ctx.needs_input_grad[0] else None
            dskip = dout[:, c_low:].float().contiguous() if ctx.needs_input_grad[1] else None
        return dx, dskip


def _run_block_standalone(block: ConvBlock, x: torch.Tensor):
    if not x.is_cuda:
        raise RuntimeError("b200unet: ConvBlock needs a CUDA tensor on an sm_100 device; there is no CPU path")
    return _BlockFunction.apply(block, x, *list(block.parameters()))
