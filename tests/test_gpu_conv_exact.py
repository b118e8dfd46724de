"""Bit-exact checks of every tensor-core convolution route with operands whose sums are exact.

The operands are small integers (regime A: values in {-2..2}) or such integers times a power of two per channel
(regime B: 2^e, e in [-3, 3]).  Every product and every partial sum is then a multiple of the finest product step
and stays far below 2^24 of those steps, so fp32 accumulation is exact in any order: the tiling, the split-K count, the
CTA-pair hand-over and the MMA order cannot change a bit.  A kernel's output must therefore equal the exact result
(float64 F.conv2d and its autograd, snapped to the value grid) at every element:
  - regime A: |y|, |dx| <= 256, so the stored bf16 output needs no rounding, and the epilogue's InstanceNorm partial sums
    (sum y, sum y^2 of the stored values, each below 2^24) are exact too;
  - regime B: the stored output is the exact value rounded to nearest even in bf16, which pins the epilogue's rounding
    mode, and a swapped channel differs by a scale factor.
Each test asserts these preconditions on its reference before it compares; a failed precondition is a test bug.

Outputs, statistics buffers and weight-gradient workspaces are filled with NaN before each call, so an element nobody
wrote, a statistics slot the call did not zero and a split partial nobody wrote all fail the comparison.  The route
table names the kernel instance each shape must reach; the launched kernels are recorded with torch.profiler.

The helpers and their CPU tests (operand generation, preconditions of every table case, assert_exact) run without a
GPU; everything else is marked gpu."""
import ctypes
import re
import zlib
from collections import Counter, namedtuple

import pytest
import torch
import torch.nn.functional as F

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
NAN = float("nan")
EXACT = 2 ** 24           # integers below this are exact in fp32
STEP = {"A": 1.0, "B": 2.0 ** -6}  # finest product step: B scales both operands of a product by 2^-3 at the least


# ------------------------------------------------------------------------------------------------------- operands
def int_operand(shape, density, gen, device="cpu"):
    """int8 tensor of values in {-2, -1, 1, 2} with probability `density`, else 0."""
    mag = torch.randint(1, 3, shape, generator=gen, device=device, dtype=torch.int8)
    neg = torch.rand(shape, generator=gen, device=device) < 0.5
    keep = torch.rand(shape, generator=gen, device=device) < density
    return torch.where(keep, torch.where(neg, -mag, mag), torch.zeros((), dtype=torch.int8, device=device))


def channel_scale(c, regime, gen, device="cpu"):
    """fp64 per-channel factor: 1 in regime A, 2^e with e in [-3, 3] in regime B."""
    if regime == "A":
        return torch.ones(c, dtype=F64, device=device)
    return torch.pow(2.0, torch.randint(-3, 4, (c,), generator=gen, device=device).to(F64))


def out_hw(h, w, stride):
    return (h - 1) // stride + 1, (w - 1) // stride + 1


def densities(op, cin, cout, oh, ow, d_w=0.5):
    """Operand densities that keep E[y^2] (fprop) / E[dx^2] (dgrad) near a target T: a nonzero product has E = 6.25, so
    E[y^2] ~ 9 Cin d_x d_w 6.25.  fprop's T also keeps every per-channel sum y^2 well below 2^24."""
    if op in ("wgrad", "stem"):
        return 0.5, d_w, 0.5
    t_f = min(128.0, 2.0 ** 22 / (oh * ow))
    d_x = min(1.0, t_f / (9 * cin * 6.25 * d_w))
    d_dy = min(1.0, 128.0 / (9 * cout * 6.25 * d_w))
    return d_x, d_w, d_dy


def make_operands(name, op, n, h, w, cin, cout, stride, regime, device="cpu", d_w=0.5, wmask=None, dymask=None):
    """x [N,H,W,Cin], w [Cout,Cin,3,3], dy [N,OH,OW,Cout] as float64 (values exact in bf16), plus the integer parts."""
    gen = torch.Generator(device=device).manual_seed(zlib.crc32(f"{name}/{regime}".encode()))
    oh, ow = out_hw(h, w, stride)
    d_x, d_w, d_dy = densities(op, cin, cout, oh, ow, d_w)
    xi = int_operand((n, h, w, cin), d_x, gen, device)
    wi = int_operand((cout, cin, 3, 3), d_w, gen, device)
    dyi = int_operand((n, oh, ow, cout), d_dy, gen, device)
    if wmask is not None:
        wi = wi * wmask.to(device=device, dtype=torch.int8)
    if dymask is not None:
        dyi = dyi * dymask.to(device=device, dtype=torch.int8)
    sx = channel_scale(cin, regime, gen, device)
    sw = channel_scale(cout, regime, gen, device)
    sdy = channel_scale(cout, regime, gen, device)
    return dict(xi=xi, wi=wi, dyi=dyi, x=xi.to(F64) * sx, w=wi.to(F64) * sw[:, None, None, None], dy=dyi.to(F64) * sdy,
                regime=regime, stride=stride)


# ------------------------------------------------------------------------------------------------ exact reference
def snap(t, step):
    """Round to the value grid and assert that this moved nothing by more than 1e-6 (the float64 result was exact)."""
    r = torch.round(t / step) * step
    moved = float((r - t).abs().max()) if t.numel() else 0.0
    assert moved <= 1e-6, f"reference is off the value grid by {moved}"
    return r


def ref_fprop(x, w, stride):
    return F.conv2d(x.permute(0, 3, 1, 2), w, stride=stride, padding=1).permute(0, 2, 3, 1)


def ref_dgrad(dy, w, in_hw, stride):
    n, _, _, _ = dy.shape
    size = (n, w.shape[1], in_hw[0], in_hw[1])
    return torch.nn.grad.conv2d_input(size, w, dy.permute(0, 3, 1, 2), stride=stride, padding=1).permute(0, 2, 3, 1)


def ref_wgrad(x, dy, wshape, stride):
    return torch.nn.grad.conv2d_weight(x.permute(0, 3, 1, 2), wshape, dy.permute(0, 3, 1, 2), stride=stride, padding=1)


def reference(op, o, in_hw):
    """The exact result of `op` on operands `o`, snapped to the grid."""
    step, s = STEP[o["regime"]], o["stride"]
    if op in ("fprop",):
        return snap(ref_fprop(o["x"], o["w"], s), step)
    if op in ("dgrad", "dgrad_s2", "dgrad_split", "dgrad_sums"):
        return snap(ref_dgrad(o["dy"], o["w"], in_hw, s), step)
    if op == "wgrad":
        return snap(ref_wgrad(o["x"], o["dy"], tuple(o["w"].shape), s), step)
    raise ValueError(op)


def stats_of(y):
    """Exact per-(image, channel) sum y and sum y^2 of an NHWC float64 tensor: [N, C, 2]."""
    return torch.stack([y.sum((1, 2)), (y * y).sum((1, 2))], -1)


def check_preconditions(op, o, ref, stats=False):
    """The conditions under which the kernel's result must equal `ref` bit for bit."""
    for k in ("x", "w", "dy"):
        assert torch.equal(o[k].to(BF16).to(F64), o[k]), f"{k} is not exact in bf16"
    regime = o["regime"]
    if op == "wgrad":
        # every |x dy| product sum of one weight element is at most max|x| * sum over pixels of |dy| of its channel
        bound = float(o["xi"].abs().max()) * float(o["dyi"].abs().to(F64).sum((0, 1, 2)).max())
        assert bound < EXACT, f"weight-gradient sums may reach {bound}"
        assert torch.equal(ref.float().to(F64), ref)
        return
    k = 9 * (o["x"].shape[-1] if op == "fprop" else o["dy"].shape[-1])
    if regime == "A":
        assert 4 * k < EXACT
        assert float(ref.abs().max()) <= 256, f"|out| reaches {float(ref.abs().max())}: not exact in bf16"
        if stats:
            assert float(stats_of(ref)[..., 1].max()) < EXACT, "sum y^2 is not exact in fp32"
    else:
        # sum of |products| in units of the finest step, for every output element
        xa, wa, dya = o["x"].abs(), o["w"].abs(), o["dy"].abs()
        s, step = o["stride"], STEP[regime]
        if op == "fprop":
            absum = ref_fprop(xa, wa, s)
        else:
            absum = ref_dgrad(dya, wa, tuple(o["x"].shape[1:3]), s)
        assert float(absum.max()) / step < EXACT, "partial sums may leave the fp32-exact range"
        assert torch.equal(ref.float().to(F64), ref), "exact result is not an fp32 value"


def rounding_share(ref):
    """Share of elements that bf16 cannot hold exactly (regime B must exercise the rounding)."""
    return float((ref.to(BF16).to(F64) != ref).to(F64).mean())


def assert_exact(got, ref, what="output"):
    """Bitwise equality of a kernel result with the exact reference (NaN in `got`, an unwritten sentinel, fails)."""
    got = got.detach()
    ref = ref.detach().to(device=got.device, dtype=got.dtype)
    assert got.shape == ref.shape, f"{what}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    bad = got != ref
    if not bool(bad.any()):
        return
    idx = bad.nonzero()
    first = [tuple(int(v) for v in i) for i in idx[:6].cpu()]
    vals = [(float(got[c]), float(ref[c])) for c in first]
    axes = "(n, h, w, c)" if got.dim() == 4 and not what.startswith("dw") else "index"
    raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ; first {axes}: "
                         + ", ".join(f"{c} got {g!r} want {r!r}" for c, (g, r) in zip(first, vals)))


# ---------------------------------------------------------------------------------------------------- route table
Route = namedtuple("Route", "name op n h w cin cout stride layout expect")

# Every (operation, shape) below reaches the listed kernel instances with the default settings on a 148-SM B200.
# "k*4" means instance k launched four times.  dgrad_s2 is the parity-stacked stride-2 data gradient
# (pack_s2_dgrad_weights + conv_dgrad_s2); dgrad_split writes channels [0, 64) and the rest as two dense tensors;
# "pitched" reads and writes channel slices of wider buffers.
ROUTES = [
    # dispatch_gconv: the split-output instances (parity classes stacked on N, Cin 32)
    Route("s2_bk64", "dgrad_s2", 2, 16, 32, 32, 64, 2, "dense",
          ("pack_s2_dgrad_weights_kernel", "gconv_kernel<64,128,4,4,false,32,1,1>")),
    Route("s2_bk32_pitched_odd", "dgrad_s2", 1, 13, 21, 32, 96, 2, "pitched",
          ("pack_s2_dgrad_weights_kernel", "gconv_kernel<32,128,8,4,false,32,1,1>")),
    Route("s2_cin64", "dgrad_s2", 2, 18, 10, 64, 128, 2, "dense",
          ("pack_s2_dgrad_weights_kernel", "gconv_kernel<64,256,2,4,false,0,1,1>")),
    Route("s2_cin64_bk32_pitched_odd", "dgrad_s2", 1, 7, 9, 64, 96, 2, "pitched",
          ("pack_s2_dgrad_weights_kernel", "gconv_kernel<32,256,4,4,false,0,1,1>")),
    # CTA pairs: an even tile count per image and more pair tiles than half the SMs; ragged in both directions
    Route("pair_bn256", "fprop", 1, 150, 124, 128, 256, 1, "dense", ("gconv_kernel<64,256,3,6,false,0,1,2>",)),
    Route("pair_bn192", "dgrad", 1, 150, 124, 192, 128, 1, "dense", ("gconv_kernel<64,192,3,8,false,0,1,2>",)),
    Route("pair_bn128_mt2", "fprop", 2, 150, 124, 128, 128, 1, "dense", ("gconv_kernel<64,128,2,8,false,0,2,2>",)),
    Route("pair_bn64_mt4", "fprop", 2, 300, 124, 128, 64, 1, "dense", ("gconv_kernel<64,64,2,6,false,0,4,2>",)),
    # 40 pair tiles: single CTAs on 148 SMs, CTA pairs once half the SMs are fewer than 40
    Route("pair_threshold", "fprop", 1, 160, 64, 128, 256, 1, "dense", ("gconv_kernel<64,256,2,4,false,0,1,1>",)),
    # single-CTA multi-M-tile forms
    Route("mt2", "fprop", 1, 20, 13, 128, 128, 1, "dense", ("gconv_kernel<64,128,2,6,false,0,2,1>",)),
    Route("mt4", "fprop", 2, 21, 19, 128, 64, 1, "dense", ("gconv_kernel<64,64,2,3,false,0,4,1>",)),
    Route("mt2_pitched", "dgrad", 1, 19, 23, 128, 128, 1, "pitched", ("gconv_kernel<64,128,2,6,false,0,2,1>",)),
    # one line per GC(...) instance
    Route("gc_64_256", "fprop", 1, 8, 16, 256, 256, 1, "dense", ("gconv_kernel<64,256,2,4,false,0,1,1>",)),
    Route("gc_64_192", "dgrad", 1, 16, 16, 192, 64, 1, "dense", ("gconv_kernel<64,192,3,4,false,0,1,1>",)),
    Route("gc_64_64_res", "fprop", 2, 13, 21, 64, 64, 1, "dense", ("gconv_kernel<64,64,4,1,true,0,1,1>",)),
    Route("gc_64_64_res_pitched", "fprop", 1, 11, 30, 64, 64, 1, "pitched", ("gconv_kernel<64,64,4,1,true,0,1,1>",)),
    Route("gc_64_32", "fprop", 2, 13, 21, 64, 96, 2, "dense", ("gconv_kernel<64,32,8,4,false,0,1,1>",)),
    Route("gc_64_32_res", "fprop", 1, 11, 37, 64, 32, 1, "dense", ("gconv_kernel<64,32,4,1,true,0,1,1>",)),
    Route("gc_32_256", "fprop", 1, 9, 12, 96, 256, 1, "dense", ("gconv_kernel<32,256,4,4,false,0,1,1>",)),
    Route("gc_32_128", "fprop", 1, 13, 21, 32, 128, 2, "dense", ("gconv_kernel<32,128,8,4,false,0,1,1>",)),
    Route("gc_32_96", "fprop", 1, 9, 11, 96, 96, 2, "dense", ("gconv_kernel<32,96,8,4,false,0,1,1>",)),
    Route("gc_32_96_res", "fprop", 1, 13, 21, 32, 96, 2, "dense", ("gconv_kernel<32,96,8,1,true,0,1,1>",)),
    Route("gc_32_64", "fprop", 1, 10, 14, 96, 64, 2, "dense", ("gconv_kernel<32,64,8,4,false,0,1,1>",)),
    Route("gc_32_64_res", "fprop", 2, 16, 16, 32, 64, 2, "dense", ("gconv_kernel<32,64,8,1,true,0,1,1>",)),
    Route("gc_32_32", "fprop", 1, 9, 20, 160, 32, 1, "dense", ("gconv_kernel<32,32,8,4,false,0,1,1>",)),
    Route("gc_32_32_res", "fprop", 1, 5, 7, 32, 32, 1, "dense", ("gconv_kernel<32,32,8,1,true,0,1,1>",)),
    # stride-2 data gradient of a Cin >= 128 conv: one launch per parity class of the input pixel
    Route("dgrad_s2_four_launches", "dgrad", 1, 15, 17, 128, 256, 2, "dense",
          ("gconv_kernel<64,128,2,6,false,0,2,1>*4",)),
    # nconv_kernel: BK 64/32 x CO 64/32, forward and data gradient
    Route("nconv_64_64_f", "fprop", 2, 8, 96, 64, 64, 1, "dense", ("nconv_kernel<64,64,4,false,2>",)),
    Route("nconv_64_64_d", "dgrad", 2, 8, 96, 64, 64, 1, "dense", ("nconv_kernel<64,64,4,true,2>",)),
    Route("nconv_64_64_f_pitched", "fprop", 1, 7, 70, 64, 64, 1, "pitched", ("nconv_kernel<64,64,4,false,2>",)),
    Route("nconv_64_32_f", "fprop", 1, 6, 121, 64, 32, 1, "dense", ("nconv_kernel<64,32,4,false,2>",)),
    Route("nconv_64_32_f_ktail", "fprop", 1, 9, 64, 96, 32, 1, "dense", ("nconv_kernel<64,32,4,false,2>",)),
    Route("nconv_64_32_d", "dgrad", 1, 7, 90, 32, 64, 1, "dense", ("nconv_kernel<64,32,4,true,2>",)),
    Route("nconv_32_64_f", "fprop", 1, 7, 90, 32, 64, 1, "dense", ("nconv_kernel<32,64,8,false,2>",)),
    Route("nconv_32_64_d", "dgrad", 1, 6, 121, 64, 32, 1, "dense", ("nconv_kernel<32,64,8,true,2>",)),
    Route("nconv_32_32_f", "fprop", 1, 12, 70, 32, 32, 1, "dense", ("nconv_kernel<32,32,8,false,2>",)),
    Route("nconv_32_32_d", "dgrad", 1, 12, 70, 32, 32, 1, "dense", ("nconv_kernel<32,32,8,true,2>",)),
    Route("nconv_32_32_f_pitched", "fprop", 1, 8, 136, 32, 32, 1, "pitched", ("nconv_kernel<32,32,8,false,2>",)),
    Route("nconv_32_32_d_oddw", "dgrad", 1, 6, 129, 32, 32, 1, "dense", ("nconv_kernel<32,32,8,true,2>",)),
    # pconv_kernel: dense 32 -> 32, even width >= 128
    Route("pconv_f", "fprop", 1, 12, 128, 32, 32, 1, "dense", ("pconv_kernel<false>",)),
    Route("pconv_f_ragged", "fprop", 2, 9, 190, 32, 32, 1, "dense", ("pconv_kernel<false>",)),
    Route("pconv_d", "dgrad", 1, 12, 128, 32, 32, 1, "dense", ("pconv_kernel<true>",)),
    Route("pconv_d_ragged", "dgrad", 3, 5, 250, 32, 32, 1, "dense", ("pconv_kernel<true>",)),
    # wgrad_kernel: U x BN
    Route("wg_64_256", "wgrad", 1, 8, 16, 256, 256, 1, "dense", ("wgrad_kernel<64,256>",)),
    Route("wg_64_128", "wgrad", 1, 16, 16, 64, 128, 2, "dense", ("wgrad_kernel<64,128>",)),
    Route("wg_64_64", "wgrad", 1, 13, 21, 64, 64, 2, "dense", ("wgrad_kernel<64,64>",)),
    Route("wg_64_32", "wgrad", 2, 13, 21, 64, 96, 2, "dense", ("wgrad_kernel<64,32>",)),
    Route("wg_32_256", "wgrad", 1, 9, 11, 32, 256, 2, "dense", ("wgrad_kernel<32,256>",)),
    Route("wg_32_128", "wgrad", 1, 16, 16, 32, 128, 2, "pitched", ("wgrad_kernel<32,128>",)),
    Route("wg_32_64_splits", "wgrad", 2, 32, 64, 32, 64, 2, "dense",
          ("wgrad_kernel<32,64>", "wgrad_finalize_splits_kernel")),
    Route("wg_32_32", "wgrad", 1, 7, 9, 32, 32, 2, "dense", ("wgrad_kernel<32,32>",)),
    # 6 CTAs per split: S = 24 on 148 SMs (splits finalize), 12 on 75 (tiled finalize)
    Route("wg_splits_threshold", "wgrad", 1, 64, 48, 64, 384, 1, "dense",
          ("wgrad_kernel<64,128>", "wgrad_finalize_splits_kernel")),
    Route("wg_tiled", "wgrad", 1, 16, 16, 1024, 512, 1, "dense",
          ("wgrad_kernel<64,256>", "wgrad_finalize_tiled_kernel")),
    # wgradn_kernel
    Route("wgn_32_32", "wgrad", 1, 9, 64, 96, 32, 1, "dense", ("wgradn_kernel<32,32,0>",)),
    Route("wgn_32_32_oddw", "wgrad", 1, 6, 129, 32, 32, 1, "dense", ("wgradn_kernel<32,32,0>",)),
    Route("wgn_32_32_pitched", "wgrad", 1, 8, 136, 32, 32, 1, "pitched", ("wgradn_kernel<32,32,0>",)),
    Route("wgn_32_64", "wgrad", 1, 7, 90, 32, 64, 1, "dense", ("wgradn_kernel<32,64,0>",)),
    Route("wgn_64_32", "wgrad", 1, 6, 121, 64, 32, 1, "dense", ("wgradn_kernel<64,32,0>",)),
    Route("wgn_64_32_splits", "wgrad", 2, 40, 96, 64, 32, 1, "dense",
          ("wgradn_kernel<64,32,0>", "wgrad_finalize_splits_kernel")),
    Route("wgn_64_64", "wgrad", 2, 8, 96, 64, 64, 1, "dense", ("wgradn_kernel<64,64,1>",)),
    Route("wgn_pairs", "wgrad", 1, 12, 128, 32, 32, 1, "dense",
          ("wgradn_kernel<64,64,2>", "wgrad_finalize_pairs_window_kernel")),
    Route("wgn_pairs_ragged", "wgrad", 2, 9, 190, 32, 32, 1, "dense",
          ("wgradn_kernel<64,64,2>", "wgrad_finalize_pairs_window_kernel")),
    # the data gradient of a concat buffer written as two dense tensors
    Route("split_bk32", "dgrad_split", 2, 24, 40, 96, 32, 1, "dense", ("gconv_kernel<32,96,8,1,true,0,1,1>",)),
    Route("split_bk32_ragged", "dgrad_split", 1, 13, 21, 96, 32, 1, "dense", ("gconv_kernel<32,96,8,1,true,0,1,1>",)),
    Route("split_bk64", "dgrad_split", 1, 21, 26, 128, 64, 1, "dense", ("gconv_kernel<64,128,2,6,false,0,2,1>",)),
    # producer-side norm-backward sums in the narrow data-gradient kernels
    Route("sums_pconv", "dgrad_sums", 1, 9, 128, 32, 32, 1, "dense", ("pconv_kernel<true>",)),
    Route("sums_nconv_32", "dgrad_sums", 1, 7, 131, 32, 32, 1, "dense", ("nconv_kernel<32,32,8,true,2>",)),
    Route("sums_nconv_64", "dgrad_sums", 2, 21, 70, 64, 64, 1, "dense", ("nconv_kernel<64,64,4,true,2>",)),
]
ROUTE_IDS = [r.name for r in ROUTES]

# Every conv kernel instance the library compiles, and those no argument set reaches with the default settings.
ALL_INSTANCES = {
    *(f"gconv_kernel<{a}>" for a in (
        "32,128,8,4,false,0,1,1", "32,128,8,4,false,32,1,1", "32,256,4,4,false,0,1,1", "32,32,8,1,true,0,1,1",
        "32,32,8,4,false,0,1,1", "32,64,8,1,true,0,1,1", "32,64,8,4,false,0,1,1", "32,96,8,1,true,0,1,1",
        "32,96,8,4,false,0,1,1", "64,128,2,6,false,0,2,1", "64,128,2,8,false,0,2,2", "64,128,4,4,false,0,1,1",
        "64,128,4,4,false,32,1,1", "64,192,3,4,false,0,1,1", "64,192,3,8,false,0,1,2", "64,256,2,4,false,0,1,1",
        "64,256,3,6,false,0,1,2", "64,32,4,1,true,0,1,1", "64,32,8,4,false,0,1,1", "64,64,2,3,false,0,4,1",
        "64,64,2,6,false,0,4,2", "64,64,4,1,true,0,1,1", "64,64,6,4,false,0,1,1")),
    *(f"nconv_kernel<{bk},{co},{8 if bk == 32 else 4},{rev},2>" for bk in (32, 64) for co in (32, 64)
      for rev in ("false", "true")),
    "pconv_kernel<false>", "pconv_kernel<true>",
    *(f"wgrad_kernel<{u},{bn}>" for u in (32, 64) for bn in (32, 64, 128, 256)),
    "wgradn_kernel<32,32,0>", "wgradn_kernel<32,64,0>", "wgradn_kernel<64,32,0>", "wgradn_kernel<64,64,0>",
    "wgradn_kernel<64,64,1>", "wgradn_kernel<64,64,2>",
    "wgrad_finalize_kernel", "wgrad_finalize_tiled_kernel", "wgrad_finalize_splits_kernel", "wgrad_finalize_pairs_kernel",
    "wgrad_finalize_pairs_window_kernel", "pack_s2_dgrad_weights_kernel",
}
UNREACHABLE = {
    "gconv_kernel<64,128,4,4,false,0,1,1>":
        "GC(64, 128, 4, 4, false) needs one M tile, but pick_mt gives every BK 64 / BN 128 launch two; the only "
        "one-M-tile launcher with BN 128 (conv_dgrad_s2, Cin 32) takes the split-output instance first",
    "gconv_kernel<64,64,6,4,false,0,1,1>":
        "GC(64, 64, 6, 4, false) needs one M tile, but pick_mt gives every streamed-weight BK 64 / BN 64 launch four",
    "wgradn_kernel<64,64,0>": "only with the developer switches B200UNET_WGRAD_ONEDY=0 or B200UNET_WGRAD_PAIRS=1",
    "wgrad_finalize_pairs_kernel": "only with the developer switch B200UNET_WGRAD_PAIRS=1",
    "wgrad_finalize_kernel":
        "launch_wgrad_finalize takes the splits or tiled form whenever Cout % 32 == 0 and Cin % 8 == 0, which the "
        "tensor-core envelope (channels in multiples of 32) always satisfies",
}


def expected_counts(route):
    out = Counter()
    for e in route.expect:
        k, _, times = e.partition("*")
        out[k] += int(times or 1)
    return out


# ------------------------------------------------------------------------------------------------- CPU-side tests
@pytest.mark.parametrize("regime", ["A", "B"])
def test_operands_are_exact_in_bf16(regime):
    o = make_operands("probe", "fprop", 2, 9, 11, 64, 96, 1, regime)
    for k in ("x", "w", "dy"):
        assert torch.equal(o[k].to(BF16).to(F64), o[k]) and torch.equal(o[k].float().to(F64), o[k])
    assert set(torch.unique(o["xi"]).tolist()) <= {-2, -1, 0, 1, 2}
    scales = (o["x"][o["xi"] != 0] / o["xi"][o["xi"] != 0].to(F64)).abs()
    want = {1.0} if regime == "A" else {2.0 ** e for e in range(-3, 4)}
    assert set(scales.unique().tolist()) <= want
    if regime == "B":
        assert len(set(scales.unique().tolist())) > 1


@pytest.mark.parametrize("regime", ["A", "B"])
@pytest.mark.parametrize("route", ROUTES, ids=ROUTE_IDS)
def test_preconditions_hold_for_every_route(route, regime):
    o = make_operands(route.name, route.op, route.n, route.h, route.w, route.cin, route.cout, route.stride, regime)
    ref = reference(route.op, o, (route.h, route.w))
    check_preconditions(route.op, o, ref, stats=route.op == "fprop" and regime == "A")
    if regime == "B" and route.op != "wgrad":
        assert rounding_share(ref) >= 0.01, "regime B would not exercise the epilogue's rounding"
    if route.op == "dgrad_sums" and regime == "A":
        sums_reference(o, ref)  # asserts its own exactness conditions


def test_preconditions_hold_for_the_pdl_chain():
    o = chain_operands("cpu")
    chain_reference(o)


@pytest.mark.parametrize("case", ["simt", "f32"])
def test_preconditions_hold_for_the_direct_kernels(case):
    for shape in DIRECT_SHAPES:
        for regime in ("A", "B"):
            for op in ("fprop", "dgrad", "wgrad"):
                o = make_operands(f"{case}/{shape}/{op}", op, *shape, regime)
                check_preconditions(op, o, reference(op, o, shape[1:3]), stats=op == "fprop" and regime == "A")


def test_assert_exact_catches_one_wrong_element():
    ref = torch.arange(-60, 60, dtype=F64).reshape(1, 2, 3, 20) * 1.5
    got = ref.to(BF16)
    assert_exact(got, ref)
    for change in ("ulp_up", "ulp_down", "nan", "sign"):
        bad = got.clone()
        flat = bad.view(-1)
        i = 77
        bits = flat.view(torch.int16)
        if change == "ulp_up":
            bits[i] += 1
        elif change == "ulp_down":
            bits[i] -= 1
        elif change == "nan":
            flat[i] = NAN
        else:
            flat[i] = -flat[i]
        assert float((bad.to(F64) - ref).abs().max()) > 0 or change == "nan"
        with pytest.raises(AssertionError, match=r"1 of 120 elements differ; first \(n, h, w, c\): \(0, 1, 0, 17\)"):
            assert_exact(bad, ref)
    dw = torch.zeros(4, 3, 3, 3)
    dw_bad = dw.clone()
    dw_bad[2, 1, 0, 2] = 2.0 ** -149  # the smallest fp32 step
    with pytest.raises(AssertionError, match=r"dw: 1 of 108 .*index: \(2, 1, 0, 2\)"):
        assert_exact(dw_bad, dw, "dw")


def test_route_table_covers_every_reachable_instance():
    covered = set()
    for r in ROUTES:
        covered |= set(expected_counts(r))
    assert not (covered & set(UNREACHABLE)), "a route lists an instance marked unreachable"
    assert set(UNREACHABLE) <= ALL_INSTANCES
    missing = ALL_INSTANCES - set(UNREACHABLE) - covered
    assert not missing, f"no route reaches {sorted(missing)}"
    assert covered <= ALL_INSTANCES, sorted(covered - ALL_INSTANCES)


def test_kernel_key_reads_demangled_profiler_names():
    assert kernel_key("void b200::gconv_kernel<64, 128, 2, 6, false, 0, 2, 1>(b200::GConvMaps, b200::GConvParams)") == \
        "gconv_kernel<64,128,2,6,false,0,2,1>"
    assert kernel_key("b200::wgrad_finalize_splits_kernel(float const*, float*, int, int, int)") == \
        "wgrad_finalize_splits_kernel"
    assert kernel_key("pack_s2_dgrad_weights_kernel(__nv_bfloat16 const*, __nv_bfloat16*, int, int)") == \
        "pack_s2_dgrad_weights_kernel"
    assert kernel_key("Memset (Device)") is None


# ------------------------------------------------------------------------------------------------- GPU harness
def kernel_key(name):
    """'void b200::gconv_kernel<64, 128, ...>(...)' -> 'gconv_kernel<64,128,...>'; None for a name without one."""
    m = re.search(r"([A-Za-z_]\w*_kernel(?:<[^<>()]*>)?)\(", re.sub(r"\s+", "", name))
    return m.group(1) if m else None


def launched(fn):
    """Run fn() under torch.profiler (CUDA activity); returns (fn's result, Counter of launched kernel keys)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    keys = Counter(k for k in map(kernel_key, names) if k)
    if not keys:
        kr = getattr(prof.profiler, "kineto_results", None)
        raw = [e.name() for e in kr.events()] if kr is not None else []
        keys = Counter(k for k in map(kernel_key, raw) if k)
        names += raw
    assert keys, f"the profiler recorded no kernel names (events: {names[:20]})"
    return out, keys


def _ops():
    from unet_implementations_b200 import _lib, ops
    ops.require_device()
    return _lib, ops


def place(t, layout):
    """A CUDA view of t: dense, or channels [8, 8 + C) of a buffer 16 channels wider."""
    if layout == "dense":
        return t.contiguous()
    n, h, w, c = t.shape
    buf = torch.full((n, h, w, c + 16), NAN, dtype=t.dtype, device=t.device)
    buf[..., 8:8 + c] = t
    return buf[..., 8:8 + c]


def nan_out(shape, layout, dtype=BF16):
    """(buffer, view) of NaN: dense, or channels [16, 16 + C) of a buffer 24 channels wider."""
    n, h, w, c = shape
    if layout == "dense":
        buf = torch.full(shape, NAN, dtype=dtype, device="cuda")
        return buf, buf
    buf = torch.full((n, h, w, c + 24), NAN, dtype=dtype, device="cuda")
    return buf, buf[..., 16:16 + c]


def assert_margins_untouched(buf, view):
    if buf is view:
        return
    c0 = view.data_ptr() - buf.data_ptr()
    c0 //= buf.element_size()
    c = view.shape[-1]
    assert bool(torch.isnan(buf[..., :c0]).all()) and bool(torch.isnan(buf[..., c0 + c:]).all()), \
        "a kernel wrote outside its channel slice"


def fprop_stats_buffer(x, cout, stride, simt=False):
    """NaN-filled [N, P, Cout, 2] statistics buffer of the fprop entry point that runs for x."""
    _lib, _ = _ops()
    n, h, w, _ = x.shape
    oh, ow = out_hw(h, w, stride)
    direct = simt or x.dtype == F32
    parts = _lib.call("b200unet_conv_fprop_simt_partials", oh, ow) if direct else \
        _lib.call("b200unet_conv_fprop_partials", n, oh, ow, cout)
    assert parts > 0
    return torch.full((n, parts, cout, 2), NAN, dtype=F32, device="cuda")


def launch_fprop(x, wf, stride, y, stats, simt=False):
    """conv_fprop through the C ABI into caller-owned buffers (stats may be None); enqueues nothing else."""
    _lib, ops = _ops()
    n, h, w, cin = x.shape
    cout = wf.shape[0]
    a = _lib.ConvFpropArgs(ops._p(x), ops.pitch_of(x), ops._p(wf), ops._p(y), ops.pitch_of(y), ops._p(stats), n, h, w,
                           cin, cout, stride)
    name = "b200unet_conv_fprop_f32" if x.dtype == F32 else ("b200unet_conv_fprop_simt" if simt else "b200unet_conv_fprop")
    _lib.call(name, ctypes.byref(a), ops._stream())


def run_fprop(x, wf, stride, y, simt=False):
    """conv_fprop with a NaN-filled statistics buffer; returns the statistics."""
    stats = fprop_stats_buffer(x, wf.shape[0], stride, simt)
    launch_fprop(x, wf, stride, y, stats, simt)
    return stats


def wgrad_buffers(x, dy, stride, simt=False):
    """NaN-filled dw [Cout, Cin, 3, 3] and split-K workspace (None for the direct kernels) of a weight gradient."""
    _lib, _ = _ops()
    n, h, w, cin = x.shape
    cout = dy.shape[3]
    dw = torch.full((cout, cin, 3, 3), NAN, dtype=F32, device="cuda")
    if simt or x.dtype == F32:
        return dw, None
    nbytes = _lib.call("b200unet_conv_wgrad_workspace", n, h, w, cin, cout, stride)
    assert nbytes >= 0, _lib.last_error()
    return dw, torch.full((max(nbytes, 4) // 4,), NAN, dtype=F32, device="cuda")


def launch_wgrad(x, dy, stride, dw, ws, simt=False):
    """conv_wgrad through the C ABI into caller-owned buffers; enqueues nothing else."""
    _lib, ops = _ops()
    n, h, w, cin = x.shape
    cout = dy.shape[3]
    if simt or x.dtype == F32:
        a = _lib.ConvWgradArgs(ops._p(x), ops.pitch_of(x), ops._p(dy), ops.pitch_of(dy), ops._p(dw), None, 0, n, h, w,
                               cin, cout, stride)
        _lib.call("b200unet_conv_wgrad_f32" if x.dtype == F32 else "b200unet_conv_wgrad_simt", ctypes.byref(a),
                  ops._stream())
        return
    a = _lib.ConvWgradArgs(ops._p(x), ops.pitch_of(x), ops._p(dy), ops.pitch_of(dy), ops._p(dw), ops._p(ws),
                           ws.numel() * 4, n, h, w, cin, cout, stride)
    _lib.call("b200unet_conv_wgrad", ctypes.byref(a), ops._stream())


def run_wgrad(x, dy, stride, simt=False):
    """conv_wgrad with NaN-filled dw and workspace; returns dw."""
    dw, ws = wgrad_buffers(x, dy, stride, simt)
    launch_wgrad(x, dy, stride, dw, ws, simt)
    return dw


def sums_operands(o):
    """y, a, b of the unit whose dz the data gradient is: y integer, a in {+-1/2, +-1, +-2}, b an odd multiple of 1/4,
    so a*y + b is never 0 and every term of T1 = sum gm, T2 = sum gm*y (gm = dx * lrelu'(a*y + b), slope 1/4) is exact."""
    n, h, w, cin = o["x"].shape
    gen = torch.Generator().manual_seed(7)
    y = int_operand((n, h, w, cin), 0.7, gen).to(F64)
    a = torch.tensor([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0], dtype=F64)[torch.randint(0, 6, (n, cin), generator=gen)]
    b = torch.tensor([-0.75, -0.25, 0.25, 0.75], dtype=F64)[torch.randint(0, 4, (n, cin), generator=gen)]
    return y, a, b


def sums_reference(o, dx_ref):
    y, a, b = sums_operands(o)
    y, a, b = y.to(dx_ref.device), a.to(dx_ref.device), b.to(dx_ref.device)
    pre = y * a[:, None, None, :] + b[:, None, None, :]
    assert bool((pre != 0).all())
    gm = dx_ref * torch.where(pre > 0, 1.0, 0.25)
    t = stats_of_pair(gm, y)
    bound = torch.stack([gm.abs().sum((1, 2)), (gm * y).abs().sum((1, 2))], -1)
    assert float(bound.max()) * 4 < EXACT, "norm-backward sums leave the fp32-exact range"
    return t


def stats_of_pair(gm, y):
    return torch.stack([gm.sum((1, 2)), (gm * y).sum((1, 2))], -1)


def to_cuda(o):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in o.items()}


_CACHE = {}


@pytest.fixture(scope="module", autouse=True)
def _release_cached_operands():
    """The cached float64 operands and references live for this module only."""
    yield
    _CACHE.clear()
    _DEFAULT_KEYS.clear()


def prepared(route, regime):
    """Operands (CUDA) and the exact reference of a route, computed once per module."""
    key = (route.name, regime)
    if key not in _CACHE:
        o = to_cuda(make_operands(route.name, route.op, route.n, route.h, route.w, route.cin, route.cout, route.stride,
                                  regime))
        ref = reference(route.op, o, (route.h, route.w))
        stats = route.op == "fprop" and regime == "A"
        check_preconditions(route.op, o, ref, stats=stats)
        extra = stats_of(ref) if stats else None
        if route.op == "dgrad_sums" and regime == "A":
            extra = sums_reference(o, ref)  # in regime B only dx is exact
        _CACHE[key] = (o, ref, extra)
    return _CACHE[key]


def run_route(route, regime):
    """Run the route's operation on fresh NaN-filled outputs and check every result bit for bit."""
    _lib, ops = _ops()
    o, ref, extra = prepared(route, regime)
    n, h, w, cin, cout, s = route.n, route.h, route.w, route.cin, route.cout, route.stride
    lay = route.layout
    wf, wd = ops.pack_conv_weights(o["w"].float())
    oh, ow = out_hw(h, w, s)
    if route.op == "fprop":
        x = place(o["x"].to(BF16), lay)
        buf, y = nan_out((n, oh, ow, cout), lay)
        stats = run_fprop(x, wf, s, y)
        torch.cuda.synchronize()
        want = ref.to(BF16) if regime == "B" else ref
        assert_exact(y, want, "y")
        assert_margins_untouched(buf, y)
        if extra is not None:
            assert_exact(stats.to(F64).sum(1), extra, "stats")
        return
    if route.op == "wgrad":
        dw = run_wgrad(place(o["x"].to(BF16), lay), place(o["dy"].to(BF16), lay), s)
        torch.cuda.synchronize()
        assert_exact(dw, ref, "dw")
        return
    dy = place(o["dy"].to(BF16), lay)
    want = ref.to(BF16) if regime == "B" else ref
    if route.op == "dgrad":
        buf, dx = nan_out((n, h, w, cin), lay)
        ops.conv_dgrad(dy, wd, (h, w), s, out=dx)
        torch.cuda.synchronize()
        assert_exact(dx, want, "dx")
        assert_margins_untouched(buf, dx)
    elif route.op == "dgrad_s2":
        ws2 = ops.pack_s2_dgrad_weights(wd)
        assert ws2 is not None
        buf, dx = nan_out((n, h, w, cin), lay)
        ops.conv_dgrad_s2(dy, ws2, (h, w), out=dx)
        torch.cuda.synchronize()
        assert_exact(dx, want, "dx")
        assert_margins_untouched(buf, dx)
    elif route.op == "dgrad_split":
        split = 64
        d1 = torch.full((n, h, w, split), NAN, dtype=BF16, device="cuda")
        d2 = torch.full((n, h, w, cin - split), NAN, dtype=BF16, device="cuda")
        a = _lib.ConvDgradArgs(ops._p(dy), ops.pitch_of(dy), ops._p(wd), ops._p(d1), ops.pitch_of(d1), n, h, w, cin,
                               cout, 1)
        a.dx2, a.dx2_pitch, a.dx_split = d2.data_ptr(), ops.pitch_of(d2), split
        _lib.call("b200unet_conv_dgrad", ctypes.byref(a), ops._stream())
        torch.cuda.synchronize()
        assert_exact(d1, want[..., :split], "dx[..., :split]")
        assert_exact(d2, want[..., split:], "dx[..., split:]")
    elif route.op == "dgrad_sums":
        y, sa, sb = (t.cuda() for t in sums_operands(o))
        yb = y.to(BF16).contiguous()
        sa, sb = sa.float().contiguous(), sb.float().contiguous()
        slots = _lib.call("b200unet_conv_dgrad_bwd_slots", n, h, w, cin, cout, 1)
        assert slots > 0, "this shape is expected on a kernel that produces the sums"
        part = torch.full((n, slots, cin, 2), NAN, dtype=F32, device="cuda")
        dx = torch.full((n, h, w, cin), NAN, dtype=BF16, device="cuda")
        a = _lib.ConvDgradArgs(ops._p(dy), ops.pitch_of(dy), ops._p(wd), ops._p(dx), ops.pitch_of(dx), n, h, w, cin,
                               cout, 1)
        a.bs_y, a.bs_y_pitch, a.bs_a, a.bs_b = yb.data_ptr(), ops.pitch_of(yb), sa.data_ptr(), sb.data_ptr()
        a.bs_slope, a.bs_part = 0.25, part.data_ptr()
        _lib.call("b200unet_conv_dgrad", ctypes.byref(a), ops._stream())
        torch.cuda.synchronize()
        assert_exact(dx, want, "dx")
        if extra is not None:
            assert_exact(part.to(F64).sum(1), extra, "norm-backward sums")
    else:
        raise ValueError(route.op)


_DEFAULT_KEYS = {}


def route_kernels(route):
    """Run a route in regime A under the profiler; the reference is computed first, outside the profiled region."""
    prepared(route, "A")
    out, keys = launched(lambda: run_route(route, "A"))
    return out, Counter({k: v for k, v in keys.items() if k in ALL_INSTANCES})


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, ids=ROUTE_IDS)
def test_route_reaches_its_kernel_and_is_exact(route):
    _, keys = route_kernels(route)
    _DEFAULT_KEYS[route.name] = keys
    for k, times in expected_counts(route).items():
        assert keys[k] >= times, f"{route.name}: expected {k} x{times}; launched {dict(keys)}"


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, ids=ROUTE_IDS)
def test_route_rounds_to_nearest_even_with_dyadic_operands(route):
    run_route(route, "B")


@pytest.mark.gpu
@pytest.mark.parametrize("reserved", [1, 9, 37, 73])
def test_routes_stay_exact_when_sms_are_reserved(reserved):
    """b200unet_set_reserved_sms moves every persistent grid, the statistics slot count, the split-K count S (and with it
    the finalize form) and the CTA-pair threshold.  Every route stays exact; the routes that changed are listed."""
    _lib, _ = _ops()
    changed = []
    for route in ROUTES:
        if route.name not in _DEFAULT_KEYS:
            _DEFAULT_KEYS[route.name] = route_kernels(route)[1]
        prev = _lib.call("b200unet_set_reserved_sms", reserved)
        try:
            _, keys = route_kernels(route)
        finally:
            _lib.call("b200unet_set_reserved_sms", prev)
        before, after = set(_DEFAULT_KEYS[route.name]), set(keys)
        if before != after:
            changed.append((route.name, sorted(before - after), sorted(after - before)))
    print(f"\nreserved SMs {reserved}: {len(changed)} routes changed kernels")
    for name, gone, new in changed:
        print(f"  {name}: {gone} -> {new}")
    moved = {name: new for name, _, new in changed}
    if reserved == 73:  # 75 SMs: 40 pair tiles exceed half of them, and 75 // 6 = 12 splits take the tiled finalize
        assert "gconv_kernel<64,256,3,6,false,0,1,2>" in moved.get("pair_threshold", [])
        assert "wgrad_finalize_tiled_kernel" in moved.get("wg_splits_threshold", [])
    else:
        assert "pair_threshold" not in moved and "wg_splits_threshold" not in moved


# ------------------------------------------------------------------------------------------- programmatic launch
CHAIN = dict(n=2, h=24, w=80, c0=64, c1=64, c2=128)


def chain_operands(device):
    gen = torch.Generator(device=device).manual_seed(31)
    c = CHAIN
    x = int_operand((c["n"], c["h"], c["w"], c["c0"]), 0.5, gen, device).to(F64)
    w1 = int_operand((c["c1"], c["c0"], 3, 3), 0.005, gen, device).to(F64)
    w2 = int_operand((c["c2"], c["c1"], 3, 3), 0.002, gen, device).to(F64)
    return dict(x=x, w1=w1, w2=w2)


def chain_reference(o):
    y1 = snap(ref_fprop(o["x"], o["w1"], 1), 1.0)
    y2 = snap(ref_fprop(y1, o["w2"], 1), 1.0)
    dx = snap(ref_dgrad(y2, o["w2"], (CHAIN["h"], CHAIN["w"]), 1), 1.0)
    dw = snap(ref_wgrad(y1, y2, tuple(o["w2"].shape), 1), 1.0)
    for t in (y1, y2, dx):
        assert float(t.abs().max()) <= 256
    for t in (y1, y2):
        assert float(stats_of(t)[..., 1].max()) < EXACT
    assert float(y1.abs().max()) * float(y2.abs().sum((0, 1, 2)).max()) < EXACT
    assert float(y2.abs().max()) > 0 and float(dw.abs().max()) > 0
    return y1, y2, dx, dw


@pytest.mark.gpu
def test_dependent_launches_with_pdl_are_exact():
    """With programmatic dependent launch a kernel becomes resident under its producer's tail, and one that touched
    global memory before griddepcontrol.wait would read that producer's output early.  The chain: fprop1 (nconv, with
    statistics) -> fprop2 of its output (gconv, no statistics) -> data gradient of conv 2 with dy = y2 (gconv) -> weight
    gradient of conv 2 from y1 and y2 (wgrad_kernel + finalize).  Every buffer is allocated and NaN-filled before PDL is
    switched on, and the four calls go back to back through the C ABI, so nothing else is on the stream between them.
    Edges covered: fprop1 -> fprop2 (no statistics memset in front of fprop2), fprop2 -> dgrad, dgrad -> wgrad (which
    may start while fprop2 still writes y2) and wgrad -> its finalize.  fprop1 follows the library's own statistics
    memset, as every fprop with statistics does."""
    _lib, ops = _ops()
    o = to_cuda(chain_operands("cuda"))
    y1r, y2r, dxr, dwr = chain_reference(o)
    c = CHAIN
    w1f, _ = ops.pack_conv_weights(o["w1"].float(), need_dgrad=False)
    w2f, w2d = ops.pack_conv_weights(o["w2"].float())
    x = o["x"].to(BF16)
    y1 = torch.full((c["n"], c["h"], c["w"], c["c1"]), NAN, dtype=BF16, device="cuda")
    y2 = torch.full((c["n"], c["h"], c["w"], c["c2"]), NAN, dtype=BF16, device="cuda")
    dx = torch.full((c["n"], c["h"], c["w"], c["c1"]), NAN, dtype=BF16, device="cuda")
    st1 = fprop_stats_buffer(x, c["c1"], 1)
    dw, ws = wgrad_buffers(y1, y2, 1)
    torch.cuda.synchronize()
    prev = _lib.call("b200unet_set_pdl", 1)
    try:
        launch_fprop(x, w1f, 1, y1, st1)
        launch_fprop(y1, w2f, 1, y2, None)
        ops.conv_dgrad(y2, w2d, (c["h"], c["w"]), 1, out=dx)
        launch_wgrad(y1, y2, 1, dw, ws)
        torch.cuda.synchronize()
    finally:
        _lib.call("b200unet_set_pdl", prev)
    assert_exact(y1, y1r, "y1")
    assert_exact(st1.to(F64).sum(1), stats_of(y1r), "stats of y1")
    assert_exact(y2, y2r, "y2")
    assert_exact(dx, dxr, "dx")
    assert_exact(dw, dwr, "dw")


# ------------------------------------------------------------------------------------------ stem and direct kernels
@pytest.mark.gpu
def test_stem_kernels_are_exact_on_an_integer_image():
    """stem_fprop (fp32 NCHW image -> bf16 NHWC + statistics), stem_wgrad and the tensor-core stem_wgrad_tc."""
    _lib, ops = _ops()
    n, h, w = 2, 48, 80
    o = to_cuda(make_operands("stem", "stem", n, h, w, 3, 32, 1, "A"))
    img = o["x"].permute(0, 3, 1, 2).float().contiguous()
    wt = o["w"].float().contiguous()
    y_ref = snap(ref_fprop(o["x"], o["w"], 1), 1.0)
    dw_ref = snap(ref_wgrad(o["x"], o["dy"], (32, 3, 3, 3), 1), 1.0)
    check_preconditions("fprop", o, y_ref, stats=True)
    check_preconditions("wgrad", o, dw_ref)
    y = torch.full((n, h, w, 32), NAN, dtype=BF16, device="cuda")
    parts = _lib.call("b200unet_stem_partials", h, w)
    stats = torch.full((n, parts, 32, 2), NAN, dtype=F32, device="cuda")
    _lib.call("b200unet_stem_fprop", ops._p(img), ops._p(wt), ops._p(y), ops.pitch_of(y), ops._p(stats), n, h, w,
              ops._stream())
    dy = o["dy"].to(BF16)
    nbytes = _lib.call("b200unet_stem_wgrad_workspace", n, h, w)
    ws = torch.full((nbytes // 4,), NAN, dtype=F32, device="cuda")
    dw = torch.full((32, 3, 3, 3), NAN, dtype=F32, device="cuda")
    _lib.call("b200unet_stem_wgrad", ops._p(img), ops._p(dy), ops.pitch_of(dy), ops._p(dw), ops._p(ws), nbytes, n, h, w,
              ops._stream())
    dw32 = run_wgrad(ops.image_to_nhwc32(img), dy, 1)
    torch.cuda.synchronize()
    assert_exact(y, y_ref, "y")
    assert_exact(stats.to(F64).sum(1), stats_of(y_ref), "stats")
    assert_exact(dw, dw_ref, "dw")
    assert_exact(dw32[:, :3], dw_ref, "dw (tensor cores)")
    assert_exact(dw32[:, 3:], torch.zeros_like(dw32[:, 3:]), "dw of the zero-padded channels")


DIRECT_SHAPES = [(2, 12, 20, 64, 96, 1), (2, 13, 21, 64, 96, 2), (1, 9, 13, 32, 8, 1)]  # Cout 8: the fp32 head


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["A", "B"])
@pytest.mark.parametrize("shape", DIRECT_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("case", ["simt", "f32"])
def test_direct_kernels_are_exact(case, shape, regime):
    """The CUDA-core kernels: simt=True on bf16 tensors and the fp32 verification mode (_f32 entry points)."""
    _, ops = _ops()
    n, h, w, cin, cout, s = shape
    oh, ow = out_hw(h, w, s)
    dt = F32 if case == "f32" else BF16
    wf = wd = None
    for op in ("fprop", "dgrad", "wgrad"):
        o = to_cuda(make_operands(f"{case}/{shape}/{op}", op, *shape, regime))
        ref = reference(op, o, (h, w))
        check_preconditions(op, o, ref, stats=op == "fprop" and regime == "A")
        want = ref.to(BF16) if (regime == "B" and dt == BF16 and op != "wgrad") else ref
        wf, wd = ops.pack_conv_weights(o["w"].float(), dtype=dt)
        if op == "fprop":
            y = torch.full((n, oh, ow, cout), NAN, dtype=dt, device="cuda")
            stats = run_fprop(o["x"].to(dt), wf, s, y, simt=True)
            torch.cuda.synchronize()
            assert_exact(y, want, "y")
            if regime == "A":
                assert_exact(stats.to(F64).sum(1), stats_of(ref), "stats")
        elif op == "dgrad":
            dx = torch.full((n, h, w, cin), NAN, dtype=dt, device="cuda")
            ops.conv_dgrad(o["dy"].to(dt), wd, (h, w), s, out=dx, simt=True)
            torch.cuda.synchronize()
            assert_exact(dx, want, "dx")
        else:
            dw = run_wgrad(o["x"].to(dt), o["dy"].to(dt), s, simt=True)
            torch.cuda.synchronize()
            assert_exact(dw, ref, "dw")


# ------------------------------------------------------------------------------------------------------ full size
def _full_layers():
    from test_gpu_fullsize import FULL_LAYERS
    return list(FULL_LAYERS) + [
        ("clip_fusion_centre_tap", 1024, 512, 1, 16),  # the CLIP fusion 1x1 conv as the centre tap of a 3x3 conv
        ("ae_head_29_zero_channels", 32, 32, 1, 512),  # the autoencoder head: 3 live output channels of 32
    ]


FULL_B = 32
CHUNK = 4  # images per float64 reference evaluation


@pytest.mark.gpu
@pytest.mark.parametrize("name,cin,cout,stride,hw", _full_layers(), ids=[lay[0] for lay in _full_layers()])
def test_full_size_layers_are_exact(name, cin, cout, stride, hw):
    """Batch 32 at the benchmark's layer shapes, regime A: y and its statistics, dx (and the parity-stacked dx where
    the model uses it), dw.  The float64 reference runs on the device, a few images at a time."""
    _, ops = _ops()
    wmask = dymask = None
    if name.startswith("clip"):
        wmask = torch.zeros(cout, cin, 3, 3)
        wmask[:, :, 1, 1] = 1
    if name.startswith("ae_head"):
        wmask = torch.zeros(cout, cin, 3, 3)
        wmask[:3] = 1
        dymask = torch.zeros(cout)
        dymask[:3] = 1
    o = make_operands(name, "fprop", FULL_B, hw, hw, cin, cout, stride, "A", device="cuda", wmask=wmask, dymask=dymask)
    oh, ow = out_hw(hw, hw, stride)
    wf, wd = ops.pack_conv_weights(o["w"].float())
    x, dy = o["x"].to(BF16), o["dy"].to(BF16)
    y = torch.full((FULL_B, oh, ow, cout), NAN, dtype=BF16, device="cuda")
    stats = run_fprop(x, wf, stride, y)
    dx = torch.full((FULL_B, hw, hw, cin), NAN, dtype=BF16, device="cuda")
    ops.conv_dgrad(dy, wd, (hw, hw), stride, out=dx)
    dx2 = None
    if stride == 2 and cin <= 64:
        dx2 = torch.full((FULL_B, hw, hw, cin), NAN, dtype=BF16, device="cuda")
        ops.conv_dgrad_s2(dy, ops.pack_s2_dgrad_weights(wd), (hw, hw), out=dx2)
    dw = run_wgrad(x, dy, stride)
    torch.cuda.synchronize()
    assert float(o["dyi"].abs().to(F64).sum((0, 1, 2)).max()) * 2 < EXACT  # the weight-gradient sums stay exact
    for k in ("x", "w", "dy"):
        assert torch.equal(o[k].to(BF16).to(F64), o[k])
    stats_sum = stats.to(F64).sum(1)
    dw_ref = torch.zeros(cout, cin, 3, 3, dtype=F64, device="cuda")
    for i in range(0, FULL_B, CHUNK):
        sl = slice(i, i + CHUNK)
        y_ref = snap(ref_fprop(o["x"][sl], o["w"], stride), 1.0)
        assert float(y_ref.abs().max()) <= 256
        s_ref = stats_of(y_ref)
        assert float(s_ref[..., 1].max()) < EXACT
        assert_exact(y[sl], y_ref, f"y (images {i}..)")
        assert_exact(stats_sum[sl], s_ref, f"stats (images {i}..)")
        del y_ref
        dx_ref = snap(ref_dgrad(o["dy"][sl], o["w"], (hw, hw), stride), 1.0)
        assert float(dx_ref.abs().max()) <= 256
        assert_exact(dx[sl], dx_ref, f"dx (images {i}..)")
        if dx2 is not None:
            assert_exact(dx2[sl], dx_ref, f"dx, parity-stacked (images {i}..)")
        del dx_ref
        dw_ref += ref_wgrad(o["x"][sl], o["dy"][sl], (cout, cin, 3, 3), stride)
    assert_exact(dw, snap(dw_ref, 1.0), "dw")
