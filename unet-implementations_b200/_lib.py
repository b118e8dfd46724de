"""ctypes binding of libb200unet.so (C ABI declared in include/b200unet.h).

There is no fallback: if the shared library is missing or an entry point fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200UNET_LIB") or os.path.join(_HERE, "libb200unet.so")  # env: developer A/B of two builds

_lib = None


class ConvFpropArgs(Structure):
    _fields_ = [
        ("x", c_void_p), ("x_pitch", c_int64), ("w", c_void_p), ("y", c_void_p), ("y_pitch", c_int64),
        ("stats", c_void_p), ("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int), ("Cout", c_int),
        ("stride", c_int),
    ]


class ConvDgradArgs(Structure):
    _fields_ = [
        ("dy", c_void_p), ("dy_pitch", c_int64), ("wt", c_void_p), ("dx", c_void_p), ("dx_pitch", c_int64),
        ("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int), ("Cout", c_int), ("stride", c_int),
        ("bs_y", c_void_p), ("bs_y_pitch", c_int64), ("bs_a", c_void_p), ("bs_b", c_void_p), ("bs_slope", c_float),
        ("bs_part", c_void_p), ("dx2", c_void_p), ("dx2_pitch", c_int64), ("dx_split", c_int),
    ]


class ConvWgradArgs(Structure):
    _fields_ = [
        ("x", c_void_p), ("x_pitch", c_int64), ("dy", c_void_p), ("dy_pitch", c_int64), ("dw", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_int64), ("N", c_int), ("H", c_int), ("W", c_int),
        ("Cin", c_int), ("Cout", c_int), ("stride", c_int),
    ]


class InBwdArgs(Structure):
    _fields_ = [
        ("dz", c_void_p), ("dz_pitch", c_int64), ("dz2", c_void_p), ("dz2_pitch", c_int64), ("y", c_void_p),
        ("y_pitch", c_int64), ("a", c_void_p), ("b", c_void_p), ("mean", c_void_p), ("rstd", c_void_p),
        ("drop_scale", c_void_p), ("gamma", c_void_p), ("slope", c_float), ("dy", c_void_p), ("dy_pitch", c_int64),
        ("dgamma", c_void_p), ("dbeta", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_int64),
        ("N", c_int), ("HW", c_int64), ("C", c_int),
        ("ext_part", c_void_p), ("ext_P", c_int), ("ext_part2", c_void_p), ("ext_P2", c_int), ("defer_params", c_int),
    ]


class FlatTensor(Structure):
    """b200unet_flat_tensor (include/b200unet.h): one tensor of the flat optimizer step."""
    _fields_ = [
        ("offset", c_int64), ("numel", c_int), ("flags", c_int), ("first_block", c_int), ("cout", c_int), ("cin", c_int),
        ("ksize", c_int), ("cout_pad", c_int), ("cin_pad", c_int), ("wf", c_void_p), ("wd", c_void_p), ("ws", c_void_p),
    ]


_P, _I, _L, _F, _D = c_void_p, c_int, c_int64, c_float, c_double

# name -> (restype, argtypes); restype c_int means "status code, raise on non-zero"
SIGNATURES = {
    "b200unet_version": (c_int, []),
    "b200unet_last_error": (c_char_p, []),
    "b200unet_device_ok": (c_int, []),
    "b200unet_set_reserved_sms": (c_int, [_I]),
    "b200unet_set_pdl": (c_int, [_I]),
    "b200unet_launch_count": (c_int64, []),
    "b200unet_conv_fprop_partials": (c_int, [_I, _I, _I, _I]),
    "b200unet_conv_fprop": (c_int, [POINTER(ConvFpropArgs), _P]),
    "b200unet_conv_dgrad": (c_int, [POINTER(ConvDgradArgs), _P]),
    "b200unet_conv_dgrad_bwd_slots": (c_int, [_I, _I, _I, _I, _I, _I]),
    "b200unet_conv_dgrad_s2_supported": (c_int, [_I, _I]),
    "b200unet_pack_s2_dgrad_weights": (c_int, [_P, _P, _I, _I, _P]),
    "b200unet_conv_dgrad_s2": (c_int, [POINTER(ConvDgradArgs), _P]),
    "b200unet_conv_wgrad_workspace": (c_int64, [_I, _I, _I, _I, _I, _I]),
    "b200unet_conv_wgrad": (c_int, [POINTER(ConvWgradArgs), _P]),
    "b200unet_conv_fprop_simt_partials": (c_int, [_I, _I]),
    "b200unet_conv_fprop_simt": (c_int, [POINTER(ConvFpropArgs), _P]),
    "b200unet_conv_dgrad_simt": (c_int, [POINTER(ConvDgradArgs), _P]),
    "b200unet_conv_wgrad_simt": (c_int, [POINTER(ConvWgradArgs), _P]),
    "b200unet_pack_conv_weights": (c_int, [_P, _P, _P, _I, _I, _P]),
    "b200unet_stem_partials": (c_int, [_I, _I]),
    "b200unet_stem_fprop": (c_int, [_P, _P, _P, _L, _P, _I, _I, _I, _P]),
    "b200unet_stem_wgrad_workspace": (c_int64, [_I, _I, _I]),
    "b200unet_stem_wgrad": (c_int, [_P, _P, _L, _P, _P, _L, _I, _I, _I, _P]),
    "b200unet_in_finalize": (c_int, [_P, _I, _P, _P, _P, _F, _P, _P, _P, _P, _I, _I, _L, _P]),
    "b200unet_in_apply": (c_int, [_P, _L, _P, _P, _F, _P, _L, _I, _L, _I, _P]),
    "b200unet_in_backward_workspace": (c_int64, [_I, _L, _I]),
    "b200unet_in_backward": (c_int, [POINTER(InBwdArgs), _P]),
    "b200unet_in_bwd_params": (c_int, [_P, _I, _L, _I, _P, _P, _P]),
    "b200unet_upsample2x_fwd": (c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_upsample2x_bwd": (c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_head_fwd": (c_int, [_P, _L, _P, _P, _P, _I, _L, _I, _I, _P]),
    "b200unet_head_bwd_workspace": (c_int64, [_I, _L, _I, _I]),
    "b200unet_head_bwd": (c_int, [_P, _P, _L, _P, _P, _L, _P, _P, _P, _L, _I, _L, _I, _I, _P]),
    "b200unet_loss_workspace": (c_int64, [_I, _L]),
    "b200unet_loss_fwd": (c_int, [_P, _P, _P, _I, _F, _F, _I, _F, _P, _P, _P, _L, _I, _L, _P]),
    "b200unet_loss_bwd": (c_int, [_P, _P, _P, _P, _F, _F, _I, _P, _I, _L, _P]),
    "b200unet_loss_fwd_u8": (c_int, [_P, _P, _P, _I, _F, _F, _I, _F, _P, _P, _P, _L, _I, _L, _P]),
    "b200unet_loss_bwd_u8": (c_int, [_P, _P, _P, _P, _F, _F, _I, _P, _I, _L, _P]),
    "b200unet_nchw_f32_to_nhwc_bf16": (c_int, [_P, _P, _L, _I, _I, _L, _P]),
    "b200unet_nhwc_bf16_to_nchw_f32": (c_int, [_P, _L, _P, _I, _I, _L, _P]),
    # fp32 verification mode: same signatures as the bf16 entry points
    "b200unet_pack_conv_weights_f32": (c_int, [_P, _P, _P, _I, _I, _P]),
    "b200unet_conv_fprop_f32": (c_int, [POINTER(ConvFpropArgs), _P]),
    "b200unet_conv_dgrad_f32": (c_int, [POINTER(ConvDgradArgs), _P]),
    "b200unet_conv_wgrad_f32": (c_int, [POINTER(ConvWgradArgs), _P]),
    "b200unet_in_apply_f32": (c_int, [_P, _L, _P, _P, _F, _P, _L, _I, _L, _I, _P]),
    "b200unet_in_backward_f32": (c_int, [POINTER(InBwdArgs), _P]),
    "b200unet_upsample2x_fwd_f32": (c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_upsample2x_bwd_f32": (c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_head_fwd_f32": (c_int, [_P, _L, _P, _P, _P, _I, _L, _I, _I, _P]),
    "b200unet_head_bwd_f32": (c_int, [_P, _P, _L, _P, _P, _L, _P, _P, _P, _L, _I, _L, _I, _I, _P]),
    "b200unet_nchw_f32_to_nhwc_f32": (c_int, [_P, _P, _L, _I, _I, _L, _P]),
    "b200unet_image_to_nhwc32_bf16": (c_int, [_P, _P, _I, _I, _L, _P]),
    "b200unet_upsample2x_norm_fwd": (c_int, [_P, _L, _P, _P, _F, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_upsample2x_norm_fwd_f32": (c_int, [_P, _L, _P, _P, _F, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_head_norm_fwd": (c_int, [_P, _L, _P, _P, _F, _P, _P, _P, _I, _L, _I, _I, _P]),
    "b200unet_head_norm_fwd_f32": (c_int, [_P, _L, _P, _P, _F, _P, _P, _P, _I, _L, _I, _I, _P]),
    "b200unet_head_norm_bwd": (c_int, [_P, _P, _L, _P, _P, _F, _P, _P, _L, _P, _P, _P, _L, _I, _L, _I, _I, _P]),
    "b200unet_head_norm_bwd_f32": (c_int, [_P, _P, _L, _P, _P, _F, _P, _P, _L, _P, _P, _P, _L, _I, _L, _I, _I, _P]),
    "b200unet_head_bwd_stat_slots": (c_int, [_I, _L]),
    "b200unet_head_norm_bwd_stats": (c_int, [_P, _P, _L, _P, _P, _F, _P, _P, _L, _P, _P, _P, _L, _P, _I, _L, _I, _I, _P]),
    "b200unet_head_norm_bwd_stats_f32": (c_int, [_P, _P, _L, _P, _P, _F, _P, _P, _L, _P, _P, _P, _L, _P, _I, _L, _I, _I, _P]),
    "b200unet_preprocess_u8": (c_int, [_P, _P, _P, _P, _P, _P, _I, _L, _P]),
    "b200unet_preprocess_u8_nhwc32": (c_int, [_P, _P, _P, _P, _I, _L, _P]),
    "b200unet_sgd_flat_block_elems": (c_int, []),
    "b200unet_sgd_flat_step": (c_int, [_P, _I, _I, _P, _P, _P, _F, _F, _F, _I, _F, _P, _P]),
    "b200unet_sgd_max_tensors": (c_int, []),
    "b200unet_sgd_nesterov_step": (c_int, [_P, _P, _P, _P, _I, _F, _F, _F, _I, _I, _P]),
    "b200unet_adam_flat_step": (c_int, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _D, _P, _D, _D, _D, _D, _I, _F, _P]),
    "b200unet_argmax_counts": (c_int, [_P, _P, _I, _P, _P, _I, _L, _P]),
    "b200unet_recon_head_fwd": (c_int, [_P, _L, _P, _P, _I, _L, _I, _P]),
    "b200unet_recon_head_fwd_f32": (c_int, [_P, _L, _P, _P, _I, _L, _I, _P]),
    "b200unet_recon_head_bwd_workspace": (c_int64, [_I, _L]),
    "b200unet_recon_head_bwd": (c_int, [_P, _P, _P, _L, _I, _P, _P, _L, _I, _L, _I, _P]),
    "b200unet_recon_head_bwd_f32": (c_int, [_P, _P, _P, _L, _I, _P, _P, _L, _I, _L, _I, _P]),
    "b200unet_mse_workspace": (c_int64, [_L]),
    "b200unet_mse_fwd": (c_int, [_P, _P, _P, _P, _L, _L, _P]),
    "b200unet_mse_bwd": (c_int, [_P, _P, _P, _P, _L, _P]),
}

# entry points that return a value rather than a status code
_VALUE_FUNCS = {
    "b200unet_version", "b200unet_last_error", "b200unet_device_ok", "b200unet_set_reserved_sms", "b200unet_set_pdl", "b200unet_launch_count", "b200unet_conv_fprop_partials",
    "b200unet_conv_fprop_simt_partials", "b200unet_sgd_max_tensors", "b200unet_sgd_flat_block_elems", "b200unet_head_bwd_stat_slots", "b200unet_conv_dgrad_bwd_slots", "b200unet_recon_head_bwd_workspace",
    "b200unet_conv_dgrad_s2_supported",
    "b200unet_mse_workspace",
    "b200unet_conv_wgrad_workspace", "b200unet_stem_partials", "b200unet_stem_wgrad_workspace",
    "b200unet_in_backward_workspace", "b200unet_head_bwd_workspace", "b200unet_loss_workspace",
}


def load():
    """Load the shared library (once) and declare every signature.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"b200unet: {LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C unet-implementations_b200/csrc`). There is no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().b200unet_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


class EventProfiler:
    """Optional per-entry-point device timing with CUDA events on torch's current stream (bench.py's roofline leg).
    Recording an event pair costs about a microsecond on the host and nothing on the device."""

    def __init__(self):
        self.pairs = {}

    def totals_ms(self):
        """name -> (total ms, calls); call after a synchronize."""
        return {k: (sum(a.elapsed_time(b) for a, b in v), len(v)) for k, v in self.pairs.items()}


PROFILER = None  # set to an EventProfiler to time every entry point


def call(name: str, *args):
    """Call a status-returning entry point; raise RuntimeError(last_error) on failure."""
    fn = getattr(load(), name)
    prof = PROFILER
    if prof is not None and name not in _VALUE_FUNCS:
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        prof.pairs.setdefault(name, []).append((e0, e1))
    else:
        rc = fn(*args)
    if name in _VALUE_FUNCS:
        return rc
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")
    return 0
