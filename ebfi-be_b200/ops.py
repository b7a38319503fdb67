"""The ops a model's forward and backward call, registered as torch custom operators (`torch.ops.ebfi_b200.*`), so
that torch.compile and torch.export see them as single graph nodes instead of breaking the graph at a ctypes call.

Each op runs the existing Python body (argument checks, then the C entry of libebfi_b200.so) and has a fake that
gives the eager outputs' shapes and dtypes, in SymInt arithmetic, and raises where the eager checks raise. The
autograd Functions, the shim functions and frame_ops call these ops only while torch.compile / torch.export traces
them (`torch.compiler.is_compiling()`); eager calls go straight to the bodies, so eager results and host cost are
those of the direct calls.

Under the ops the DCN entries neither leave nor read the forward's blocked input copy (`_ext._blocked_cache`): a
compiled backward re-blocks its input, with the same bits. Out of scope (eager only, a graph break when compiled):
the event encoders and EventSliceFeeder, `dcn_v2_backward_dp` and any call with `comm`, HostPipeline, the PS-ROI
stubs and channels_last.
"""
import types
from typing import Optional

import torch
from torch import Tensor

from . import _lib as L
from . import frame_ops, kernelconv2d, modification
from .shims import _ext, kernelconv2d_cuda

_f32 = torch.float32


# ---------------------------------------------------------------------------------------------------------- DCNv2
def _out_len(n, k, stride, pad, dilation):
    """One output extent as ebfi_dcnv2_output_size computes it (C division truncates toward zero)."""
    num = n + 2 * pad - (dilation * (k - 1) + 1)
    return (num // stride if num >= 0 else -((-num) // stride)) + 1


def _fake_geom(input, weight, ints):
    """_ext._geom for fake tensors: the same checks, and the geometry fields the shape checks read."""
    kh, kw, sh, sw, ph, pw, dh, dw, dg = ints
    _ext._check_weight(input, weight, kh, kw)
    B, C, H, W = input.shape
    Co = weight.shape[0]
    if not (B > 0 and C > 0 and H > 0 and W > 0 and Co > 0):
        raise RuntimeError("dcn_v2 geometry failed: dcn: non-positive tensor size")
    if not (kh > 0 and kw > 0 and sh > 0 and sw > 0 and dh > 0 and dw > 0 and ph >= 0 and pw >= 0):
        raise RuntimeError("dcn_v2 geometry failed: dcn: bad kernel/stride/dilation/padding")
    if not (dg > 0 and C % dg == 0):
        raise RuntimeError(f"dcn_v2 geometry failed: dcn: channels ({C}) not divisible by deformable_group ({dg})")
    ho, wo = _out_len(H, kh, sh, ph, dh), _out_len(W, kw, sw, pw, dw)
    if not (ho > 0 and wo > 0):
        raise RuntimeError(f"dcn_v2 geometry failed: dcn: empty output {ho}x{wo}")
    g = types.SimpleNamespace(batch=B, channels_out=Co, kernel_h=kh, kernel_w=kw, deformable_group=dg)
    return g, ho, wo


def _require_contiguous(input, weight):
    # dcn_v2_backward / dcn_v2_backward_packed
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")


def _grad_dtypes(dt, weight, bias, n_act):
    """Activation gradients in the call's dtype, grad_weight / grad_bias in the parameters' (fp32 under autocast)."""
    return [dt] * n_act + [weight.dtype, bias.dtype] if dt in _ext._HALF else [_f32] * (n_act + 2)


@torch.library.custom_op("ebfi_b200::dcn_v2_forward", mutates_args=())
def dcn_v2_forward(input: Tensor, weight: Tensor, bias: Tensor, offset: Tensor, mask: Tensor, kernel_h: int,
                   kernel_w: int, stride_h: int, stride_w: int, pad_h: int, pad_w: int, dilation_h: int,
                   dilation_w: int, deformable_group: int) -> Tensor:
    return _ext.dcn_v2_forward(input, weight, bias, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h,
                               pad_w, dilation_h, dilation_w, deformable_group, reuse_blocked=False)


@dcn_v2_forward.register_fake
def _(input, weight, bias, offset, mask, *ints):
    dt = _ext._check_cuda(input=input, weight=weight, bias=bias, offset=offset, mask=mask)
    g, ho, wo = _fake_geom(input, weight, ints)
    _ext._check_offset_mask(g, ho, wo, offset, mask)
    return input.new_empty((g.batch, g.channels_out, ho, wo), dtype=dt)


@torch.library.custom_op("ebfi_b200::dcn_v2_backward", mutates_args=())
def dcn_v2_backward(input: Tensor, weight: Tensor, bias: Tensor, offset: Tensor, mask: Tensor, grad_output: Tensor,
                    kernel_h: int, kernel_w: int, stride_h: int, stride_w: int, pad_h: int, pad_w: int,
                    dilation_h: int, dilation_w: int,
                    deformable_group: int) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    return tuple(_ext.dcn_v2_backward(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h,
                                      stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group,
                                      reuse_blocked=False))


@dcn_v2_backward.register_fake
def _(input, weight, bias, offset, mask, grad_output, *ints):
    _require_contiguous(input, weight)
    dt = _ext._check_cuda(input=input, weight=weight, bias=bias, offset=offset, mask=mask, grad_output=grad_output)
    g, ho, wo = _fake_geom(input, weight, ints)
    _ext._check_offset_mask(g, ho, wo, offset, mask)
    if tuple(grad_output.shape) != (g.batch, g.channels_out, ho, wo):
        raise RuntimeError("dcn_v2_backward: grad_output has the wrong shape")
    return tuple(t.new_empty(t.shape, dtype=d)
                 for t, d in zip((input, offset, mask, weight, bias), _grad_dtypes(dt, weight, bias, 3)))


@torch.library.custom_op("ebfi_b200::dcn_v2_forward_packed", mutates_args=("abs_offset_sum",))
def dcn_v2_forward_packed(input: Tensor, weight: Tensor, bias: Tensor, offset_mask: Tensor, kernel_h: int,
                          kernel_w: int, stride_h: int, stride_w: int, pad_h: int, pad_w: int, dilation_h: int,
                          dilation_w: int, deformable_group: int, abs_offset_sum: Optional[Tensor]) -> Tensor:
    return _ext.dcn_v2_forward_packed(input, weight, bias, offset_mask, kernel_h, kernel_w, stride_h, stride_w,
                                      pad_h, pad_w, dilation_h, dilation_w, deformable_group, abs_offset_sum,
                                      reuse_blocked=False)


@dcn_v2_forward_packed.register_fake
def _(input, weight, bias, offset_mask, *ints_and_stat):
    *ints, abs_offset_sum = ints_and_stat
    dt = _ext._check_cuda(input=input, weight=weight, bias=bias, offset_mask=offset_mask)
    g, ho, wo = _fake_geom(input, weight, ints)
    _ext._check_packed(g, ho, wo, offset_mask)
    if abs_offset_sum is not None and not (abs_offset_sum.is_cuda and abs_offset_sum.dtype == _f32
                                           and abs_offset_sum.numel() == 1):
        raise RuntimeError("dcn_v2_forward_packed: abs_offset_sum must be a 1-element float32 CUDA tensor")
    return input.new_empty((g.batch, g.channels_out, ho, wo), dtype=dt)


@torch.library.custom_op("ebfi_b200::dcn_v2_backward_packed", mutates_args=())
def dcn_v2_backward_packed(input: Tensor, weight: Tensor, bias: Tensor, offset_mask: Tensor, grad_output: Tensor,
                           kernel_h: int, kernel_w: int, stride_h: int, stride_w: int, pad_h: int, pad_w: int,
                           dilation_h: int, dilation_w: int,
                           deformable_group: int) -> tuple[Tensor, Tensor, Tensor, Tensor]:
    return tuple(_ext.dcn_v2_backward_packed(input, weight, bias, offset_mask, grad_output, kernel_h, kernel_w,
                                             stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                                             deformable_group, reuse_blocked=False))


@dcn_v2_backward_packed.register_fake
def _(input, weight, bias, offset_mask, grad_output, *ints):
    _require_contiguous(input, weight)
    dt = _ext._check_cuda(input=input, weight=weight, bias=bias, offset_mask=offset_mask, grad_output=grad_output)
    g, ho, wo = _fake_geom(input, weight, ints)
    _ext._check_packed(g, ho, wo, offset_mask)
    if tuple(grad_output.shape) != (g.batch, g.channels_out, ho, wo):
        raise RuntimeError("dcn_v2_backward_packed: grad_output has the wrong shape")
    return tuple(t.new_empty(t.shape, dtype=d)
                 for t, d in zip((input, offset_mask, weight, bias), _grad_dtypes(dt, weight, bias, 2)))


# ------------------------------------------------------------------------------------------------------------ FAC
# kernelconv2d_cuda writes into tensors its caller allocated, as the reference's extension does (SURVEY §8b); the ops
# declare those writes.
@torch.library.custom_op("ebfi_b200::fac_forward", mutates_args=("output",))
def fac_forward(input: Tensor, kernel: Tensor, kernel_size: int, output: Tensor) -> None:
    kernelconv2d_cuda.forward(input, kernel, kernel_size, output)


@fac_forward.register_fake
def _(input, kernel, kernel_size, output):
    kernelconv2d_cuda._check_forward(input, kernel, kernel_size, output)


@torch.library.custom_op("ebfi_b200::fac_backward", mutates_args=("grad_input", "grad_kernel"))
def fac_backward(input: Tensor, kernel: Tensor, kernel_size: int, grad_output: Tensor, grad_input: Tensor,
                 grad_kernel: Tensor) -> None:
    kernelconv2d_cuda.backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel)


@fac_backward.register_fake
def _(input, kernel, kernel_size, grad_output, grad_input, grad_kernel):
    kernelconv2d_cuda._check_backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel)


@torch.library.custom_op("ebfi_b200::fac_replpad_forward", mutates_args=())
def fac_replpad_forward(input: Tensor, kernel: Tensor, kernel_size: int) -> Tensor:
    L.require_cuda(input, kernel)
    return kernelconv2d._replpad_forward(input, kernel, kernel_size)


@fac_replpad_forward.register_fake
def _(input, kernel, kernel_size):
    L.require_cuda(input, kernel)
    kernelconv2d._replpad_dims(input, kernel, kernel_size)
    return input.new_empty(input.shape)


@torch.library.custom_op("ebfi_b200::fac_replpad_backward", mutates_args=())
def fac_replpad_backward(input: Tensor, kernel: Tensor, kernel_size: int,
                         grad_output: Tensor) -> tuple[Tensor, Tensor]:
    L.require_cuda(input, kernel, grad_output)
    return kernelconv2d._replpad_backward(input, kernel, kernel_size, grad_output)


@fac_replpad_backward.register_fake
def _(input, kernel, kernel_size, grad_output):
    L.require_cuda(input, kernel, grad_output)
    kernelconv2d._check_replpad_grad(input, grad_output)
    kernelconv2d._replpad_dims(input, kernel, kernel_size)
    return input.new_empty(input.shape), kernel.new_empty(kernel.shape)


# -------------------------------------------------------------------------------- fused KernelConv -> FAC block
def _kpn_check(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, grad_output=None):
    """What the module-level callers of modification._fused_forward / _fused_backward guarantee: CUDA tensors,
    activations all fp32, all bf16 or all fp16, fp32 weight and bias, a shape the fused kernel supports."""
    acts = (event_feat, frame_feat) if grad_output is None else (event_feat, frame_feat, grad_output)
    L.require_cuda(*acts, conv_weight, conv_bias)
    if len({t.dtype for t in acts}) != 1 or event_feat.dtype not in modification._SUFFIX \
            or conv_weight.dtype != _f32 or conv_bias.dtype != _f32:
        raise RuntimeError("kpn_fused: the activations must be all float32, all bfloat16 or all float16 and "
                           f"conv_weight / conv_bias float32, got {[str(t.dtype) for t in acts]} / "
                           f"{conv_weight.dtype} / {conv_bias.dtype}")
    dims = modification._block_dims(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, "kpn_fused")
    if grad_output is not None and tuple(grad_output.shape) != tuple(event_feat.shape):
        raise RuntimeError("kpn_fused_backward: grad_output must have the event features' shape")
    if not modification.kernelconv_fac_fused_supported(event_feat.shape[1], frame_feat.shape[1], kernel_size):
        raise RuntimeError(f"kpn_fused: Ce + Cf = {event_feat.shape[1] + frame_feat.shape[1]}, K = {kernel_size} "
                           "is not a shape the fused kernel supports")
    return dims


@torch.library.custom_op("ebfi_b200::kpn_fused_forward", mutates_args=())
def kpn_fused_forward(event_feat: Tensor, frame_feat: Tensor, conv_weight: Tensor, conv_bias: Tensor,
                      kernel_size: int, negative_slope: float) -> Tensor:
    _kpn_check(event_feat, frame_feat, conv_weight, conv_bias, kernel_size)
    return modification._fused_forward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope)


@kpn_fused_forward.register_fake
def _(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope):
    _kpn_check(event_feat, frame_feat, conv_weight, conv_bias, kernel_size)
    return event_feat.new_empty(event_feat.shape)


@torch.library.custom_op("ebfi_b200::kpn_fused_backward", mutates_args=())
def kpn_fused_backward(event_feat: Tensor, frame_feat: Tensor, conv_weight: Tensor, conv_bias: Tensor,
                       kernel_size: int, negative_slope: float,
                       grad_output: Tensor) -> tuple[Tensor, Tensor, Tensor]:
    _kpn_check(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, grad_output)
    return modification._fused_backward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope,
                                        grad_output, "kpn_fused_backward")


@kpn_fused_backward.register_fake
def _(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope, grad_output):
    B, Ce, Cf, H, W, K = _kpn_check(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, grad_output)
    return (event_feat.new_empty((B, Ce * K * K, H, W)), event_feat.new_empty((B, Ce, H, W), dtype=_f32),
            event_feat.new_empty((Ce * K * K,), dtype=_f32))


# ----------------------------------------------------------------------------------------------------- frame maps
@torch.library.custom_op("ebfi_b200::frame_to_lap", mutates_args=())
def frame_to_lap(ims: Tensor) -> Tensor:
    return frame_ops.Frame2Lap(ims)


@frame_to_lap.register_fake
def _(ims):
    x = frame_ops._frames(ims)
    return x.new_empty((x.shape[0], 1, x.shape[2], x.shape[3]))


@torch.library.custom_op("ebfi_b200::frame_to_dcp", mutates_args=())
def frame_to_dcp(ims: Tensor, sz: int = 35) -> Tensor:
    return frame_ops.Frame2DCP(ims, sz)


@frame_to_dcp.register_fake
def _(ims, sz=35):
    x = frame_ops._frames(ims)
    return x.new_empty((x.shape[0], 1, x.shape[2], x.shape[3]))
