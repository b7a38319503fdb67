"""Host-side mirror of the reference's kernel-prediction block (models/Ours/model_singleframe.py:138-165,
class `Modification`): `KernelConv` (3x3 ConvLayer, LeakyReLU) producing the per-pixel (B, C*K*K, H, W) kernel
tensor that `KPN = KernelConv2D(K)` consumes once.

`kernelconv_fac_fused` runs producer and consumer as ONE sm_100a kernel (csrc/kpn.cu): the kernel tensor —
1.68 GB at the benchmark shape — never exists in HBM. It is the inference path (no autograd). `KernelConvFACFunction`
is the same forward with a fused backward (ebfi_kpn_fused_backward): the kernel recomputes the conv's pre-activation
on the tensor cores and writes dL/dP, the FAC/ReplicationPad part of dL/dEvent and dL/dbias; the conv's own weight
and input gradients then run on torch's convolution backward, as the reference's nn.Conv2d does. Neither the
pre-activation nor the kernel tensor is kept for the backward. `KernelPrediction.fused_backward = True` trains
through it; by default the module trains on the reference's op sequence. `KernelConvFACBF16Function` is the same
fused forward and backward for bf16 or fp16 activations (torch.autocast's mixed precision): the kernel reads and writes
the 16-bit activations and keeps P and the kernel tensor in fp32 registers, and the conv's gradients run as the 16-bit
convolution backward autocast's nn.Conv2d would run.
"""
import torch
from torch import nn

from . import _lib as L
from .kernelconv2d import KernelConv2D


# activation dtype -> suffix of the fused block's C entries
_SUFFIX = {torch.float32: "", torch.bfloat16: "_bf16", torch.float16: "_fp16"}


def kernelconv_fac_fused(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope=0.01):
    """out = KernelConv2D(K)(event_feat, LeakyReLU(conv3x3(cat([event_feat, frame_feat], 1)))) — CUDA tensors, all fp32,
    all bf16 or all fp16; conv operands are rounded to bf16 for the tensor cores (fp32 accumulate, fp32 FAC)."""
    L.require_cuda(event_feat, frame_feat, conv_weight, conv_bias)
    dts = {t.dtype for t in (event_feat, frame_feat, conv_weight, conv_bias)}
    if len(dts) != 1 or not dts <= set(_SUFFIX):
        raise RuntimeError("kernelconv_fac_fused: all tensors must be float32, all bfloat16 or all float16, got "
                           f"{sorted(str(d) for d in dts)}")
    if torch.is_grad_enabled() and any(t.requires_grad for t in (event_feat, frame_feat, conv_weight, conv_bias)):
        raise RuntimeError("kernelconv_fac_fused is forward-only; run it under torch.no_grad() "
                           "(training goes through KernelConv2DFunction)")
    # bfloat16 / float16 model (the 720p inference config runs bf16): the kernel reads the 16-bit activations and
    # rounds its output once; the weights' fp32 copies are exact (and small)
    return _fused_forward(event_feat, frame_feat, conv_weight.float(), conv_bias.float(), kernel_size, negative_slope)


def _block_dims(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, what):
    B, Ce, H, W = event_feat.shape
    Cf = frame_feat.shape[1]
    K = int(kernel_size)
    if tuple(frame_feat.shape) != (B, Cf, H, W) or tuple(conv_weight.shape) != (Ce * K * K, Ce + Cf, 3, 3) \
            or tuple(conv_bias.shape) != (Ce * K * K,):
        raise RuntimeError(f"{what}: shapes do not match (event (B,Ce,H,W), frame (B,Cf,H,W), "
                           "weight (Ce*K*K, Ce+Cf, 3, 3), bias (Ce*K*K))")
    return B, Ce, Cf, H, W, K


def _fused_forward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope):
    """ebfi_kpn_fused_forward (fp32 activations) or its _bf16 / _fp16 variant (16-bit activations) on CUDA tensors
    with fp32 weight and bias: the one forward of kernelconv_fac_fused, KernelConvFACFunction and
    KernelConvFACBF16Function. The output has the activations' dtype."""
    if torch.compiler.is_compiling():
        return torch.ops.ebfi_b200.kpn_fused_forward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size,
                                                     negative_slope)
    B, Ce, Cf, H, W, K = _block_dims(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, "kernelconv_fac_fused")
    event_feat, frame_feat, conv_weight, conv_bias = (t.contiguous() for t in (event_feat, frame_feat, conv_weight, conv_bias))
    lib = L.load()
    with torch.cuda.device(event_feat.device):
        out = torch.empty_like(event_feat)
        nbytes = lib.ebfi_kpn_fused_workspace_bytes(B, Ce, Cf, H, W, K)
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=event_feat.device)
        fwd = getattr(lib, "ebfi_kpn_fused_forward" + _SUFFIX[event_feat.dtype])
        L.check(fwd(L.stream_ptr(event_feat.device), L.ptr(event_feat), L.ptr(frame_feat),
                    L.ptr(conv_weight), L.ptr(conv_bias), float(negative_slope), L.ptr(out),
                    B, Ce, Cf, H, W, K, L.ptr(ws), nbytes), "kernelconv_fac_fused")
    return out


def kernelconv_fac_fused_backward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope,
                                  grad_output):
    """ebfi_kpn_fused_backward on fp32 CUDA tensors -> (grad_pre (B, Ce*K*K, H, W), grad_event_fac (B, Ce, H, W),
    grad_bias (Ce*K*K)) of out = kernelconv_fac_fused(...). grad_pre is dL/d(conv pre-activation); the conv's weight
    and input gradients follow from it by an ordinary convolution backward (KernelConvFACFunction.backward)."""
    L.require_cuda(event_feat, frame_feat, conv_weight, conv_bias, grad_output)
    L.require_f32(event_feat=event_feat, frame_feat=frame_feat, conv_weight=conv_weight, conv_bias=conv_bias,
                  grad_output=grad_output)
    return _fused_backward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope, grad_output,
                           "kernelconv_fac_fused_backward")


def kernelconv_fac_fused_backward_bf16(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope,
                                       grad_output):
    """ebfi_kpn_fused_backward_bf16 / _fp16: kernelconv_fac_fused_backward for event_feat, frame_feat and grad_output
    all bf16 or all fp16 (weight and bias fp32 or of that type; they are used as fp32) -> (grad_pre of that type,
    grad_event_fac fp32, grad_bias fp32). grad_pre is the fp32 kernel's grad_pre rounded once to the 16-bit type;
    grad_event_fac and grad_bias are the fp32 kernel's."""
    L.require_cuda(event_feat, frame_feat, conv_weight, conv_bias, grad_output)
    _require_half_io("kernelconv_fac_fused_backward_bf16", dict(event_feat=event_feat, frame_feat=frame_feat,
                                                                grad_output=grad_output),
                     dict(conv_weight=conv_weight, conv_bias=conv_bias))
    return _fused_backward(event_feat, frame_feat, conv_weight.float(), conv_bias.float(), kernel_size,
                           negative_slope, grad_output, "kernelconv_fac_fused_backward_bf16")


def _require_half_io(what, activations, parameters):
    """Activations all bf16 or all fp16; parameters fp32 (autocast) or of the activations' type (a .bfloat16() or
    .half() model)."""
    dts = {t.dtype for t in activations.values()}
    if len(dts) != 1 or not dts <= {torch.bfloat16, torch.float16}:
        got = ", ".join(f"{k} {t.dtype}" for k, t in activations.items())
        raise RuntimeError(f"{what}: the activations must be all bfloat16 or all float16, got {got} "
                           "(fp32 activations go through the fp32 entries)")
    half = dts.pop()
    for k, t in parameters.items():
        if t.dtype not in (torch.float32, half):
            raise RuntimeError(f"{what}: {k} must be float32 or {half}, got {t.dtype}")


def _fused_backward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope, grad_output, what):
    """ebfi_kpn_fused_backward or its _bf16 / _fp16 variant, chosen by the activations' dtype; fp32 weight and bias."""
    if torch.compiler.is_compiling():
        return torch.ops.ebfi_b200.kpn_fused_backward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size,
                                                      negative_slope, grad_output)
    B, Ce, Cf, H, W, K = _block_dims(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, what)
    if tuple(grad_output.shape) != tuple(event_feat.shape):
        raise RuntimeError(f"{what}: grad_output must have the event features' shape")
    event_feat, frame_feat, conv_weight, conv_bias, grad_output = (
        t.contiguous() for t in (event_feat, frame_feat, conv_weight, conv_bias, grad_output))
    lib = L.load()
    dev = event_feat.device
    with torch.cuda.device(dev):
        grad_pre = torch.empty(B, Ce * K * K, H, W, device=dev, dtype=event_feat.dtype)
        grad_event_fac = torch.empty(B, Ce, H, W, device=dev)
        grad_bias = torch.empty(Ce * K * K, device=dev)
        nbytes = lib.ebfi_kpn_fused_backward_workspace_bytes(B, Ce, Cf, H, W, K)
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        bwd = getattr(lib, "ebfi_kpn_fused_backward" + _SUFFIX[event_feat.dtype])
        L.check(bwd(L.stream_ptr(dev), L.ptr(event_feat), L.ptr(frame_feat), L.ptr(conv_weight),
                    L.ptr(conv_bias), float(negative_slope), L.ptr(grad_output),
                    L.ptr(grad_pre), L.ptr(grad_event_fac), L.ptr(grad_bias),
                    B, Ce, Cf, H, W, K, L.ptr(ws), nbytes), what)
    return grad_pre, grad_event_fac, grad_bias


class KernelConvFACFunction(torch.autograd.Function):
    """out = KernelConv2D(K)(event, LeakyReLU(conv3x3(cat([event, frame], 1)))) with a fused forward AND backward.

    Saves only the four inputs. Backward: ebfi_kpn_fused_backward recomputes the pre-activation (bf16 conv operands,
    as in the forward) and writes dL/dP, dL/dbias and the FAC part of dL/devent; the conv's weight and input gradients
    are torch's convolution backward of dL/dP under the same torch/cuDNN settings as the reference's nn.Conv2d (TF32
    by default). fp32 CUDA tensors only."""

    @staticmethod
    def forward(ctx, event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope=0.01):
        L.require_cuda(event_feat, frame_feat, conv_weight, conv_bias)
        L.require_f32(event_feat=event_feat, frame_feat=frame_feat, conv_weight=conv_weight, conv_bias=conv_bias)
        ctx.kernel_size, ctx.negative_slope = int(kernel_size), float(negative_slope)
        ctx.save_for_backward(event_feat, frame_feat, conv_weight, conv_bias)
        return _fused_forward(event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope)

    @staticmethod
    def backward(ctx, grad_output):
        ev, fr, w, b = ctx.saved_tensors
        need_ev, need_fr, need_w, need_b = ctx.needs_input_grad[:4]
        grad_pre, grad_ev, grad_b = kernelconv_fac_fused_backward(ev, fr, w, b, ctx.kernel_size, ctx.negative_slope,
                                                                  grad_output)
        need_x = need_ev or need_fr
        grad_x = grad_w = grad_fr = None
        if need_x or need_w:
            x = torch.cat([ev, fr], 1) if fr.shape[1] else ev
            grad_x, grad_w, _ = torch.ops.aten.convolution_backward(
                grad_pre, x, w, None, [1, 1], [1, 1], [1, 1], False, [0, 0], 1, [need_x, need_w, False])
        if need_x:
            Ce = ev.shape[1]
            grad_ev = grad_ev + grad_x[:, :Ce]
            grad_fr = grad_x[:, Ce:] if need_fr else None
        return (grad_ev if need_ev else None, grad_fr, grad_w if need_w else None, grad_b if need_b else None,
                None, None)


class KernelConvFACBF16Function(torch.autograd.Function):
    """KernelConvFACFunction for 16-bit activations, as torch.autocast feeds the block (dtype=torch.bfloat16, or its
    default torch.float16): event_feat and frame_feat both bf16 or both fp16; conv_weight and conv_bias fp32 (autocast
    parameters) or of the activations' type (a .bfloat16() / .half() model); all CUDA. Returns the activations' type.

    Saves only the four inputs. The forward and the fused backward kernel read the 16-bit activations and use the
    weights as fp32 (exact for 16-bit ones); P and LeakyReLU(P) stay fp32 in registers, the output and dL/dP are
    rounded once to the 16-bit type. The conv's weight and input gradients are the 16-bit convolution backward of
    dL/dP that autocast's nn.Conv2d runs (16-bit cat(event, frame) and weight). grad_event = (FAC part + conv part)
    summed in fp32 and rounded once; weight and bias gradients come back in the parameters' dtype. The backward does
    not depend on the autocast state it runs under."""

    @staticmethod
    def forward(ctx, event_feat, frame_feat, conv_weight, conv_bias, kernel_size, negative_slope=0.01):
        L.require_cuda(event_feat, frame_feat, conv_weight, conv_bias)
        _require_half_io("KernelConvFACBF16Function", dict(event_feat=event_feat, frame_feat=frame_feat),
                         dict(conv_weight=conv_weight, conv_bias=conv_bias))
        ctx.kernel_size, ctx.negative_slope = int(kernel_size), float(negative_slope)
        ctx.save_for_backward(event_feat, frame_feat, conv_weight, conv_bias)
        return _fused_forward(event_feat, frame_feat, conv_weight.float(), conv_bias.float(), kernel_size,
                              negative_slope)

    @staticmethod
    def backward(ctx, grad_output):
        ev, fr, w, b = ctx.saved_tensors
        need_ev, need_fr, need_w, need_b = ctx.needs_input_grad[:4]
        half = ev.dtype
        with torch.autocast("cuda", enabled=False):
            grad_pre, grad_ev, grad_b = kernelconv_fac_fused_backward_bf16(
                ev, fr, w, b, ctx.kernel_size, ctx.negative_slope, grad_output.to(half))
            need_x = need_ev or need_fr
            grad_x = grad_w = grad_fr = None
            if need_x or need_w:
                x = torch.cat([ev, fr], 1) if fr.shape[1] else ev
                grad_x, grad_w, _ = torch.ops.aten.convolution_backward(
                    grad_pre, x, w.to(half), None, [1, 1], [1, 1], [1, 1], False, [0, 0], 1, [need_x, need_w, False])
            if need_x:
                Ce = ev.shape[1]
                grad_ev = (grad_ev + grad_x[:, :Ce].float()).to(half)
                grad_fr = grad_x[:, Ce:] if need_fr else None
        return (grad_ev if need_ev else None, grad_fr, grad_w.to(w.dtype) if need_w else None,
                grad_b.to(b.dtype) if need_b else None, None, None)


def kernelconv_fac_fused_supported(channels_event, channels_frame, kernel_size):
    """Shapes `ebfi_kpn_fused_forward` accepts (csrc/kpn.cu `fill`): odd K <= 5, (Ce + Cf) a multiple of 32 and <= 128."""
    K, cin = int(kernel_size), int(channels_event) + int(channels_frame)
    return K >= 1 and K % 2 == 1 and K <= 5 and cin % 32 == 0 and cin <= 128


class _ConvLayer(nn.Module):
    """ConvLayer(norm=None, activation='LeakyReLU') of models/model_misc/submodules.py:159-200: parameter names
    `conv2d.weight`, `conv2d.bias` as in the reference's checkpoints."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv2d = nn.Conv2d(in_channels, out_channels, 3, 1, 1, bias=True)
        self.activation = nn.LeakyReLU()

    def forward(self, x):
        return self.activation(self.conv2d(x))


class KernelPrediction(nn.Module):
    """`KernelConv` + `KPN` of Modification (model_singleframe.py:145-146,161-162): forward(EventTensor, FrameTensor)
    -> KPN(EventTensor, KernelConv(cat([EventTensor, FrameTensor], 1))).

    `fused = True` (class or instance attribute, like `DCN.fused`): when no gradient is needed and the shape is one the
    fused kernel supports, producer and consumer run as one kernel whose conv operands are rounded to bf16 — eval
    outputs then differ from the training / reference path (cuDNN TF32 or fp32 conv) by up to 1e-2 of max|out|
    (bound tested in tests/test_kpn_gpu.py; measured 1.5e-3). Set `fused = False` for the reference's op sequence
    in every mode. Unsupported shapes (e.g. FrameBasech = 24 or 96, KernelSize = 7) always take that sequence.

    `fused_backward = False` (class or instance attribute): when True and a gradient is needed, fp32 CUDA tensors of
    a supported shape train through `KernelConvFACFunction` (fused forward and backward; nothing but the inputs is
    kept for the backward). Opt-in because it changes training precision: the pre-activation comes from bf16 conv
    operands, so the gradients differ more from the fp64 op sequence than the TF32 reference sequence's do (measured
    ratio in DESIGN §3). With event and frame tensors both bf16 or both fp16 (torch.autocast mixed precision, or a
    .bfloat16() / .half() model) and parameters fp32 or of that type, the same opt-in trains through
    `KernelConvFACBF16Function` instead: 16-bit activation I/O, P and the kernel tensor in fp32 registers, the conv's
    gradients as autocast's 16-bit convolution backward (precision and measured numbers in DESIGN §3). Every other case
    does exactly what it does with `fused_backward = False`."""

    fused = True
    fused_backward = False

    def __init__(self, FrameBasech=64, KernelSize=5):
        super().__init__()
        self.KernelConv = _ConvLayer(FrameBasech + FrameBasech, FrameBasech * KernelSize ** 2)
        self.KPN = KernelConv2D(kernel_size=KernelSize)
        self.kernel_size = KernelSize

    def forward(self, EventTensor, FrameTensor):
        conv = self.KernelConv.conv2d
        needs_grad = torch.is_grad_enabled() and (EventTensor.requires_grad or FrameTensor.requires_grad
                                                  or conv.weight.requires_grad)
        if self.fused and not needs_grad and EventTensor.is_cuda and EventTensor.dtype in _SUFFIX \
                and FrameTensor.dtype == EventTensor.dtype and conv.weight.dtype == EventTensor.dtype \
                and kernelconv_fac_fused_supported(EventTensor.shape[1], FrameTensor.shape[1], self.kernel_size):
            return kernelconv_fac_fused(EventTensor, FrameTensor, conv.weight, conv.bias, self.kernel_size,
                                        self.KernelConv.activation.negative_slope)
        if self.fused_backward and needs_grad and EventTensor.is_cuda and EventTensor.dtype == torch.float32 \
                and FrameTensor.dtype == torch.float32 and conv.weight.dtype == torch.float32 \
                and kernelconv_fac_fused_supported(EventTensor.shape[1], FrameTensor.shape[1], self.kernel_size):
            return KernelConvFACFunction.apply(EventTensor, FrameTensor, conv.weight, conv.bias, self.kernel_size,
                                               self.KernelConv.activation.negative_slope)
        if self.fused_backward and needs_grad and EventTensor.is_cuda \
                and EventTensor.dtype in (torch.bfloat16, torch.float16) and FrameTensor.dtype == EventTensor.dtype \
                and conv.weight.dtype in (torch.float32, EventTensor.dtype) \
                and conv.bias.dtype == conv.weight.dtype \
                and kernelconv_fac_fused_supported(EventTensor.shape[1], FrameTensor.shape[1], self.kernel_size):
            return KernelConvFACBF16Function.apply(EventTensor, FrameTensor, conv.weight, conv.bias, self.kernel_size,
                                                   self.KernelConv.activation.negative_slope)
        Kernel = self.KernelConv(torch.cat([EventTensor, FrameTensor], dim=1))
        return self.KPN(EventTensor, Kernel)
