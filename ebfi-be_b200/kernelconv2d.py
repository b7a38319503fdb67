"""Host-side mirror of the reference's FAC operator interface
(models/FAC/kernelconv2d/KernelConv2D.py): `KernelConv2DFunction` (:12-58) and the
`KernelConv2D` module (:77-87), on top of the sm_100a kernels.

Kept from the reference: contiguity asserts (:19-20), the K == sqrt(C_k/C) and
H_in - K == H_out - 1 asserts (:22,:31-32), NotImplementedError for CPU tensors (:38-39,:55-56).
Dropped: the zero fill of output / grad_input / grad_kernel (:35,:50-51) — 1.7 GB of pure
memset at the benchmark shape; the kernels write every element.

The module folds its ReplicationPad2d into the kernels (`KernelConv2DReplPadFunction`): no padded copy of the
input is written, saved or read, and the backward sums the pad's gradient in a fixed order without atomics (ATen's
CUDA pad backward accumulates with atomics and raises under torch.use_deterministic_algorithms(True)), so the
module trains bit-reproducibly, with or without that switch.
"""
import torch
from torch import nn
from torch.autograd import Function

from . import _lib as L
from .shims import kernelconv2d_cuda
from .shims.kernelconv2d_cuda import _SUFFIX


class KernelConv2DFunction(Function):
    @staticmethod
    def forward(ctx, input, kernel, kernel_size):
        assert input.is_contiguous()
        assert kernel.is_contiguous()
        assert kernel_size == int((kernel.size(1) / input.size(1)) ** 0.5)
        assert input.size(2) - kernel_size == kernel.size(2) - 1
        assert input.size(3) - kernel_size == kernel.size(3) - 1
        if not input.is_cuda:
            raise NotImplementedError()      # CPU VERSION NOT IMPLEMENTED (KernelConv2D.py:38-39)
        ctx.kernel_size = kernel_size
        ctx.save_for_backward(input, kernel)
        with torch.cuda.device_of(input):
            output = torch.empty((input.size(0), input.size(1), kernel.size(2), kernel.size(3)),
                                 dtype=input.dtype, device=input.device)
            kernelconv2d_cuda.forward(input, kernel, kernel_size, output)
        return output

    @staticmethod
    def backward(ctx, grad_output):
        input, kernel = ctx.saved_tensors
        grad_output = grad_output.contiguous()
        if not grad_output.is_cuda:
            raise NotImplementedError()      # KernelConv2D.py:55-56
        with torch.cuda.device_of(input):
            grad_input, grad_kernel = torch.empty_like(input), torch.empty_like(kernel)
            kernelconv2d_cuda.backward(input, kernel, ctx.kernel_size, grad_output, grad_input, grad_kernel)
        return grad_input, grad_kernel, None


def _replpad_dims(input, kernel, kernel_size):
    if input.dtype not in _SUFFIX or kernel.dtype != input.dtype:
        raise RuntimeError(f"KernelConv2D: input and kernel must both be float32, both bfloat16 or both float16, "
                           f"got {input.dtype} / {kernel.dtype}")
    K = int(kernel_size)
    if input.dim() != 4 or kernel.dim() != 4 or kernel.shape[0] != input.shape[0] or \
            kernel.shape[1] != input.shape[1] * K * K or kernel.shape[2:] != input.shape[2:]:
        raise RuntimeError(f"KernelConv2D: shapes input {tuple(input.shape)} / kernel {tuple(kernel.shape)} "
                           f"do not fit kernel_size {K}")
    return (*input.shape, K)


class KernelConv2DReplPadFunction(Function):
    """ReplicationPad2d((K-1)/2)(input) followed by KernelConv2DFunction, with the pad folded into the kernels:
    input (B, C, H, W), kernel (B, C*K*K, H, W). Saves only input and kernel. Forward and grad_kernel are
    bit-identical to the padded sequence; grad_input is the pad's gradient summed in a fixed order (fp32)."""

    @staticmethod
    def forward(ctx, input, kernel, kernel_size):
        if not (input.is_cuda and kernel.is_cuda):
            raise NotImplementedError()      # CPU VERSION NOT IMPLEMENTED (KernelConv2D.py:38-39)
        input, kernel = input.contiguous(), kernel.contiguous()
        B, C, H, W, K = _replpad_dims(input, kernel, kernel_size)
        ctx.kernel_size = K
        ctx.save_for_backward(input, kernel)
        lib = L.load()
        with torch.cuda.device_of(input):
            output = torch.empty((B, C, H, W), dtype=input.dtype, device=input.device)
            fn = getattr(lib, "ebfi_fac_replpad_forward" + _SUFFIX[input.dtype])
            L.check(fn(L.stream_ptr(input.device), L.ptr(input), L.ptr(kernel), L.ptr(output), B, C, H, W, K),
                    "ebfi_fac_replpad_forward")
        return output

    @staticmethod
    def backward(ctx, grad_output):
        input, kernel = ctx.saved_tensors
        if not grad_output.is_cuda:
            raise NotImplementedError()      # KernelConv2D.py:55-56
        grad_output = grad_output.contiguous()
        if grad_output.dtype != input.dtype:
            raise RuntimeError(f"KernelConv2D: grad_output is {grad_output.dtype}, the input {input.dtype}")
        B, C, H, W, K = _replpad_dims(input, kernel, ctx.kernel_size)
        lib = L.load()
        with torch.cuda.device_of(input):
            grad_input, grad_kernel = torch.empty_like(input), torch.empty_like(kernel)
            nbytes = lib.ebfi_fac_backward_workspace_bytes(B, C, H, W, K)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
            fn = getattr(lib, "ebfi_fac_replpad_backward" + _SUFFIX[input.dtype])
            L.check(fn(L.stream_ptr(input.device), L.ptr(input), L.ptr(kernel), L.ptr(grad_output),
                       L.ptr(grad_input), L.ptr(grad_kernel), B, C, H, W, K, L.ptr(ws), nbytes),
                    "ebfi_fac_replpad_backward")
        return grad_input, grad_kernel, None


class KernelConv2D(nn.Module):
    """ReplicationPad2d((K-1)/2) followed by the per-pixel K x K filter (KernelConv2D.py:77-87), the pad folded
    into the kernels. No parameters or buffers: the reference's checkpoints load unchanged."""

    def __init__(self, kernel_size):
        super().__init__()
        assert kernel_size % 2 == 1
        self.kernel_size = kernel_size

    def forward(self, input, kernel):
        return KernelConv2DReplPadFunction.apply(input, kernel, self.kernel_size)
