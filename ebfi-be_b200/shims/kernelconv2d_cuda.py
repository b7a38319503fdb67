"""`kernelconv2d_cuda` — same two functions as the reference's pybind module
(models/FAC/kernelconv2d/KernelConv2D_cuda.cpp:10-61), backed by libebfi_b200.so.

forward(input, kernel, kernel_size, output) -> 1 and
backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel) -> 1 write into the
caller-allocated tensors like the reference; a failing launch raises RuntimeError (the
reference's AT_ERROR("CUDA call failed"), KernelConv2D_cuda.cpp:26-28). Under torch.compile they run as
torch.ops.ebfi_b200.fac_forward / fac_backward, which declare those writes.
"""
import torch

try:
    from ebfi_be_b200 import _lib as L
except ImportError:  # shims directory used stand-alone on sys.path
    import os as _os
    import sys as _sys
    _sys.path.insert(0, _os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))))
    from ebfi_be_b200 import _lib as L


# dtype -> suffix of the C entries (bf16 / fp16: storage only, fp32 arithmetic)
_SUFFIX = {torch.float32: "", torch.bfloat16: "_bf16", torch.float16: "_fp16"}


def _dims(input, kernel, kernel_size, what):
    L.require_cuda(input, kernel)
    if input.dtype not in _SUFFIX or kernel.dtype != input.dtype:
        raise RuntimeError(f"{what}: input and kernel must both be float32 (the reference's dtype), both "
                           f"bfloat16 or both float16, got {input.dtype} / {kernel.dtype}")
    if input.dim() != 4 or kernel.dim() != 4:
        raise RuntimeError(f"{what}: input and kernel must be 4-D")
    B, C, Hi, Wi = input.shape
    K = int(kernel_size)
    H, W = kernel.shape[2], kernel.shape[3]
    if kernel.shape[0] != B or kernel.shape[1] != C * K * K or Hi != H + K - 1 or Wi != W + K - 1:
        raise RuntimeError(f"{what}: shapes input {tuple(input.shape)} / kernel {tuple(kernel.shape)} "
                           f"do not fit kernel_size {K}")
    if not (input.is_contiguous() and kernel.is_contiguous()):
        raise RuntimeError(f"{what}: input and kernel must be contiguous")   # KernelConv2D.py:19-20
    return B, C, H, W, K


def _check_forward(input, kernel, kernel_size, output):
    B, C, H, W, K = _dims(input, kernel, kernel_size, "kernelconv2d_cuda.forward")
    if tuple(output.shape) != (B, C, H, W) or not output.is_contiguous() or output.dtype != input.dtype:
        raise RuntimeError("kernelconv2d_cuda.forward: output must be a contiguous (B, C, H, W) tensor of the input dtype")
    return B, C, H, W, K


def forward(input, kernel, kernel_size, output):
    if torch.compiler.is_compiling():
        torch.ops.ebfi_b200.fac_forward(input, kernel, kernel_size, output)
        return 1
    B, C, H, W, K = _check_forward(input, kernel, kernel_size, output)
    lib = L.load()
    fn = getattr(lib, "ebfi_fac_forward" + _SUFFIX[input.dtype])
    with torch.cuda.device(input.device):
        L.check(fn(L.stream_ptr(input.device), L.ptr(input), L.ptr(kernel), L.ptr(output), B, C, H, W, K), "CUDA call")
    return 1


def _check_backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel):
    B, C, H, W, K = _dims(input, kernel, kernel_size, "kernelconv2d_cuda.backward")
    L.require_cuda(grad_output, grad_input, grad_kernel)
    if tuple(grad_output.shape) != (B, C, H, W) or not grad_output.is_contiguous() or grad_output.dtype != input.dtype:
        raise RuntimeError("kernelconv2d_cuda.backward: grad_output must be contiguous (B, C, H, W) of the input dtype")
    if grad_input.dtype != input.dtype or grad_kernel.dtype != input.dtype:
        raise RuntimeError("kernelconv2d_cuda.backward: gradients must have the input dtype")
    if grad_input.shape != input.shape or grad_kernel.shape != kernel.shape or \
            not grad_input.is_contiguous() or not grad_kernel.is_contiguous():
        raise RuntimeError("kernelconv2d_cuda.backward: grad_input / grad_kernel must match input / kernel")
    return B, C, H, W, K


def backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel):
    if torch.compiler.is_compiling():
        torch.ops.ebfi_b200.fac_backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel)
        return 1
    B, C, H, W, K = _check_backward(input, kernel, kernel_size, grad_output, grad_input, grad_kernel)
    lib = L.load()
    with torch.cuda.device(input.device):
        nbytes = lib.ebfi_fac_backward_workspace_bytes(B, C, H, W, K)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        fn = getattr(lib, "ebfi_fac_backward" + _SUFFIX[input.dtype])
        L.check(fn(L.stream_ptr(input.device), L.ptr(input), L.ptr(kernel), L.ptr(grad_output), L.ptr(grad_input),
                   L.ptr(grad_kernel), B, C, H, W, K, L.ptr(ws), nbytes), "CUDA call")
    return 1
