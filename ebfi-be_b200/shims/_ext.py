"""`_ext` — same functions, argument order and error behaviour as the reference's pybind module
(models/DCNv2/src/vision.cpp:4-9, src/dcn_v2.h:9-92), backed by libebfi_b200.so.

Differences, all deliberate:
  * CUDA only. The reference dispatches CPU tensors to dcn_v2_cpu_* (dcn_v2.h:35-44), whose
    forward returns uninitialised memory (cpu/dcn_v2_cpu.cpp:65,127); here a CPU tensor raises.
  * 16-bit floats, bf16 or fp16 (new; the reference is fp32-only). Activations (input, offset, mask / offset_mask,
    grad_output) of one 16-bit type — all of them, or some with the rest fp32, as under torch.autocast — run in that
    type: fp32 activations are rounded to it once (autocast's own cast). weight / bias may then be fp32 or of that type
    and are used as fp32. Outputs and activation gradients have the 16-bit type, grad_weight / grad_bias the
    parameter's dtype. The tensor-core kernels read and write the 16-bit activations directly, the backward's box
    kernel in the deterministic mode too; every other call (the CUDA-core kernels: other shapes or EBFI_DCN_IMPL=simt;
    the deterministic backward of footprints beyond the box; a misaligned grad_output) converts at this boundary
    (_via_fp32) with the same result dtypes. Both give the bits of the fp32 kernels on the widened values, rounded
    once; an fp16 result beyond the fp16 range is inf, as tensor.half() gives. bf16 mixed with fp16 raises. With fp32
    activations everything must be fp32, as in the reference.
  * the deformable PS-ROI pooling pair (dcn_v2.h:94-190) is out of scope and raises
    NotImplementedError (it is never imported by EBFI-BE).
"""
import functools
import os

import torch

try:
    from ebfi_be_b200 import _lib as L
except ImportError:  # shims directory used stand-alone on sys.path
    import importlib.util as _u
    import os as _os
    import sys as _sys
    _root = _os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))))
    _sys.path.insert(0, _root)
    from ebfi_be_b200 import _lib as L


def _deterministic():
    """Deterministic backward (new; the reference's col2im atomics are not reproducible, im2col_cuda.cu:249):
    follows torch.use_deterministic_algorithms(True), or EBFI_DCN_DETERMINISTIC=1."""
    return (L.EBFI_DCN_DETERMINISTIC
            if (torch.are_deterministic_algorithms_enabled() or os.environ.get("EBFI_DCN_DETERMINISTIC") == "1") else 0)


# The forward leaves a group-blocked copy of `input` in its workspace; the backward of the SAME tensor (same storage,
# same version counter, same geometry) reads it instead of re-blocking (EBFI_DCN_INPUT_BLOCKED). One entry per device:
# a training step runs backward right after forward; anything else simply misses and re-blocks. The entry holds the
# input's storage, so its address cannot be recycled for another tensor while the entry is alive.
_blocked_cache = {}


def _blocked_key(input, g):
    return (input.data_ptr(), input._version, tuple(input.shape), g.kernel_h, g.kernel_w, g.stride_h, g.stride_w,
            g.pad_h, g.pad_w, g.dilation_h, g.dilation_w, g.deformable_group)


def _remember_blocked(lib, g, input, ws):
    """After a forward: note where its workspace holds the group-blocked copy of `input`."""
    off_blk = lib.ebfi_dcnv2_blocked_input_offset(g)
    if off_blk and os.environ.get("EBFI_DCN_NO_BLOCKED_REUSE") != "1":
        # keeps `ws` alive until the next forward on this device; the stream that runs the backward is the one that
        # ran the forward in autograd (and in the reference's trainer), which orders the read after the write
        _blocked_cache[input.device.index] = (_blocked_key(input, g), ws, off_blk, torch.cuda.current_stream(input.device),
                                              input.untyped_storage())


def _blocked_input_ptr(g, input, grad_output):
    """Before a backward: the forward's blocked copy of this very tensor if it is still alive and this backward runs the
    box kernel that reads it (sets the geometry flag), else the tensor itself. The box kernel runs in both modes; it
    needs a 16-byte aligned grad_output and no EBFI_DCN_IMPL=simt, which may have changed since the forward."""
    hit = _blocked_cache.get(input.device.index)
    if (hit is not None and g.flags in (0, L.EBFI_DCN_DETERMINISTIC) and hit[0] == _blocked_key(input, g)
            and hit[3] == torch.cuda.current_stream(input.device) and grad_output.data_ptr() % 16 == 0
            and L.load().ebfi_dcnv2_blocked_input_offset(g) == hit[2]):
        g.flags |= L.EBFI_DCN_INPUT_BLOCKED
        return L.c_void(hit[1].data_ptr() + hit[2])
    return L.ptr(input)


def _geom(input, weight, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
          dilation_h, dilation_w, deformable_group, flags=0):
    if input.dim() != 4 or weight.dim() != 4:
        raise RuntimeError("dcn_v2: input and weight must be 4-D")
    channels_out, channels_kernel, kh_, kw_ = weight.shape
    # same two shape checks as dcn_v2_cuda.cu:58-62
    if kh_ != kernel_h or kw_ != kernel_w:
        raise RuntimeError("Input shape and kernel shape wont match: (%d x %d vs %d x %d)."
                           % (kernel_h, kernel_w, kh_, kw_))
    if input.shape[1] != channels_kernel:
        raise RuntimeError("Input shape and kernel channels wont match: (%d vs %d)."
                           % (input.shape[1], channels_kernel))
    g = L.DcnGeom(input.shape[0], input.shape[1], input.shape[2], input.shape[3], channels_out,
                  kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                  deformable_group, flags)
    ho, wo = L.c_int(), L.c_int()
    L.check(L.load().ebfi_dcnv2_output_size(g, ho, wo), "dcn_v2 geometry")
    return g, ho.value, wo.value


_PARAMS = ("weight", "bias")


# 16-bit activation dtypes -> suffix of their C entries
_HALF = {torch.bfloat16: "_bf16", torch.float16: "_fp16"}


def _check_cuda(**named):
    """float32: every tensor is fp32 (the reference). bfloat16 / float16: the activations are of that type, or of it
    and fp32 mixed, and the parameters fp32 or of that type. Anything else (bf16 with fp16, fp64) raises."""
    for k, t in named.items():
        if not t.is_cuda:
            raise RuntimeError(f"{k} must be a CUDA tensor")   # AT_ASSERTM, dcn_v2_cuda.cu:38-42
    dts = {t.dtype for t in named.values()}
    acts = {t.dtype for k, t in named.items() if k not in _PARAMS}
    if dts == {torch.float32}:
        return torch.float32
    for half in _HALF:
        if half in acts and dts <= {torch.float32, half}:
            return half
    raise RuntimeError("dcn_v2: all tensors must be float32 (the reference's `using scalar_t = float`), or the "
                       "activations one 16-bit type (bfloat16 or float16) with parameters of it or float32, got "
                       f"{sorted(str(d) for d in dts)}")


def _via_fp32(dtype, fn, tensors, ints, out_dtypes=None):
    """16-bit activations at the boundary: the fp32 entry `fn` on exactly widened copies, results rounded once to
    `dtype` (or converted to `out_dtypes`, one per result). This is what a bf16 / fp16 call runs where the kernels have
    no native 16-bit I/O: the CUDA-core kernels (shapes outside the tensor-core ones, EBFI_DCN_IMPL=simt), the
    deterministic backward where the box kernel does not run (dcn_bwd_tc.cu), and a grad_output that is not 16-byte
    aligned. It costs extra elementwise passes, and the
    widened input is a new tensor, so a backward through here re-blocks it."""
    out = fn(*(t.float() for t in tensors), *ints)
    if torch.is_tensor(out):
        return out.to(out_dtypes[0] if out_dtypes else dtype)
    return [o.to(dt) for o, dt in zip(out, out_dtypes or [dtype] * len(out))]


_bf16_via_fp32 = functools.partial(_via_fp32, torch.bfloat16)


def _ran_native(rc, what):
    """True when a 16-bit entry ran; False when it declined the call (EBFI_ERR_UNSUPPORTED, nothing was enqueued)."""
    if rc == L.EBFI_ERR_UNSUPPORTED:
        return False
    L.check(rc, what)
    return True


def _check_offset_mask(g, ho, wo, offset, mask):
    kk = g.kernel_h * g.kernel_w
    want_o = (g.batch, 2 * g.deformable_group * kk, ho, wo)
    want_m = (g.batch, g.deformable_group * kk, ho, wo)
    if tuple(offset.shape) != want_o or tuple(mask.shape) != want_m:
        raise RuntimeError(f"dcn_v2: offset/mask shapes {tuple(offset.shape)}/{tuple(mask.shape)} "
                           f"do not match the geometry (expected {want_o}/{want_m})")


def dcn_v2_forward(input, weight, bias, offset, mask, kernel_h, kernel_w, stride_h, stride_w,
                   pad_h, pad_w, dilation_h, dilation_w, deformable_group):
    """dcn_v2_cuda_forward (src/cuda/dcn_v2_cuda.cu:20-95). Returns a new (B, Cout, Ho, Wo) tensor."""
    dt = _check_cuda(input=input, weight=weight, bias=bias, offset=offset, mask=mask)
    half = _HALF.get(dt)
    ints = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group)
    if half:
        input, offset, mask = (t.to(dt) for t in (input, offset, mask))
        weight, bias = weight.float(), bias.float()
    g, ho, wo = _geom(input, weight, *ints)
    _check_offset_mask(g, ho, wo, offset, mask)
    input, weight, bias, offset, mask = (t.contiguous() for t in (input, weight, bias, offset, mask))
    with torch.cuda.device(input.device):
        output = torch.empty((g.batch, g.channels_out, ho, wo), dtype=input.dtype, device=input.device)
        lib = L.load()
        nbytes = lib.ebfi_dcnv2_forward_workspace_bytes(g)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        args = (L.stream_ptr(input.device), g, L.ptr(input), L.ptr(weight), L.ptr(bias), L.ptr(offset), L.ptr(mask),
                L.ptr(output), L.ptr(ws), nbytes)
        if not half:
            L.check(lib.ebfi_dcnv2_forward(*args), "dcn_v2_forward")
        elif not _ran_native(getattr(lib, "ebfi_dcnv2_forward" + half)(*args), "dcn_v2_forward" + half):
            return _via_fp32(dt, dcn_v2_forward, (input, weight, bias, offset, mask), ints)
        _remember_blocked(lib, g, input, ws)
    return output


def dcn_v2_backward(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h,
                    stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group, comm=None, defer=False):
    """dcn_v2_cuda_backward (dcn_v2_cuda.cu:97-216).
    Returns [grad_input, grad_offset, grad_mask, grad_weight, grad_bias].
    comm (new, optional): a parallel.GradComm — grad_weight / grad_bias then come back summed over its ranks, the
    exchange fused into the kernel that reduces them (ebfi_dcnv2_backward_dp). defer=True: the kernel only publishes
    this rank's sums; `comm.complete(grad_weight, grad_bias)` finishes the exchange where the sums are needed."""
    # THArgCheck(input.is_contiguous()) / (weight.is_contiguous()), dcn_v2_cuda.cu:110-111
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")
    dt = _check_cuda(input=input, weight=weight, bias=bias, offset=offset, mask=mask, grad_output=grad_output)
    half = _HALF.get(dt)
    ints = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group)
    if half:
        input, offset, mask, grad_output = (t.to(dt) for t in (input, offset, mask, grad_output))
        param_dtypes = [weight.dtype, bias.dtype]
        weight, bias = weight.float(), bias.float()
    g, ho, wo = _geom(input, weight, *ints, _deterministic())
    _check_offset_mask(g, ho, wo, offset, mask)
    if tuple(grad_output.shape) != (g.batch, g.channels_out, ho, wo):
        raise RuntimeError("dcn_v2_backward: grad_output has the wrong shape")
    bias, offset, mask, grad_output = (t.contiguous() for t in (bias, offset, mask, grad_output))
    lib = L.load()
    with torch.cuda.device(input.device):
        grads = [torch.empty_like(t) for t in (input, offset, mask, weight, bias)]
        nbytes = lib.ebfi_dcnv2_backward_workspace_bytes(g)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        in_ptr = _blocked_input_ptr(g, input, grad_output)
        args = (L.stream_ptr(input.device), g, in_ptr, L.ptr(weight), L.ptr(bias), L.ptr(offset), L.ptr(mask),
                L.ptr(grad_output), *(L.ptr(t) for t in grads), L.ptr(ws), nbytes)
        if not half:
            if comm is None:
                L.check(lib.ebfi_dcnv2_backward(*args), "dcn_v2_backward")
            else:
                L.check(lib.ebfi_dcnv2_backward_dp(*args, comm.struct, 1 if defer else 0), "dcn_v2_backward_dp")
            return grads
        if comm is None:
            ran = _ran_native(getattr(lib, "ebfi_dcnv2_backward" + half)(*args), "dcn_v2_backward" + half)
        else:
            ran = _ran_native(getattr(lib, "ebfi_dcnv2_backward_dp" + half)(*args, comm.struct, 1 if defer else 0),
                              "dcn_v2_backward_dp" + half)
    out_dtypes = [dt] * 3 + param_dtypes
    if not ran:
        return _via_fp32(dt, dcn_v2_backward, (input, weight, bias, offset, mask, grad_output), ints + (comm, defer),
                         out_dtypes)
    return [t.to(dt) for t, dt in zip(grads, out_dtypes)]


def dcn_v2_backward_dp(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h,
                       stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group, comm, defer=False):
    """dcn_v2_backward with grad_weight / grad_bias all-reduced over `comm` inside the producing kernel."""
    return dcn_v2_backward(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h,
                           stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group, comm, defer)


def _check_packed(g, ho, wo, offset_mask):
    want = (g.batch, 3 * g.deformable_group * g.kernel_h * g.kernel_w, ho, wo)
    if tuple(offset_mask.shape) != want:
        raise RuntimeError(f"dcn_v2: offset_mask shape {tuple(offset_mask.shape)} does not match the geometry "
                           f"(expected {want})")


def dcn_v2_forward_packed(input, weight, bias, offset_mask, kernel_h, kernel_w, stride_h, stride_w,
                          pad_h, pad_w, dilation_h, dilation_w, deformable_group, abs_offset_sum=None):
    """NEW (no reference counterpart in `_ext`): dcn_v2_forward fed with the raw `conv_offset_mask`
    output, i.e. chunk / cat / sigmoid of DCN.forward / DCN_sep.forward (dcn_v2.py:179-187, :217-227)
    folded into the kernel. `abs_offset_sum`: optional 1-element fp32 CUDA tensor that receives
    sum |offset| (for the `offset_mean > 100` warning, :221-223)."""
    dt = _check_cuda(input=input, weight=weight, bias=bias, offset_mask=offset_mask)
    half = _HALF.get(dt)
    ints = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group)
    if half:
        input, offset_mask = input.to(dt), offset_mask.to(dt)
        weight, bias = weight.float(), bias.float()
    g, ho, wo = _geom(input, weight, *ints)
    _check_packed(g, ho, wo, offset_mask)
    if abs_offset_sum is not None and not (abs_offset_sum.is_cuda and abs_offset_sum.dtype == torch.float32
                                           and abs_offset_sum.numel() == 1):
        raise RuntimeError("dcn_v2_forward_packed: abs_offset_sum must be a 1-element float32 CUDA tensor")
    input, weight, bias, offset_mask = (t.contiguous() for t in (input, weight, bias, offset_mask))
    with torch.cuda.device(input.device):
        output = torch.empty((g.batch, g.channels_out, ho, wo), dtype=input.dtype, device=input.device)
        lib = L.load()
        nbytes = lib.ebfi_dcnv2_forward_workspace_bytes(g)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        args = (L.stream_ptr(input.device), g, L.ptr(input), L.ptr(weight), L.ptr(bias), L.ptr(offset_mask),
                L.ptr(output), L.ptr(abs_offset_sum) if abs_offset_sum is not None else None, L.ptr(ws), nbytes)
        if not half:
            L.check(lib.ebfi_dcnv2_forward_packed(*args), "dcn_v2_forward_packed")
        elif not _ran_native(getattr(lib, "ebfi_dcnv2_forward_packed" + half)(*args), "dcn_v2_forward_packed" + half):
            return _via_fp32(dt, dcn_v2_forward_packed, (input, weight, bias, offset_mask), ints + (abs_offset_sum,))
        _remember_blocked(lib, g, input, ws)
    return output


def dcn_v2_backward_packed(input, weight, bias, offset_mask, grad_output, kernel_h, kernel_w, stride_h,
                           stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group):
    """Backward of dcn_v2_forward_packed. Returns [grad_input, grad_offset_mask, grad_weight, grad_bias];
    grad_offset_mask has the layout of offset_mask, its last third already multiplied by sigmoid'."""
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")
    dt = _check_cuda(input=input, weight=weight, bias=bias, offset_mask=offset_mask, grad_output=grad_output)
    half = _HALF.get(dt)
    ints = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, deformable_group)
    if half:
        input, offset_mask, grad_output = (t.to(dt) for t in (input, offset_mask, grad_output))
        param_dtypes = [weight.dtype, bias.dtype]
        weight, bias = weight.float(), bias.float()
    g, ho, wo = _geom(input, weight, *ints, _deterministic())
    _check_packed(g, ho, wo, offset_mask)
    if tuple(grad_output.shape) != (g.batch, g.channels_out, ho, wo):
        raise RuntimeError("dcn_v2_backward_packed: grad_output has the wrong shape")
    bias, offset_mask, grad_output = (t.contiguous() for t in (bias, offset_mask, grad_output))
    lib = L.load()
    with torch.cuda.device(input.device):
        grads = [torch.empty_like(t) for t in (input, offset_mask, weight, bias)]
        nbytes = lib.ebfi_dcnv2_backward_workspace_bytes(g)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        in_ptr = _blocked_input_ptr(g, input, grad_output)
        args = (L.stream_ptr(input.device), g, in_ptr, L.ptr(weight), L.ptr(bias), L.ptr(offset_mask),
                L.ptr(grad_output), *(L.ptr(t) for t in grads), L.ptr(ws), nbytes)
        if not half:
            L.check(lib.ebfi_dcnv2_backward_packed(*args), "dcn_v2_backward_packed")
            return grads
        ran = _ran_native(getattr(lib, "ebfi_dcnv2_backward_packed" + half)(*args), "dcn_v2_backward_packed" + half)
    out_dtypes = [dt] * 2 + param_dtypes
    if not ran:
        return _via_fp32(dt, dcn_v2_backward_packed, (input, weight, bias, offset_mask, grad_output), ints, out_dtypes)
    return [t.to(dt) for t, dt in zip(grads, out_dtypes)]


def dcn_v2_psroi_pooling_forward(*args, **kwargs):
    raise NotImplementedError("deformable PS-ROI pooling is outside the EBFI-BE alignment hot path "
                              "(models/DCNv2/src/dcn_v2.h:94-145); not provided by ebfi_be_b200")


def dcn_v2_psroi_pooling_backward(*args, **kwargs):
    raise NotImplementedError("deformable PS-ROI pooling is outside the EBFI-BE alignment hot path "
                              "(models/DCNv2/src/dcn_v2.h:147-190); not provided by ebfi_be_b200")
