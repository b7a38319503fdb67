"""Host-side mirror of the reference's DCNv2 operator interface (models/DCNv2/dcn_v2.py).

Same names, argument meaning and error behaviour for the convolution classes that EBFI-BE
uses — `_DCNv2` / `dcn_v2_conv` (dcn_v2.py:17-95), `DCNv2` (:98-146), `DCN` (:149-194),
`DCN_sep` (:197-227) — on top of the sm_100a kernels. The pooling classes (:230-435) are
out of scope. The reference file itself also runs unchanged once `ebfi_be_b200.shims` is on
sys.path; this module exists so the operator can be used and tested where /root/reference
is absent.
"""
import logging
import math
import threading

import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.nn.modules.utils import _pair

from .shims import _ext as _backend

logger = logging.getLogger("base")


def _as_dtypes(grads, tensors):
    """Gradients in the dtype of the tensor each one belongs to (bf16 / fp16 calls return 16-bit activation gradients;
    under autocast an input can be fp32)."""
    return tuple(gr.to(t.dtype) for gr, t in zip(grads, tensors))


class _DCNv2(Function):
    """Modulated deformable convolution; arguments as dcn_v2.py:18-21. bf16 or fp16 tensors, also mixed with fp32 ones
    (autocast), follow shims/_ext.py: the output is 16-bit, each gradient has its input's dtype."""

    @staticmethod
    def forward(ctx, input, offset, mask, weight, bias, stride, padding, dilation, deformable_groups):
        ctx.stride, ctx.padding, ctx.dilation = _pair(stride), _pair(padding), _pair(dilation)
        ctx.kernel_size = _pair(weight.shape[2:4])
        ctx.deformable_groups = deformable_groups
        out = _backend.dcn_v2_forward(input, weight, bias, offset, mask, *ctx.kernel_size,
                                      *ctx.stride, *ctx.padding, *ctx.dilation, deformable_groups)
        ctx.save_for_backward(input, offset, mask, weight, bias)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        input, offset, mask, weight, bias = ctx.saved_tensors
        g_in, g_off, g_mask, g_w, g_b = _backend.dcn_v2_backward(
            input, weight, bias, offset, mask, grad_output, *ctx.kernel_size, *ctx.stride,
            *ctx.padding, *ctx.dilation, ctx.deformable_groups)
        return (*_as_dtypes((g_in, g_off, g_mask, g_w, g_b), (input, offset, mask, weight, bias)),
                None, None, None, None)


dcn_v2_conv = _DCNv2.apply


class _DCNv2Packed(Function):
    """dcn_v2_conv(input, cat(o1, o2), sigmoid(mask), ...) with (o1, o2, mask) = chunk(offset_mask, 3, 1)
    (dcn_v2.py:217-227) as ONE op: the kernels read the raw conv output and apply the sigmoid themselves,
    the backward returns one gradient of the same layout. `stat` (optional 1-element fp32 CUDA tensor)
    receives sum |offset|."""

    @staticmethod
    def forward(ctx, input, offset_mask, weight, bias, stride, padding, dilation, deformable_groups, stat):
        ctx.stride, ctx.padding, ctx.dilation = _pair(stride), _pair(padding), _pair(dilation)
        ctx.kernel_size = _pair(weight.shape[2:4])
        ctx.deformable_groups = deformable_groups
        out = _backend.dcn_v2_forward_packed(input, weight, bias, offset_mask, *ctx.kernel_size, *ctx.stride,
                                             *ctx.padding, *ctx.dilation, deformable_groups, stat)
        ctx.save_for_backward(input, offset_mask, weight, bias)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        input, offset_mask, weight, bias = ctx.saved_tensors
        g_in, g_om, g_w, g_b = _backend.dcn_v2_backward_packed(
            input, weight, bias, offset_mask, grad_output, *ctx.kernel_size, *ctx.stride,
            *ctx.padding, *ctx.dilation, ctx.deformable_groups)
        return (*_as_dtypes((g_in, g_om, g_w, g_b), (input, offset_mask, weight, bias)),
                None, None, None, None, None)


def dcn_v2_conv_packed(input, offset_mask, weight, bias, stride, padding, dilation, deformable_groups, stat=None):
    return _DCNv2Packed.apply(input, offset_mask, weight, bias, stride, padding, dilation, deformable_groups, stat)


class DCNv2(nn.Module):
    """Parameters and init as dcn_v2.py:98-128: weight ~ U(-1/sqrt(C*kh*kw), +), bias = 0."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation=1,
                 deformable_groups=1):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride = _pair(kernel_size), _pair(stride)
        self.padding, self.dilation = _pair(padding), _pair(dilation)
        self.deformable_groups = deformable_groups
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels, *self.kernel_size))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1.0 / math.sqrt(self.in_channels * self.kernel_size[0] * self.kernel_size[1])
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)
            self.bias.zero_()

    def _taps(self):
        return self.deformable_groups * self.kernel_size[0] * self.kernel_size[1]

    def forward(self, input, offset, mask):
        assert 2 * self._taps() == offset.shape[1]      # dcn_v2.py:131-135
        assert self._taps() == mask.shape[1]
        return dcn_v2_conv(input, offset, mask, self.weight, self.bias, self.stride, self.padding,
                           self.dilation, self.deformable_groups)


class _DCNWithOffsetConv(DCNv2):
    """Shared part of DCN / DCN_sep: a zero-initialised conv predicting 3*dg*kh*kw channels that
    are split into (o1, o2, mask); offset = cat(o1, o2), mask = sigmoid(mask) (dcn_v2.py:163-183)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.conv_offset_mask = nn.Conv2d(self.in_channels, 3 * self._taps(), kernel_size=self.kernel_size,
                                          stride=self.stride, padding=self.padding, bias=True)
        self.init_offset()

    def init_offset(self):
        with torch.no_grad():
            self.conv_offset_mask.weight.zero_()
            self.conv_offset_mask.bias.zero_()

    def _offset_mask(self, features):
        o1, o2, mask = torch.chunk(self.conv_offset_mask(features), 3, dim=1)
        return torch.cat((o1, o2), dim=1), mask


class DCN(_DCNWithOffsetConv):
    """`fused=True` (default) feeds the conv output straight to the packed kernels; `fused=False` runs
    the reference's op sequence chunk -> cat -> sigmoid -> dcn_v2_conv (dcn_v2.py:179-187)."""
    fused = True

    def forward(self, input):
        if self.fused and input.is_cuda:
            return dcn_v2_conv_packed(input, self.conv_offset_mask(input), self.weight, self.bias, self.stride,
                                      self.padding, self.dilation, self.deformable_groups)
        offset, mask = self._offset_mask(input)
        return dcn_v2_conv(input, offset, torch.sigmoid(mask), self.weight, self.bias, self.stride,
                           self.padding, self.dilation, self.deformable_groups)


class _OffsetWatch:
    """The reference's `if offset_mean > 100: logger.warning(...)` (dcn_v2.py:221-223) forces a host
    sync in every forward. Here the kernel accumulates sum |offset| on the device; the value is copied
    to pinned memory asynchronously and examined when it has arrived (at the next forward of the module,
    or on `flush()`), so the warning is the same but may be logged one call late."""

    def __init__(self):
        self._pending = []          # (event, pinned value, element count)
        self._free = []             # pinned 1-float buffers, reused (cudaHostAlloc is slow)
        self._lock = threading.Lock()   # nn.DataParallel replicas share the module attribute across threads

    # CUDA events and pinned buffers are per-process runtime state: copies (copy.deepcopy for EMA models,
    # torch.save(model), DataParallel replicas) start with a fresh, empty watcher — pending warnings stay with the original
    def __getstate__(self):
        return {}

    def __setstate__(self, state):
        self.__init__()

    def __deepcopy__(self, memo):
        return _OffsetWatch()

    def submit(self, stat, count):
        with self._lock:
            host = self._free.pop() if self._free else torch.empty(1, dtype=torch.float32, pin_memory=True)
        host.copy_(stat, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        with self._lock:
            self._pending.append((ev, host, count))

    def poll(self, wait=False):
        with self._lock:
            pending, self._pending = self._pending, []
        keep = []
        for ev, host, count in pending:
            if wait:
                ev.synchronize()
            if ev.query():
                mean = float(host[0]) / count
                if mean > 100:
                    logger.warning("Offset mean is {}, larger than 100.".format(mean))
                with self._lock:
                    self._free.append(host)
            else:
                keep.append((ev, host, count))
        with self._lock:
            self._pending = keep + self._pending

    def flush(self):
        self.poll(wait=True)


class DCN_sep(_DCNWithOffsetConv):
    """Offsets and masks come from a second feature map `fea` (dcn_v2.py:197-227). `fused=False` runs
    the reference's op sequence including its per-call host sync. Under torch.compile the fused path does not
    evaluate the `offset mean > 100` warning: its pinned copies and events are host work outside the graph."""
    fused = True

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._watch = _OffsetWatch()

    def flush_offset_warnings(self):
        self._watch.flush()

    def forward(self, input, fea):
        if self.fused and input.is_cuda:
            om = self.conv_offset_mask(fea)
            if torch.compiler.is_compiling():
                return dcn_v2_conv_packed(input, om, self.weight, self.bias, self.stride, self.padding,
                                          self.dilation, self.deformable_groups)
            self._watch.poll()
            stat = torch.empty(1, dtype=torch.float32, device=input.device)
            out = dcn_v2_conv_packed(input, om, self.weight, self.bias, self.stride, self.padding,
                                     self.dilation, self.deformable_groups, stat)
            self._watch.submit(stat, om.numel() // 3 * 2)
            return out
        offset, mask = self._offset_mask(fea)
        offset_mean = torch.mean(torch.abs(offset))
        if offset_mean > 100:                           # host sync, as in the reference (:221-223)
            logger.warning("Offset mean is {}, larger than 100.".format(offset_mean))
        return dcn_v2_conv(input, offset, torch.sigmoid(mask), self.weight, self.bias, self.stride,
                           self.padding, self.dilation, self.deformable_groups)
