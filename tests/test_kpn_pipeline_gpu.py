"""The fused KernelConv -> FAC kernels (csrc/kpn.cu) where each persistent CTA walks several work items, compared
EXACTLY with float64: every halo-part count (Cin / 32 = 1..4), every occupancy of the last weight slice, CTA ranges
that cross weight slices and samples, ragged and tiny tiles (test_kpn_gpu.PIPELINE_SHAPES), and the full cfg2 size
with real conv weights. The inputs lie on the integer lattice of _lattice_case, on which the block's fp32 arithmetic
does not round at all, so any indexing, pipeline-phase, halo, weight-slice reload, box-fold or bias-collect error
fails the comparison, however few pixels it touches."""
import numpy as np
import pytest
import torch

import kpn_train_oracle as KO
from conftest import rel_err
from test_kpn_gpu import PIPELINE_SHAPES, kpn_work_split
from test_kpn_train_gpu import no_tf32  # noqa: F401  (fixture)

SLOPE = 0.25
BF16, F16 = torch.bfloat16, torch.float16


@pytest.fixture(scope="module")
def mod():
    from ebfi_be_b200 import modification
    return modification


def _lattice_case(rng, B, Ce, Cf, H, W, K):
    """(ev, fr, w, b, G) float32 on which the block is exact in fp32: event, frame and grad_output integers in
    [-2, 2], conv weights in {-1, 0, 1}, conv bias an integer + 1/2 in [-7.5, 7.5], used with negative_slope 0.25.

    - Every input is exactly representable in bf16 and fp16: the kernels' bf16 conv operands and 16-bit activations
      carry the same values as fp32.
    - P = conv + bias is an integer + 1/2, so |P| >= 1/2 and no LeakyReLU branch is ever in doubt (the backward needs
      no branch separation), and LeakyReLU(P) is a multiple of 1/8.
    - Every product and partial sum of out, grad_pre, the dL/dEpad boxes and their replication-pad fold, and grad_bias
      is a multiple of 1/8 below 2^21 in magnitude, even summed in absolute value at the full cfg2 size (B=4, 64+64
      channels, 256x256, K=5): fewer than 2^24 units of 1/8. fp32 therefore gives the float64 value in any summation
      order, and the kernels must equal the float64 restatements bit for bit."""
    def ints(lo, hi, shape):
        return rng.integers(lo, hi + 1, shape).astype(np.float32)
    ev = ints(-2, 2, (B, Ce, H, W))
    fr = ints(-2, 2, (B, Cf, H, W))
    w = ints(-1, 1, (Ce * K * K, Ce + Cf, 3, 3))
    b = ints(-8, 7, Ce * K * K) + np.float32(0.5)
    G = ints(-2, 2, (B, Ce, H, W))
    return ev, fr, w, b, G


def _mismatch(name, got, want, shape, kk=1, backward=False):
    """Failure message of an exact comparison: how many elements differ, and for the first few their (b, channel,
    y, x) with the work item (slice, tile) and the CTA that kpn_work_split assigns them. kk = K*K for grad_pre
    (one channel per tap), 1 for (B, Ce, H, W) results; grad_bias gives its column and slice."""
    got, want = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    bad = torch.nonzero(got != want).tolist()
    sp = kpn_work_split(shape, torch.cuda.get_device_properties(0).multi_processor_count, backward)
    where = []
    for idx in bad[:6]:
        if len(idx) == 1:
            where.append(f"column {idx[0]} (slice {idx[0] // kk // 3})")
            continue
        b, ch, y, x = idx
        s = ch // kk // 3
        item = s * sp["ntile"] + (b * sp["tiles_y"] + y // 16) * sp["tiles_x"] + x // 8
        where.append(f"{tuple(idx)}: {float(got[tuple(idx)])} != {float(want[tuple(idx)])}, item {item} "
                     f"(slice {s}), CTA {item // sp['per']}")
    return f"{name}: {len(bad)} of {want.numel()} elements differ at {shape}, per = {sp['per']}; " + "; ".join(where)


# ---------------------------------------------------------------- the work split the shapes are chosen for
def _check_coverage(sms):
    assert {s[-1] for s in PIPELINE_SHAPES} == {1, 3, 5}
    assert any(Cf == 0 for _, _, Cf, _, _, _ in PIPELINE_SHAPES) and any(Ce % 8 for _, Ce, _, _, _, _ in PIPELINE_SHAPES)
    assert any(H < K for _, _, _, H, _, K in PIPELINE_SHAPES) and any(W < 8 for _, _, _, _, W, _ in PIPELINE_SHAPES)
    assert any(H == W == 1 for _, _, _, H, W, _ in PIPELINE_SHAPES)
    for backward in (False, True):
        splits = [kpn_work_split(s, sms, backward) for s in PIPELINE_SHAPES]
        for npart in (1, 2, 3, 4):
            assert any(x["npart"] == npart and x["per"] >= 3 for x in splits), (npart, backward)
        assert any(x["per"] >= 6 and x["crosses_slice"] and x["crosses_sample"] for x in splits), backward
        assert {x["last"] for x in splits} == {1, 2, 3}, backward


# PIPELINE_SHAPES at 148 SMs: (npart, channels in the last slice, items per CTA, range crosses a slice, a sample)
SPLIT_AT_148 = [(3, 3, 3, True, True), (3, 3, 6, True, True), (3, 2, 2, False, False), (3, 1, 10, True, True),
                (2, 3, 3, False, False), (4, 2, 2, False, False), (4, 1, 3, True, True), (4, 1, 3, True, True),
                (1, 1, 3, True, True), (2, 2, 6, True, True), (2, 2, 3, False, False), (1, 1, 1, False, False),
                (1, 2, 1, False, False), (4, 1, 1, False, False), (4, 3, 10, True, True)]


def test_pipeline_shapes_cover_the_work_split_at_148_sms():
    for shape, want in zip(PIPELINE_SHAPES, SPLIT_AT_148, strict=True):
        for backward in (False, True):
            x = kpn_work_split(shape, 148, backward)
            assert (x["npart"], x["last"], x["per"], x["crosses_slice"], x["crosses_sample"]) == want, shape
    assert kpn_work_split((4, 64, 64, 256, 256, 5), 148)["per"] == 305
    _check_coverage(148)


@pytest.mark.gpu
def test_pipeline_shapes_cover_the_work_split_on_this_device():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for shape in PIPELINE_SHAPES:
        print(sms, "SMs", shape, kpn_work_split(shape, sms))
    _check_coverage(sms)


# ---------------------------------------------------------------- kernels at PIPELINE_SHAPES
@pytest.mark.gpu
@pytest.mark.parametrize("shape", PIPELINE_SHAPES)
def test_fp32_kernels_exact_on_the_lattice(mod, oracle, shape):
    from gpu_util import n, t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b, G = _lattice_case(np.random.default_rng(sum(shape)), *shape)
    with torch.no_grad():
        out = n(mod.kernelconv_fac_fused(t(ev), t(fr), t(w), t(b), K, SLOPE))
    want_out, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, SLOPE, bf16_operands=True)
    assert np.array_equal(out, want_out), _mismatch("out", out, want_out, shape)

    gpre, gev, gbias = (n(x) for x in mod.kernelconv_fac_fused_backward(t(ev), t(fr), t(w), t(b), K, SLOPE, t(G)))
    want_gev, _, _, want_gbias, want_gpre, _ = KO.backward_parts(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    assert np.array_equal(gpre, want_gpre), _mismatch("grad_pre", gpre, want_gpre, shape, K * K, True)
    assert np.array_equal(gev, want_gev), _mismatch("grad_event_fac", gev, want_gev, shape, 1, True)
    assert np.array_equal(gbias, want_gbias), _mismatch("grad_bias", gbias, want_gbias, shape, K * K, True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("shape", PIPELINE_SHAPES)
def test_16bit_kernels_equal_fp32_on_the_lattice(mod, shape, dtype):
    """The _bf16 / _fp16 entries on the same lattice inputs (exact in both types): out is the fp32 kernel's output
    rounded once; grad_pre (a multiple of 1/4 of magnitude <= 4, exact in both types), grad_event_fac and grad_bias
    are the fp32 kernel's."""
    from gpu_util import t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b, G = (t(a) for a in _lattice_case(np.random.default_rng(sum(shape)), *shape))
    with torch.no_grad():
        out32 = mod.kernelconv_fac_fused(ev, fr, w, b, K, SLOPE)
        out = mod.kernelconv_fac_fused(ev.to(dtype), fr.to(dtype), w.to(dtype), b.to(dtype), K, SLOPE)
    assert out.dtype == dtype
    assert torch.equal(out, out32.to(dtype)), _mismatch("out", out, out32.to(dtype), shape)
    want = mod.kernelconv_fac_fused_backward(ev, fr, w, b, K, SLOPE, G)
    got = mod.kernelconv_fac_fused_backward_bf16(ev.to(dtype), fr.to(dtype), w, b, K, SLOPE, G.to(dtype))
    assert [x.dtype for x in got] == [dtype, torch.float32, torch.float32]
    for name, kk, g, w32 in zip(("grad_pre", "grad_event_fac", "grad_bias"), (K * K, 1, K * K), got, want):
        assert torch.equal(g.float(), w32), _mismatch(name, g, w32, shape, kk, True)


# ---------------------------------------------------------------- full cfg2 size, real weights
def _reference_on_device(ev, fr, w, b, K, slope, G):
    """The block in float64 on the device, one sample at a time: P by F.unfold and a float64 matmul (no convolution
    algorithm that could round), then LeakyReLU, ReplicationPad2d and the unfold contraction of
    test_kpn_train_cpu, with P and the event as autograd leaves: P.grad is grad_pre, the event's grad the FAC part of
    dL/dEvent. Returns (out, grad_pre, grad_event_fac, grad_bias) as float32 tensors, each checked to hold the
    float64 values exactly."""
    F = torch.nn.functional
    B, Ce, H, W = ev.shape
    KK, R = K * K, (K - 1) // 2
    wd, bd = w.double().reshape(Ce * KK, -1), b.double()[:, None]

    def exact32(x):
        assert torch.equal(x.float().double(), x)
        return x.float()

    outs, gpres, gevs = [], [], []
    gbias = torch.zeros(Ce * KK, dtype=torch.float64, device=ev.device)
    for i in range(B):
        x = torch.cat([ev[i:i + 1], fr[i:i + 1]], 1).double()
        P = (wd @ F.unfold(x, 3, padding=1)[0] + bd).reshape(1, Ce * KK, H, W).requires_grad_()
        e = ev[i:i + 1].double().requires_grad_()
        cols = F.unfold(torch.nn.ReplicationPad2d(R)(e), K).reshape(1, Ce, KK, H, W)
        out = (cols * F.leaky_relu(P, slope).reshape(1, Ce, KK, H, W)).sum(2)
        out.backward(G[i:i + 1].double())
        outs.append(exact32(out.detach()))
        gpres.append(exact32(P.grad))
        gevs.append(exact32(e.grad))
        gbias += P.grad.sum((0, 2, 3))
        del x, P, e, cols, out
    return torch.cat(outs), torch.cat(gpres), torch.cat(gevs), exact32(gbias)


FULL = (4, 64, 64, 256, 256, 5)


@pytest.fixture(scope="module")
def full_size():
    """Lattice inputs at the cfg2 size (per = 305 items per CTA at 148 SMs) and their float64 reference."""
    from gpu_util import t
    inputs = [t(a) for a in _lattice_case(np.random.default_rng(2), *FULL)]
    ev, fr, w, b, G = inputs
    return inputs, _reference_on_device(ev, fr, w, b, FULL[-1], SLOPE, G)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, BF16, F16], ids=["fp32", "bf16", "fp16"])
def test_full_size_exact_on_the_lattice(mod, full_size, dtype):
    (ev, fr, w, b, G), (want_out, want_gpre, want_gev, want_gbias) = full_size
    K = FULL[-1]
    with torch.no_grad():
        out = mod.kernelconv_fac_fused(ev.to(dtype), fr.to(dtype), w.to(dtype), b.to(dtype), K, SLOPE)
    assert out.dtype == dtype
    assert torch.equal(out, want_out.to(dtype)), _mismatch("out", out, want_out.to(dtype), FULL)
    del out
    if dtype == torch.float32:
        got = mod.kernelconv_fac_fused_backward(ev, fr, w, b, K, SLOPE, G)
    else:
        got = mod.kernelconv_fac_fused_backward_bf16(ev.to(dtype), fr.to(dtype), w, b, K, SLOPE, G.to(dtype))
    assert [x.dtype for x in got] == [dtype, torch.float32, torch.float32]
    for name, kk, g, want in zip(("grad_pre", "grad_event_fac", "grad_bias"), (K * K, 1, K * K), got,
                                 (want_gpre.to(dtype), want_gev, want_gbias)):
        assert torch.equal(g, want), _mismatch(name, g, want, FULL, kk, True)


# ---------------------------------------------------------------- KernelPrediction with three halo parts
def _lattice_module(mod, w, b):
    """KernelPrediction(48, 5) (Cin = 96: three halo parts) with lattice conv weights and negative_slope 0.25."""
    from gpu_util import dev, t
    m = mod.KernelPrediction(48, 5).to(dev())
    with torch.no_grad():
        m.KernelConv.conv2d.weight.copy_(t(w))
        m.KernelConv.conv2d.bias.copy_(t(b))
    m.KernelConv.activation.negative_slope = SLOPE
    m.fused_backward = True
    return m


@pytest.mark.gpu
def test_kernel_prediction_three_parts_on_the_lattice(mod, oracle, no_tf32):  # noqa: F811
    """The fused no-grad forward is exact; the gradients through KernelConvFACFunction are within 1e-5 of max of the
    float64 block (the conv's weight and input gradients come from cuDNN's fp32 convolution backward of grad_pre, whose
    algorithm may round); grad_bias is the kernel's, exact."""
    from gpu_util import n, t
    shape = PIPELINE_SHAPES[0]
    B, Ce, Cf, H, W, K = shape
    assert (Ce, Cf, K) == (48, 48, 5)
    ev, fr, w, b, G = _lattice_case(np.random.default_rng(48), *shape)
    m = _lattice_module(mod, w, b)
    conv = m.KernelConv.conv2d
    want_out, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, SLOPE, bf16_operands=True)
    with torch.no_grad():
        out = n(m(t(ev), t(fr)))
    assert np.array_equal(out, want_out), _mismatch("out", out, want_out, shape)

    want = KO.kpn_fused_backward(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    e, f = t(ev).requires_grad_(), t(fr).requires_grad_()
    out = m(e, f)
    assert type(out.grad_fn).__name__ == "KernelConvFACFunctionBackward"
    out.backward(t(G))
    for name, g, r in (("grad_event", e.grad, want[0]), ("grad_frame", f.grad, want[1]),
                       ("grad_weight", conv.weight.grad, want[2])):
        assert rel_err(n(g), r) <= 1e-5, name
    assert np.array_equal(n(conv.bias.grad), want[3]), _mismatch("grad_bias", conv.bias.grad, want[3], shape, K * K)


@pytest.mark.gpu
def test_kernel_prediction_three_parts_under_bf16_autocast(mod, oracle):
    """The same module under bf16 autocast (fp32 parameters, bf16 activations) through KernelConvFACBF16Function, at
    the bounds of test_kpn_bf16_gpu.test_function_against_oracle; the output (the exact value rounded once to bf16) and
    grad_bias are exact."""
    from gpu_util import n, t
    shape = PIPELINE_SHAPES[0]
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b, G = _lattice_case(np.random.default_rng(49), *shape)
    m = _lattice_module(mod, w, b)
    conv = m.KernelConv.conv2d
    want_out, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, SLOPE, bf16_operands=True)
    want = KO.kpn_fused_backward(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    e, f = t(ev).to(BF16).requires_grad_(), t(fr).to(BF16).requires_grad_()
    with torch.autocast("cuda", dtype=BF16):
        out = m(e, f)
    assert type(out.grad_fn).__name__ == "KernelConvFACBF16FunctionBackward"
    assert torch.equal(out, t(want_out).to(BF16)), _mismatch("out", out, t(want_out).to(BF16), shape)
    out.backward(t(G).to(BF16))
    assert [x.dtype for x in (e.grad, f.grad, conv.weight.grad, conv.bias.grad)] == [BF16, BF16] + [torch.float32] * 2
    for name, g, r in (("grad_event", e.grad, want[0]), ("grad_frame", f.grad, want[1]),
                       ("grad_weight", conv.weight.grad, want[2])):
        assert rel_err(n(g.float()), r) <= 2.0 ** -7, name
    assert np.array_equal(n(conv.bias.grad), want[3]), _mismatch("grad_bias", conv.bias.grad, want[3], shape, K * K)
