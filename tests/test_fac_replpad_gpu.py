"""KernelConv2D with ReplicationPad2d folded into the FAC kernels (ebfi_fac_replpad_*, KernelConv2DReplPadFunction)
against the padded op on the replicate-padded input, the CPU oracle, and float64 on the integer lattice."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GRAD_TOL, rel_err
from kpn_train_oracle import _fold_replication_pad

pytestmark = pytest.mark.gpu

BF16, F16 = torch.bfloat16, torch.float16
DTYPES = [torch.float32, BF16, F16]
DTYPE_IDS = ["fp32", "bf16", "fp16"]
# bound of one final rounding (two at the row-segment seams), relative to max|ref|
TOL16 = {BF16: 2.0 ** -7, F16: 2.0 ** -9}

# (B, C, K, H, W): test_fac_gpu.SHAPES (vector and scalar paths, several segments, K = 1, 3, 5, 7, generic K = 9,
# one-pixel images, H < K, W % 4 != 0, column blocks at W = 300, 1100, 1280, 257) plus W = 1 and H = 1 with K > 1
SHAPES = [(2, 3, 5, 40, 64), (1, 2, 5, 33, 20), (1, 2, 5, 50, 23), (2, 2, 3, 37, 36), (1, 3, 3, 9, 7),
          (1, 2, 1, 20, 16), (1, 1, 7, 35, 24), (1, 1, 7, 20, 13), (1, 2, 9, 12, 16), (1, 1, 5, 1, 1),
          (1, 1, 5, 3, 4), (1, 1, 5, 17, 512), (1, 1, 5, 18, 1100), (1, 1, 3, 40, 300),
          (1, 2, 5, 24, 1280), (1, 1, 5, 20, 257), (1, 1, 3, 33, 70), (1, 1, 5, 36, 260),
          (1, 2, 3, 6, 1), (1, 2, 5, 1, 40), (1, 1, 7, 2, 5)]


@pytest.fixture(scope="module")
def kc():
    from ebfi_be_b200 import kernelconv2d
    return kernelconv2d


def _inputs(shape, dtype, seed, lattice=False):
    from gpu_util import dev
    B, C, K, H, W = shape
    g = torch.Generator().manual_seed(seed)
    if lattice:     # integers: every fp32 sum below is exact, and every result fits a 16-bit significand
        mk = lambda *s: torch.randint(-1, 2, s, generator=g).float()
        x = torch.randint(-2, 3, (B, C, H, W), generator=g).float()
    else:
        mk = lambda *s: torch.randn(*s, generator=g)
        x = mk(B, C, H, W)
    ker, go = mk(B, C * K * K, H, W), mk(B, C, H, W)
    return tuple(a.to(dtype).to(dev()) for a in (x, ker, go))


def _padded_op(kc, x, ker, go, K):
    """ReplicationPad2d + the padded FAC entries: (out, grad of the padded input, grad_kernel)."""
    xp = F.pad(x, ((K - 1) // 2,) * 4, mode="replicate").requires_grad_()
    kg = ker.clone().requires_grad_()
    out = kc.KernelConv2DFunction.apply(xp, kg, K)
    out.backward(go)
    return out.detach(), xp.grad, kg.grad


def _folded_op(kc, x, ker, go, K):
    xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
    out = kc.KernelConv2DReplPadFunction.apply(xg, kg, K)
    out.backward(go)
    return out.detach(), xg.grad, kg.grad


def _f64_reference(x, ker, go, K):
    """float64 forward and folded grad_input."""
    x, ker, go = (a.double().cpu().numpy() for a in (x, ker, go))
    B, C, H, W = x.shape
    R = (K - 1) // 2
    xp = np.pad(x, ((0, 0), (0, 0), (R, R), (R, R)), mode="edge")
    k5 = ker.reshape(B, C, K * K, H, W)
    out = np.zeros((B, C, H, W))
    gpad = np.zeros_like(xp)
    for t in range(K * K):
        ky, kx = divmod(t, K)
        out += xp[:, :, ky:ky + H, kx:kx + W] * k5[:, :, t]
        gpad[:, :, ky:ky + H, kx:kx + W] += k5[:, :, t] * go
    return out, _fold_replication_pad(gpad, R)


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("shape", SHAPES)
def test_equals_padded_op(kc, oracle, shape, dtype):
    """Forward and grad_kernel bit-equal to the padded op; grad_input bit-equal to it away from the border, and
    the fold of the oracle's padded gradient everywhere."""
    from gpu_util import n
    B, C, K, H, W = shape
    x, ker, go = _inputs(shape, dtype, sum(shape))
    out, gi, gk = _folded_op(kc, x, ker, go, K)
    pout, pgi, pgk = _padded_op(kc, x, ker, go, K)
    assert out.dtype == dtype and gi.shape == x.shape and gi.dtype == dtype
    assert torch.equal(out, pout)
    assert torch.equal(gk, pgk)
    p = (K - 1) // 2
    assert torch.equal(gi[:, :, 1:H - 1, 1:W - 1], pgi[:, :, p + 1:p + H - 1, p + 1:p + W - 1])

    xp = F.pad(x.float(), (p,) * 4, mode="replicate")
    want = _fold_replication_pad(oracle.fac_backward(n(xp), n(ker.float()), n(go.float()), K)[0].astype(np.float64), p)
    assert rel_err(n(gi.float()), want) < (GRAD_TOL if dtype == torch.float32 else TOL16[dtype])


# the last segment is shorter than K-1 rows at H = 45, K = 5 (EBFI_FAC_SEG = 4 -> 45 = 11 * 4 + 1) and at
# H = 37, K = 7 (segments of 6 or 8 rows leave 1 or 5); W = 300 and 1100 run column blocks
LATTICE_SHAPES = [(1, 3, 5, 45, 32), (1, 2, 5, 45, 23), (1, 2, 3, 45, 300), (1, 1, 5, 45, 1100), (2, 2, 7, 37, 13),
                  (1, 2, 5, 2, 36)]


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("seg", ["4", "8", "16", "64"])
@pytest.mark.parametrize("shape", LATTICE_SHAPES)
def test_exact_on_the_lattice(kc, shape, seg, dtype, monkeypatch):
    """Integer inputs: the fold's fp32 sums are exact, so forward and grad_input equal float64 whatever the
    segmentation (top fold in segment 0, bottom fold and the overhang merge in the last segment)."""
    from gpu_util import n
    B, C, K, H, W = shape
    if dtype != torch.float32 and K == 7:
        pytest.skip("corner sums of K = 7 exceed a bf16 significand on this lattice")
    monkeypatch.setenv("EBFI_FAC_SEG", seg)
    x, ker, go = _inputs(shape, dtype, int(seg) + H, lattice=True)
    out, gi, _ = _folded_op(kc, x, ker, go, K)
    want_out, want_gi = _f64_reference(x, ker, go, K)
    assert np.array_equal(n(out.double()), want_out)
    assert np.array_equal(n(gi.double()), want_gi)


@pytest.mark.parametrize("dtype", [torch.float32, BF16], ids=["fp32", "bf16"])
def test_full_size_bit_reproducible(kc, dtype):
    """cfg2 (B=4, C=64, K=5, 256x256), three runs of the module's forward + backward."""
    from gpu_util import dev
    torch.manual_seed(4)
    B, C, K, H, W = 4, 64, 5, 256, 256
    x = torch.randn(B, C, H, W, device=dev()).to(dtype)
    ker = (0.1 * torch.randn(B, C * K * K, H, W, device=dev())).to(dtype)
    go = torch.randn(B, C, H, W, device=dev()).to(dtype)
    m = kc.KernelConv2D(K)
    runs = []
    for _ in range(3):
        xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
        out = m(xg, kg)
        out.backward(go)
        runs.append((out.detach(), xg.grad, kg.grad))
        del xg, kg, out
    for r in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(r, runs[0]))


def test_trains_under_deterministic_algorithms(kc):
    """The module and KernelPrediction's op sequence run under torch.use_deterministic_algorithms(True), with
    bit-identical gradients from two steps. ATen's CUDA replication_pad2d backward raises there (F.pad, and with it
    nn.ReplicationPad2d, sidesteps it under the switch with an index-based decomposition of the pad)."""
    from gpu_util import dev
    from ebfi_be_b200.modification import KernelPrediction
    torch.manual_seed(6)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        x = torch.randn(2, 4, 20, 24, device=dev(), requires_grad=True)
        ker = torch.randn(2, 4 * 25, 20, 24, device=dev(), requires_grad=True)
        kc.KernelConv2D(5)(x, ker).sum().backward()
        assert x.grad is not None and ker.grad is not None

        m = KernelPrediction(64, 5).to(dev())
        ev, fr = torch.randn(2, 64, 32, 40, device=dev()), torch.randn(2, 64, 32, 40, device=dev())
        G = torch.randn(2, 64, 32, 40, device=dev())
        grads = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
            m(e, f).backward(G)
            grads.append([e.grad, f.grad] + [p.grad.clone() for p in m.parameters()])
        assert all(torch.equal(a, b) for a, b in zip(*grads))

        xp = torch.ops.aten.replication_pad2d(x, [2, 2, 2, 2])
        out = kc.KernelConv2DFunction.apply(xp, ker, 5)
        with pytest.raises(RuntimeError, match="deterministic"):
            out.sum().backward()
    finally:
        torch.use_deterministic_algorithms(was)


def test_saves_no_padded_tensor_and_peak_memory(kc):
    """The module's graph saves no (B, C, H+K-1, W+K-1) tensor; at cfg2 the forward + backward peak is at least
    one padded tensor below ReplicationPad2d + KernelConv2DFunction's."""
    from gpu_util import dev
    B, C, K, H, W = 4, 64, 5, 256, 256
    torch.manual_seed(7)
    x = torch.randn(B, C, H, W, device=dev())
    ker = 0.1 * torch.randn(B, C * K * K, H, W, device=dev())
    go = torch.randn(B, C, H, W, device=dev())

    saved = []
    xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
    with torch.autograd.graph.saved_tensors_hooks(lambda t: saved.append(tuple(t.shape)) or t, lambda t: t):
        out = kc.KernelConv2D(K)(xg, kg)
    assert (B, C, H + K - 1, W + K - 1) not in saved and (B, C, H, W) in saved
    del out, xg, kg

    pad = torch.nn.ReplicationPad2d((K - 1) // 2)

    def peak(fn):
        xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn(xg, kg).backward(go)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    p_old = peak(lambda a, b: kc.KernelConv2DFunction.apply(pad(a), b, K))
    p_new = peak(kc.KernelConv2D(K))
    assert p_new <= p_old - B * C * (H + K - 1) * (W + K - 1) * 4, (p_new, p_old)


def test_mixed_dtypes_and_shapes_are_refused(kc):
    from gpu_util import dev
    x = torch.randn(1, 2, 8, 8, device=dev())
    with pytest.raises(RuntimeError, match="float32"):
        kc.KernelConv2D(3)(x, torch.randn(1, 18, 8, 8, device=dev()).bfloat16())
    with pytest.raises(RuntimeError, match="do not fit"):
        kc.KernelConv2D(3)(x, torch.randn(1, 18, 8, 9, device=dev()))
