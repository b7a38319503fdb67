"""GPU parity of FAC KernelConv2D: CUDA path (through the C ABI) vs the CPU oracle, the golden
vectors, and the stored results of the reference's own CUDA kernels compiled for sm_100a (tests/golden/ref_fac_*)."""
import os

import numpy as np
import pytest
import torch

from conftest import FAC_CASES, FWD_TOL, GRAD_TOL, load_golden, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fac():
    from ebfi_be_b200 import kernelconv2d
    return kernelconv2d


def _run(fac, x, ker, go, K):
    from gpu_util import n, t
    xg, kg = t(x).requires_grad_(), t(ker).requires_grad_()
    out = fac.KernelConv2DFunction.apply(xg, kg, K)
    out.backward(t(go))
    return n(out), n(xg.grad), n(kg.grad)


@pytest.mark.parametrize("case", FAC_CASES)
def test_golden_vectors(fac, case):
    g = load_golden(case)
    out, gi, gk = _run(fac, g["input"], g["kernel"], g["grad_output"], int(g["K"]))
    assert rel_err(out, g["output"]) < FWD_TOL
    assert rel_err(gi, g["grad_input"]) < GRAD_TOL
    assert rel_err(gk, g["grad_kernel"]) < GRAD_TOL


# (B, C, K, H, W): vector path (W % 4 == 0), scalar path, several row segments, ragged sizes,
# K = 7 and an even-free generic K = 9, one-pixel images, wide rows
SHAPES = [(2, 3, 5, 40, 64), (1, 2, 5, 33, 20), (1, 2, 5, 50, 23), (2, 2, 3, 37, 36), (1, 3, 3, 9, 7),
          (1, 2, 1, 20, 16), (1, 1, 7, 35, 24), (1, 1, 7, 20, 13), (1, 2, 9, 12, 16), (1, 1, 5, 1, 1),
          (1, 1, 5, 3, 4), (1, 1, 5, 17, 512), (1, 1, 5, 18, 1100), (1, 1, 3, 40, 300),
          (1, 2, 5, 24, 1280), (1, 1, 5, 20, 257), (1, 1, 3, 33, 70), (1, 1, 5, 36, 260)]   # column blocks + halo


@pytest.mark.parametrize("shape", SHAPES)
def test_against_oracle(fac, oracle, shape):
    B, C, K, H, W = shape
    rng = np.random.default_rng(hash(shape) % (2 ** 32))
    x = rng.standard_normal((B, C, H + K - 1, W + K - 1), dtype=np.float32)
    ker = rng.standard_normal((B, C * K * K, H, W), dtype=np.float32)
    go = rng.standard_normal((B, C, H, W), dtype=np.float32)
    out, gi, gk = _run(fac, x, ker, go, K)
    assert rel_err(out, oracle.fac_forward(x, ker, K)) < FWD_TOL
    ogi, ogk = oracle.fac_backward(x, ker, go, K)
    assert rel_err(gi, ogi) < GRAD_TOL
    assert rel_err(gk, ogk) < GRAD_TOL


@pytest.mark.parametrize("seg", ["4", "8", "16", "64"])
def test_segment_handoff_any_segment_height(fac, oracle, seg, monkeypatch):
    """grad_input rows cross row-segment (CTA) boundaries; every segmentation must agree."""
    monkeypatch.setenv("EBFI_FAC_SEG", seg)
    B, C, K, H, W = 1, 3, 5, 45, 32
    rng = np.random.default_rng(5)
    x = rng.standard_normal((B, C, H + K - 1, W + K - 1), dtype=np.float32)
    ker = rng.standard_normal((B, C * K * K, H, W), dtype=np.float32)
    go = rng.standard_normal((B, C, H, W), dtype=np.float32)
    out, gi, gk = _run(fac, x, ker, go, K)
    ogi, ogk = oracle.fac_backward(x, ker, go, K)
    assert rel_err(gi, ogi) < GRAD_TOL and rel_err(gk, ogk) < GRAD_TOL


def test_backward_is_bit_reproducible(fac):
    from gpu_util import dev
    torch.manual_seed(3)
    B, C, K, H, W = 2, 8, 5, 96, 128
    x = torch.randn(B, C, H + K - 1, W + K - 1, device=dev())
    ker = torch.randn(B, C * K * K, H, W, device=dev())
    go = torch.randn(B, C, H, W, device=dev())
    runs = []
    for _ in range(3):
        xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
        fac.KernelConv2DFunction.apply(xg, kg, K).backward(go)
        runs.append((xg.grad.clone(), kg.grad.clone()))
    for gi, gk in runs[1:]:
        assert torch.equal(gi, runs[0][0]) and torch.equal(gk, runs[0][1])


def test_matches_reference_cuda_kernels(fac):
    """The reference's own KernelConv2D_kernel.cu, compiled unmodified for sm_100a, through its stored results
    (tests/golden/ref_fac_case*.npz, see make_golden_ref.py)."""
    from gpu_util import RefGolden, ref_fac_inputs
    for i, (K, f) in enumerate(ref_fac_inputs()):
        ref = RefGolden(f"ref_fac_case{i}", f)
        xg, kg = f["x"].clone().requires_grad_(), f["ker"].clone().requires_grad_()
        out = fac.KernelConv2DFunction.apply(xg, kg, K)
        out.backward(f["go"])
        assert ref.equal("out", out), "forward uses the reference's tap order: expected bit-equality"
        assert ref.equal("grad_kernel", kg.grad), "grad_kernel is one product per element: expected bit-equality"
        assert ref.rel_err("grad_input", xg.grad) < GRAD_TOL


def test_module_pads_like_the_reference(fac, oracle):
    from gpu_util import n, t
    rng = np.random.default_rng(9)
    x = rng.standard_normal((1, 2, 10, 12), dtype=np.float32)
    ker = rng.standard_normal((1, 50, 10, 12), dtype=np.float32)
    out = fac.KernelConv2D(5).to("cuda")(t(x), t(ker))
    xp = np.pad(x, ((0, 0), (0, 0), (2, 2), (2, 2)), mode="edge")        # ReplicationPad2d, KernelConv2D.py:82-86
    assert rel_err(n(out), oracle.fac_forward(xp, ker, 5)) < FWD_TOL


def test_full_size_properties(fac):
    """BASELINE config 2 (B=4, C=64, K=5, 256x256): one-hot kernels shift the input exactly, and
    the op is bilinear, so <gO, out> == <grad_input, input> == <grad_kernel, kernel>."""
    from gpu_util import dev, dot
    torch.manual_seed(0)
    B, C, K, H, W = 4, 64, 5, 256, 256
    x = torch.randn(B, C, H + K - 1, W + K - 1, device=dev())
    ker = torch.zeros(B, C * K * K, H, W, device=dev())
    ker.view(B, C, K * K, H, W)[:, :, 7] = 1.0                            # tap (ky=1, kx=2)
    out = fac.KernelConv2DFunction.apply(x, ker, K)
    assert torch.equal(out, x[:, :, 1:1 + H, 2:2 + W])
    ker = 0.1 * torch.randn(B, C * K * K, H, W, device=dev())
    go = torch.randn(B, C, H, W, device=dev())
    xg, kg = x.clone().requires_grad_(), ker.requires_grad_()
    out = fac.KernelConv2DFunction.apply(xg, kg, K)
    out.backward(go)
    a, b, c = dot(go, out), dot(xg.grad, x), dot(kg.grad, ker)
    assert abs(a - b) <= 1e-5 * abs(a) and abs(a - c) <= 1e-5 * abs(a)


# bf16 storage variant (new capability; the reference is fp32-only). Stated tolerance: inputs are the
# bf16-rounded tensors, arithmetic is fp32, so the only error is the final rounding of each result to
# bf16: |err| <= 2^-8 * max|ref| per tensor (bf16 has 8 significand bits).
BF16_TOL = 2.0 ** -8


@pytest.mark.parametrize("shape", [(2, 4, 5, 40, 64), (1, 3, 5, 33, 20), (1, 2, 3, 37, 36), (1, 2, 5, 19, 23),
                                   (1, 2, 1, 20, 16), (1, 1, 9, 12, 16), (1, 2, 5, 22, 640), (1, 1, 5, 20, 516),
                                   (1, 1, 3, 18, 300)])
def test_bf16_variant_against_oracle(fac, oracle, shape):
    from gpu_util import dev
    B, C, K, H, W = shape
    g = torch.Generator().manual_seed(B * 100 + H)
    x = torch.randn(B, C, H + K - 1, W + K - 1, generator=g).bfloat16()
    ker = torch.randn(B, C * K * K, H, W, generator=g).bfloat16()
    go = torch.randn(B, C, H, W, generator=g).bfloat16()
    xg, kg = x.to(dev()).requires_grad_(), ker.to(dev()).requires_grad_()
    out = fac.KernelConv2DFunction.apply(xg, kg, K)
    assert out.dtype == torch.bfloat16
    out.backward(go.to(dev()))
    xf, kf, gf = x.float().numpy(), ker.float().numpy(), go.float().numpy()
    assert rel_err(out.detach().float().cpu().numpy(), oracle.fac_forward(xf, kf, K)) < BF16_TOL
    ogi, ogk = oracle.fac_backward(xf, kf, gf, K)
    assert rel_err(xg.grad.float().cpu().numpy(), ogi) < BF16_TOL
    assert rel_err(kg.grad.float().cpu().numpy(), ogk) < BF16_TOL


def test_bf16_full_size_is_reproducible_and_close_to_fp32(fac):
    from gpu_util import dev
    torch.manual_seed(0)
    B, C, K, H, W = 4, 64, 5, 256, 256
    x = torch.randn(B, C, H + K - 1, W + K - 1, device=dev()).bfloat16()
    ker = (0.1 * torch.randn(B, C * K * K, H, W, device=dev())).bfloat16()
    go = torch.randn(B, C, H, W, device=dev()).bfloat16()
    res = []
    for _ in range(2):
        xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
        o = fac.KernelConv2DFunction.apply(xg, kg, K)
        o.backward(go)
        res.append((o.detach(), xg.grad, kg.grad))
    assert all(torch.equal(a, b) for a, b in zip(*res))
    xf, kf = x.float().requires_grad_(), ker.float().requires_grad_()
    of = fac.KernelConv2DFunction.apply(xf, kf, K)
    of.backward(go.float())
    for got, want in zip(res[0], (of.detach(), xf.grad, kf.grad)):
        assert float((got.float() - want).abs().max()) <= BF16_TOL * float(want.abs().max())


def test_reference_gradient_check_recipe(fac):
    """gradient_check of the reference (KernelConv2D.py:61-74), re-expressed for the static Function API:
    10 rounds, B in [1,4], C = 1..10, K in {1,3}, H, W in {8,10}; the op is bilinear, hence eps=1e-1,
    atol=1e-5, rtol=1e-3."""
    import random
    from gpu_util import dev
    random.seed(0)
    torch.manual_seed(0)
    for i in range(10):
        B, C = random.randint(1, 4), i + 1
        K, H, W = random.choice([1, 3]), random.choice([8, 10]), random.choice([8, 10])
        input = torch.randn(B, C, H + K - 1, W + K - 1, device=dev(), dtype=torch.float32).requires_grad_()
        kernel = torch.randn(B, C * K * K, H, W, device=dev(), dtype=torch.float32).requires_grad_()
        fn = lambda a, b: fac.KernelConv2DFunction.apply(a, b, K)
        assert torch.autograd.gradcheck(fn, (input, kernel), eps=1e-1, atol=1e-5, rtol=1e-3)
