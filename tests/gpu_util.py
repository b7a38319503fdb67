"""Helpers shared by the `-m gpu` parity tests (test infrastructure)."""
import os

import numpy as np
import torch

from conftest import GOLDEN


def dev():
    return torch.device("cuda:0")


def t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).to(dev())


def n(x):
    return x.detach().cpu().numpy()


def dot(a, b):
    return float((a.double() * b.double()).sum())


# ---------------------------------------------------------------- comparisons with the reference's CUDA kernels
# The reference's dcn_v2_im2col_cuda.cu and KernelConv2D_kernel.cu are not part of this repository. What the tests
# compared against is stored instead: tests/golden/ref_*.npz, written by tests/golden/make_golden_ref.py. Each file
# holds, per output, its values at REF_SAMPLE positions spread over the tensor (every element of a smaller one) and
# the largest |value| of the whole tensor (the denominator of rel_err), plus a few input values that pin the seeded
# inputs.
REF_SAMPLE = 2048
REF_INPUT_PROBES = 64
_STRIDE = 1_000_003            # prime: k * _STRIDE % numel visits distinct positions in every channel and row
DCN_GEOM = (3, 3, 1, 1, 1, 1, 1, 1, 8)


def ref_dcn_inputs():
    """test_dcn_gpu.py::test_matches_reference_cuda_kernels: B=2, C=64 -> 64, 40x40, dg=8."""
    torch.manual_seed(2)
    B, C, Co, H, W, dg = 2, 64, 64, 40, 40, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = (torch.rand(Co, C, 3, 3, device=dev()) * 2 - 1) / 24
    b = torch.randn(Co, device=dev())
    go = torch.randn(B, Co, H, W, device=dev())
    return dict(x=x, off=off, msk=msk, w=w, b=b, go=go)


REF_FAC_SHAPES = [(2, 4, 5, 64, 64), (1, 3, 3, 30, 22), (1, 2, 5, 19, 21)]


def ref_fac_inputs():
    """test_fac_gpu.py::test_matches_reference_cuda_kernels: one (K, inputs) per REF_FAC_SHAPES entry."""
    torch.manual_seed(0)
    cases = []
    for (B, C, K, H, W) in REF_FAC_SHAPES:
        x = torch.randn(B, C, H + K - 1, W + K - 1, device=dev())
        ker = torch.randn(B, C * K * K, H, W, device=dev())
        go = torch.randn(B, C, H, W, device=dev())
        cases.append((K, dict(x=x, ker=ker, go=go)))
    return cases


def cfg1_inputs():
    """BASELINE configs[0]: DCNv2 3x3 C=64 dg=8 B=1 256x256, the seeded inputs of bench.py."""
    g = torch.Generator(device="cpu").manual_seed(1234)
    r = lambda *s: torch.randn(*s, generator=g)
    x, off, msk = r(1, 64, 256, 256), 2 * r(1, 144, 256, 256), torch.sigmoid(r(1, 72, 256, 256))
    w, b, go = (torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24, r(64), r(1, 64, 256, 256)
    return {k: v.to(dev()) for k, v in dict(x=x, off=off, msk=msk, w=w, b=b, go=go).items()}


def cfg2_inputs(shape):
    """FAC K=5 on (B, C, H, W) = shape, seeded like bench.py."""
    B, C, H, W = shape
    g = torch.Generator(device="cpu").manual_seed(1234)
    xi = torch.randn(B, C, H + 4, W + 4, generator=g).to(dev())
    ker = (0.1 * torch.randn(B, C * 25, H, W, generator=g)).to(dev())
    go = torch.randn(B, C, H, W, generator=g).to(dev())
    return dict(xi=xi, ker=ker, go=go)


def _at(x, n):
    """x's values at n positions spread over it (flattened), as float32 numpy."""
    if x.numel() <= n:
        idx = np.arange(x.numel())
    else:
        assert np.gcd(x.numel(), _STRIDE) == 1
        idx = np.arange(n, dtype=np.int64) * _STRIDE % x.numel()
    return x.detach().reshape(-1)[torch.from_numpy(idx).to(x.device)].float().cpu().numpy()


def record_ref(path, inputs, outputs):
    """Write one ref_*.npz (used by make_golden_ref.py)."""
    z = {f"in_{k}": _at(v, REF_INPUT_PROBES) for k, v in inputs.items()}
    for k, v in outputs.items():
        z[k], z[k + "_absmax"] = _at(v, REF_SAMPLE), np.float64(v.detach().abs().max().item())
    np.savez_compressed(path, **z)


class RefGolden:
    """The stored reference values of one case; checks on construction that the seeded inputs are the recorded ones."""

    def __init__(self, name, inputs):
        with np.load(os.path.join(GOLDEN, name + ".npz")) as f:
            self.z = {k: f[k] for k in f.files}
        for k, v in inputs.items():
            assert np.array_equal(_at(v, REF_INPUT_PROBES), self.z[f"in_{k}"]), (
                f"{name}: input `{k}` is not the one the stored values were computed from (did the seeded generator change?)")

    def _pair(self, key, got):
        return _at(got, REF_SAMPLE), self.z[key]

    def rel_err(self, key, got):
        """max-abs-err over the stored positions / max-abs of the whole reference tensor."""
        g, w = self._pair(key, got)
        return float(np.abs(g.astype(np.float64) - w).max() / max(float(self.z[key + "_absmax"]), 1e-30))

    def equal(self, key, got):
        g, w = self._pair(key, got)
        return np.array_equal(g, w)
