"""The deterministic DCNv2 backward (EBFI_DCN_DETERMINISTIC, torch.use_deterministic_algorithms) on the box kernel
(csrc/dcn_bwd_box.cu, DET instantiations): samples whose corners leave the staged box add into an int64 fixed-point
buffer instead of float reductions, so every gradient is bit-reproducible for any offsets, the 16-bit entries run
natively, and where no sample leaves its box the result has the default mode's bits."""
from contextlib import nullcontext as _nullcontext

import numpy as np
import pytest
import torch

from conftest import GRAD_TOL, rel_err
from test_dcn_pipeline_gpu import PIPELINE_SHAPES, _check_all, _expected, _geom, dcn_work_split

pytestmark = pytest.mark.gpu

BF16, F16 = torch.bfloat16, torch.float16
BF16_TOL, F16_TOL = 2.0 ** -8, 2.0 ** -11      # the bf16 / fp16 suites' gates: one rounding, relative to max|ref|


@pytest.fixture(scope="module")
def ext():
    from ebfi_be_b200.shims import _ext
    return _ext


def _dev():
    return torch.device("cuda:0")


def _box_runs(shape):
    """The fp32 call of `shape` takes the box backward (the plan restated by dcn_work_split, checked against the
    library's there)."""
    return dcn_work_split(shape, 148)["bwd"]["box"]


def _case(shape, seed, sigma, dtype=torch.float32, packed=False):
    """(acts, weight, bias, grad_output) with offsets sigma * randn; sigma <= 1 is clamped to |offset| <= 2, so that
    every sample stays in its box. Activations are rounded to `dtype` (the values every entry then sees)."""
    B, C, Co, H, W, dg = shape[:6]
    (kh, kw, *_), Ho, Wo = _geom(shape)
    g = torch.Generator().manual_seed(seed)
    nt = dg * kh * kw
    x = torch.randn(B, C, H, W, generator=g)
    off = sigma * torch.randn(B, 2 * nt, Ho, Wo, generator=g)
    if sigma <= 1:
        off = (2 * off).clamp(-2, 2)
    m = torch.rand(B, nt, Ho, Wo, generator=g) if not packed else torch.randn(B, nt, Ho, Wo, generator=g)
    w = torch.randn(Co, C, kh, kw, generator=g) / (C * kh * kw) ** 0.5
    b = torch.randn(Co, generator=g)
    go = torch.randn(B, Co, Ho, Wo, generator=g)
    acts = (x, torch.cat([off, m], 1)) if packed else (x, off, m)
    return [a.to(dtype).to(_dev()) for a in acts], w.to(_dev()), b.to(_dev()), go.to(dtype).to(_dev())


def _fail(*a, **k):
    raise AssertionError("_via_fp32 ran: the 16-bit call did not run natively")


def _no_conversion(ext, monkeypatch):
    monkeypatch.setattr(ext, "_via_fp32", _fail)


def _bwd(ext, acts, w, b, go, ints, packed, native=None):
    """Forward (leaves the blocked input copy for the backward to reuse) + backward through the shim. native: a
    monkeypatch; the backward (only: a 10-tap fp32-shape forward runs on the CUDA cores) must not convert."""
    x = acts[0]
    if packed:
        ext.dcn_v2_forward_packed(x, w, b, acts[1], *ints)
    else:
        ext.dcn_v2_forward(x, w, b, acts[1], acts[2], *ints)
    with native.context() if native is not None else _nullcontext() as mp:
        if native is not None:
            mp.setattr(ext, "_via_fp32", _fail)
        if packed:
            return ext.dcn_v2_backward_packed(x, w, b, acts[1], go, *ints)
        return ext.dcn_v2_backward(x, w, b, acts[1], acts[2], go, *ints)


# (B, C, Co, H, W, dg, kernel, stride, pad, dilation): cpg 8 / 16 / 32, stride 1, dilation 2, pad 0, pad_h != pad_w
DET_SHAPES = [
    (1, 64, 64, 40, 48, 8, 3, 1, 1, 1),
    (1, 64, 64, 36, 40, 4, 3, 1, 2, 2),
    (2, 64, 64, 24, 40, 2, 3, 1, 0, 1),
    (1, 64, 64, 30, 44, 8, (2, 5), 1, (0, 2), 1),
]


def test_det_shapes_take_the_box_kernel():
    for shape in DET_SHAPES:
        assert _box_runs(shape), shape
    assert {s[1] // s[5] for s in DET_SHAPES} == {8, 16, 32}


# ---------------------------------------------------------------- 1. no far sample: the default mode's bits
@pytest.mark.parametrize("packed", [False, True], ids=["plain", "packed"])
@pytest.mark.parametrize("dtype", [torch.float32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("shape", DET_SHAPES)
def test_det_equals_default_without_far_samples(ext, monkeypatch, shape, dtype, packed):
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, sum(shape[:6]), 1.0, dtype, packed)
    native = monkeypatch if dtype != torch.float32 else None
    monkeypatch.delenv("EBFI_DCN_DETERMINISTIC", raising=False)
    want = _bwd(ext, acts, w, b, go, ints, packed, native)
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    got = _bwd(ext, acts, w, b, go, ints, packed, native)
    for i, (a, c) in enumerate(zip(got, want)):
        assert a.dtype == c.dtype and torch.equal(a, c), i


# ---------------------------------------------------------------- 2. far samples: reproducible and accurate
FAR_SHAPES = [DET_SHAPES[0], DET_SHAPES[2]]


@pytest.mark.parametrize("packed", [False, True], ids=["plain", "packed"])
@pytest.mark.parametrize("dtype", [torch.float32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("shape", FAR_SHAPES)
def test_far_samples_reproducible_and_in_tolerance(ext, oracle, monkeypatch, shape, dtype, packed):
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, 7 + sum(shape[:6]), 10.0, dtype, packed)
    assert float((acts[1][:, : acts[1].shape[1] * 2 // 3 if packed else None].abs() > 8).float().mean()) > 0.3
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    if dtype != torch.float32:
        _no_conversion(ext, monkeypatch)
    runs = [_bwd(ext, acts, w, b, go, ints, packed) for _ in range(3)]
    for r in runs[1:]:
        for i, (a, c) in enumerate(zip(r, runs[0])):
            assert torch.equal(a, c), i
    monkeypatch.setenv("EBFI_DCN_NO_BLOCKED_REUSE", "1")
    ext._blocked_cache.clear()
    for i, (a, c) in enumerate(zip(_bwd(ext, acts, w, b, go, ints, packed), runs[0])):
        assert torch.equal(a, c), i
    # against the float64 oracle on the same (rounded) values
    f = lambda t: t.float().cpu().numpy()
    s, p, d, dg = ints[2:4], ints[4:6], ints[6:8], ints[8]
    if packed:
        om = f(acts[1])
        k2 = om.shape[1] * 2 // 3
        off, msk = om[:, :k2], (1 / (1 + np.exp(-om[:, k2:].astype(np.float64)))).astype(np.float32)
    else:
        off, msk = f(acts[1]), f(acts[2])
    want = oracle.dcn_backward(f(acts[0]), off, msk, f(w), f(b), f(go), s, p, d, dg)
    if packed:
        want = [want[0], np.concatenate([want[1], want[2] * msk * (1 - msk)], 1), want[3], want[4]]
    tol = {torch.float32: GRAD_TOL, BF16: BF16_TOL, F16: F16_TOL}[dtype]
    for i, (g, r) in enumerate(zip(runs[0], want)):
        assert rel_err(f(g), r) < tol + (GRAD_TOL if dtype != torch.float32 else 0), i


# ---------------------------------------------------------------- 3. native 16-bit = fp32 det on the widened values
@pytest.mark.parametrize("packed", [False, True], ids=["plain", "packed"])
@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("shape", FAR_SHAPES)
def test_native_16bit_equals_fp32_det_rounded_once(ext, monkeypatch, shape, dtype, packed):
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, 3 + sum(shape[:6]), 10.0, dtype, packed)
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    want = _bwd(ext, [a.float() for a in acts], w, b, go.float(), ints, packed)
    _no_conversion(ext, monkeypatch)
    got = _bwd(ext, acts, w, b, go, ints, packed)
    na = len(acts)
    for i, (g, r) in enumerate(zip(got, want)):
        if i < na:
            assert g.dtype == dtype and torch.equal(g, r.to(dtype)), i
        else:
            assert g.dtype == torch.float32 and torch.equal(g, r), i


# ---------------------------------------------------------------- 4. the dyadic lattice with far samples, exactly
@pytest.mark.parametrize("packed", [False, True], ids=["plain", "packed"])
@pytest.mark.parametrize("shape", [PIPELINE_SHAPES[2], PIPELINE_SHAPES[4]], ids=["cpg32", "cpg16"])
def test_det_exact_on_the_lattice(ext, oracle, monkeypatch, shape, packed):
    """_lattice_case has 1/8 of its offsets beyond the box and the image: the int64 far-sample sums convert exactly,
    so all five gradients equal float64 (and hence the default mode) bit for bit."""
    from gpu_util import t
    assert _box_runs(shape)
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    (x, off, msk, w, b, go), want = _expected(oracle, shape, packed=packed)
    ints, _, _ = _geom(shape)
    xt, wt, bt = t(x), t(w), t(b)
    if packed:
        om = t(np.concatenate([off, np.zeros((off.shape[0], off.shape[1] // 2) + off.shape[2:], np.float32)], 1))
        out = ext.dcn_v2_forward_packed(xt, wt, bt, om, *ints)
        g_in, g_om, g_w, g_b = ext.dcn_v2_backward_packed(xt, wt, bt, om, t(go), *ints)
        out_w, gi_w, goff_w, gm_w, gw_w, gb_w = want
        _check_all(shape, [out, g_in, g_om, g_w, g_b], [out_w, gi_w, np.concatenate([goff_w, gm_w / 4], 1), gw_w, gb_w])
    else:
        out = ext.dcn_v2_forward(xt, wt, bt, t(off), t(msk), *ints)
        grads = ext.dcn_v2_backward(xt, wt, bt, t(off), t(msk), t(go), *ints)
        _check_all(shape, [out, *grads], want)


# ---------------------------------------------------------------- 5. non-finite values
@pytest.mark.parametrize("bad", [float("nan"), float("inf")], ids=["nan", "inf"])
@pytest.mark.parametrize("dtype", [torch.float32, BF16, F16], ids=["fp32", "bf16", "fp16"])
def test_nonfinite_grad_output_gives_nan(ext, monkeypatch, dtype, bad):
    shape = DET_SHAPES[0]
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, 5, 10.0, dtype)
    go[0, 3, 7, 9] = bad
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    g_in = _bwd(ext, acts, w, b, go, ints, False)[0]
    assert g_in.dtype == dtype and bool(torch.isnan(g_in).all())


def test_fp16_overflow_is_inf_and_grad_scaler_skips(ext, monkeypatch):
    from ebfi_be_b200 import dcn_v2
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    shape = DET_SHAPES[0]
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, 6, 10.0, F16)
    g_in = _bwd(ext, acts, 1e6 * w, b, go, ints, False, monkeypatch)[0]      # |grad_input| beyond 65504
    assert g_in.dtype == F16
    assert bool(torch.isinf(g_in).any()) and not bool(torch.isnan(g_in).any())
    torch.manual_seed(11)
    s = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
    with torch.no_grad():
        s.conv_offset_mask.weight.normal_(0, 0.5)                  # far samples
    opt = torch.optim.SGD(s.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40)
    x, fea = torch.randn(2, 64, 24, 24, device=_dev()), torch.randn(2, 64, 24, 24, device=_dev())
    before = [p.detach().clone() for p in s.parameters()]
    with torch.autocast("cuda", dtype=F16):
        loss = s(x, fea).float().square().mean()
    scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 39
    assert all(torch.equal(p, q) for p, q in zip(s.parameters(), before))


# ---------------------------------------------------------------- 6. modules under torch.use_deterministic_algorithms
@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "fp16"])
def test_dcn_sep_autocast_under_torch_switch(ext, monkeypatch, dtype):
    from ebfi_be_b200 import dcn_v2
    monkeypatch.delenv("EBFI_DCN_DETERMINISTIC", raising=False)
    _no_conversion(ext, monkeypatch)
    torch.manual_seed(21)
    m = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
    with torch.no_grad():
        m.conv_offset_mask.weight.normal_(0, 0.3)                  # many far samples
    g = torch.Generator().manual_seed(22)
    x0, f0, go = (torch.randn(2, 64, 24, 32, generator=g).to(_dev()) for _ in range(3))

    def run():
        m.zero_grad(set_to_none=True)
        x, fea = x0.clone().requires_grad_(), f0.clone().requires_grad_()
        with torch.autocast("cuda", dtype=dtype):
            out = m(x, fea)
        out.backward(go.to(out.dtype))
        return [out, x.grad, fea.grad] + [p.grad.clone() for p in m.parameters()]

    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        assert ext._deterministic()
        a, c = run(), run()
    finally:
        torch.use_deterministic_algorithms(prev)
    assert a[0].dtype == dtype and a[1].dtype == a[2].dtype == torch.float32
    assert all(v.dtype == torch.float32 for v in a[3:])
    for i, (u, v) in enumerate(zip(a, c)):
        assert torch.equal(u, v), i
    if hasattr(m, "flush_offset_warnings"):
        m.flush_offset_warnings()


# ---------------------------------------------------------------- 7. data-parallel entry, world 1
@pytest.mark.parametrize("dtype", [torch.float32, BF16], ids=["fp32", "bf16"])
def test_world_one_dp_det_equals_det(ext, monkeypatch, dtype):
    from test_dp_gpu import _SoloComm
    shape = DET_SHAPES[0]
    ints, _, _ = _geom(shape)
    acts, w, b, go = _case(shape, 9, 10.0, dtype)
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    if dtype != torch.float32:
        _no_conversion(ext, monkeypatch)
    comm = _SoloComm(w.numel() + b.numel(), _dev())
    want = ext.dcn_v2_backward(acts[0], w, b, acts[1], acts[2], go, *ints)
    got = ext.dcn_v2_backward_dp(acts[0], w, b, acts[1], acts[2], go, *ints, comm)
    for i, (u, v) in enumerate(zip(got, want)):
        assert torch.equal(u, v), i
