"""(1) The reference's OWN, unmodified wrapper files (models/DCNv2/dcn_v2.py, models/FAC/kernelconv2d/KernelConv2D.py,
staged by tools/refmodel.py into the git-ignored baseline/_ref/ebfi_be) executed on the GPU through this repo's `_ext` /
`kernelconv2d_cuda` shims, bit-compared with the host-side mirrors in ebfi_be_b200.
(2) Element-wise parity AT THE BENCHMARKED SHAPES (BASELINE configs[0], configs[1], and the 720p FAC of configs[3])
against the stored results of the reference's own CUDA kernels compiled unmodified for sm_100a (tests/golden/ref_*).
(3) The reference's full model (models/Ours/model_singleframe.py) forward + backward on the shims.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import FWD_TOL, GRAD_TOL, ROOT
from gpu_util import DCN_GEOM, RefGolden, cfg1_inputs, cfg2_inputs, dev

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))


def trel(got, want):
    """max-abs-err / max-abs-ref (SURVEY 8d), on the device in float64."""
    assert got.shape == want.shape
    return float((got.double() - want.double()).abs().max() / want.double().abs().max().clamp_min(1e-30))


@pytest.fixture(scope="module")
def staged():
    import refmodel
    if not refmodel.available():
        pytest.skip("baseline/_ref/ebfi_be not staged (build() ran without /root/reference)")
    refmodel.load()
    return refmodel


# ------------------------------------------------------------------ (1) reference wrappers, unchanged, on the shims
def test_reference_dcn_wrapper_runs_on_shims_bit_equal_to_mirror(staged):
    ref_dcn, _ = staged.reference_wrappers()
    from ebfi_be_b200 import dcn_v2 as ours
    assert ref_dcn.__file__.startswith(staged.STAGE)
    torch.manual_seed(3)
    B, C, H, W, dg = 2, 64, 40, 48, 8
    x = torch.randn(B, C, H, W, device=dev())
    for name in ("DCN", "DCN_sep"):
        torch.manual_seed(5)
        m_ref = getattr(ref_dcn, name)(C, 64, 3, 1, 1, deformable_groups=dg).to(dev())
        m_our = getattr(ours, name)(C, 64, 3, 1, 1, deformable_groups=dg).to(dev())
        m_our.fused = False                           # the mirror's reference-sequence path (chunk / cat / sigmoid)
        m_our.load_state_dict(m_ref.state_dict())
        with torch.no_grad():                         # zero-initialised offset conv (dcn_v2.py:175-177): make it deform
            for m in (m_ref, m_our):
                m.conv_offset_mask.weight.normal_(0, 0.05, generator=torch.Generator(device=dev()).manual_seed(9))
        xs = [x.clone().requires_grad_() for _ in range(2)]
        args = [(xs[0],), (xs[1],)] if name == "DCN" else [(xs[0], xs[0] * 0.5), (xs[1], xs[1] * 0.5)]
        o_ref, o_our = m_ref(*args[0]), m_our(*args[1])
        assert torch.equal(o_ref, o_our)
        go = torch.randn_like(o_ref)
        o_ref.backward(go); o_our.backward(go)
        # grad_input accumulates with float atomics in both runs (order-dependent last bits) -> tolerance, the
        # owner-computed / fixed-order gradients must agree bit for bit
        assert trel(xs[1].grad, xs[0].grad) < 1e-5
        assert torch.equal(m_ref.weight.grad, m_our.weight.grad)
        assert torch.equal(m_ref.bias.grad, m_our.bias.grad)
        assert trel(m_our.conv_offset_mask.weight.grad, m_ref.conv_offset_mask.weight.grad) < 1e-5


def test_reference_dcnv2_function_and_module(staged):
    ref_dcn, _ = staged.reference_wrappers()
    from ebfi_be_b200 import dcn_v2 as ours
    torch.manual_seed(1)
    B, C, H, W, dg = 1, 64, 32, 32, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = (torch.rand(64, C, 3, 3, device=dev()) * 2 - 1) / 24
    b = torch.randn(64, device=dev())
    o_ref = ref_dcn.dcn_v2_conv(x, off, msk, w, b, 1, 1, 1, dg)
    o_our = ours.dcn_v2_conv(x, off, msk, w, b, 1, 1, 1, dg)
    assert torch.equal(o_ref, o_our)
    m = ref_dcn.DCNv2(C, 64, 3, 1, 1, deformable_groups=dg).to(dev())
    assert m(x, off, msk).shape == (B, 64, H, W)


def test_reference_fac_wrapper_runs_on_shims_bit_equal_to_mirror(staged):
    _, ref_fac = staged.reference_wrappers()
    from ebfi_be_b200 import kernelconv2d as ours
    assert ref_fac.__file__.startswith(staged.STAGE)
    torch.manual_seed(2)
    B, C, K, H, W = 2, 16, 5, 40, 56
    x = torch.randn(B, C, H, W, device=dev())
    ker = 0.1 * torch.randn(B, C * K * K, H, W, device=dev())
    go = torch.randn(B, C, H, W, device=dev())
    res = []
    for modu in (ref_fac, ours):
        xi, ki = x.clone().requires_grad_(), ker.clone().requires_grad_()
        out = modu.KernelConv2D(kernel_size=K)(xi, ki)
        out.backward(go)
        res.append((out.detach(), xi.grad, ki.grad))
    (o_r, gx_r, gk_r), (o_o, gx_o, gk_o) = res
    assert torch.equal(o_r, o_o) and torch.equal(gk_r, gk_o)
    assert trel(gx_o, gx_r) < 1e-6          # ReplicationPad2d's backward (ATen) accumulates with atomics


# ------------------------------------------------------------------ (2) exact benchmark shapes vs the reference CUDA kernels
def test_cfg1_exact_shape_vs_reference_cuda():
    """BASELINE configs[0]: DCNv2 3x3 C=64 dg=8 B=1 256x256, same seeded inputs as bench.py; the reference kernels'
    results are stored in tests/golden/ref_cfg1_dcn.npz (see make_golden_ref.py)."""
    from ebfi_be_b200.shims import _ext
    d = cfg1_inputs()
    ref = RefGolden("ref_cfg1_dcn", d)
    args = [d[k] for k in ("x", "w", "b", "off", "msk")]
    o = _ext.dcn_v2_forward(*args, *DCN_GEOM)
    gr = _ext.dcn_v2_backward(*args, d["go"], *DCN_GEOM)
    assert ref.rel_err("out", o) < FWD_TOL
    for name, a in zip(("grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias"), gr):
        assert ref.rel_err(name, a) < GRAD_TOL, name


@pytest.mark.parametrize("shape", [(4, 64, 256, 256), (1, 64, 360, 640)], ids=["cfg2_B4_256", "cfg4_720p_half_res"])
def test_cfg2_exact_shape_vs_reference_cuda(shape, request):
    """BASELINE configs[1] (FAC K=5 C=64 B=4 256x256) and the FAC call of the 720p model (configs[3]); the reference
    kernels' results are stored in tests/golden/ref_<id>.npz (see make_golden_ref.py)."""
    from ebfi_be_b200.shims import kernelconv2d_cuda as kc
    f = cfg2_inputs(shape)
    ref = RefGolden("ref_" + request.node.callspec.id, f)
    out = torch.empty_like(f["go"])
    kc.forward(f["xi"], f["ker"], 5, out)
    assert ref.equal("out", out)                            # same tap order -> bit-identical
    gi, gk = torch.empty_like(f["xi"]), torch.empty_like(f["ker"])
    kc.backward(f["xi"], f["ker"], 5, f["go"], gi, gk)
    assert ref.equal("grad_kernel", gk)
    del gk
    assert ref.rel_err("grad_input", gi) < GRAD_TOL


# ------------------------------------------------------------------ (3) the reference model on the shims
def test_reference_model_forward_backward_on_shims(staged):
    m = staged.build_model(seed=0).to(dev()).train()
    g = torch.Generator(device="cpu").manual_seed(8)
    frame = torch.rand(2, 3, 64, 96, generator=g).to(dev())
    event = torch.round(2 * torch.rand(2, 16, 2, 64, 96, generator=g)).to(dev())
    t = torch.rand(2, 1, generator=g).to(dev())
    pre, fin = m(frame, event, t)
    assert pre.shape == fin.shape == (2, 3, 64, 96)
    (pre.mean() + fin.mean()).backward()
    gk = m.Modification.KernelConv.conv2d.weight.grad
    assert gk is not None and torch.isfinite(gk).all() and float(gk.abs().max()) > 0
    # A/B: the same forward on the reference's own FAC CUDA kernels
    with torch.no_grad():
        a = m(frame, event, t)[1]
        if staged.use_reference_cuda_fac(True):
            try:
                b = m(frame, event, t)[1]
            finally:
                staged.use_reference_cuda_fac(False)
            assert trel(a, b) < 1e-4        # the FAC outputs are bit-identical; cuDNN may pick other algorithms per call
