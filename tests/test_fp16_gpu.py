"""fp16 activations (torch.autocast's default dtype): the *_fp16 entry points of DCNv2, FAC and the fused
KernelConv -> FAC block, the boundary conversion where the DCN kernels have no native 16-bit I/O, overflow to inf for
GradScaler, and the modules under torch.autocast("cuda").

The fp16 instantiations change only the activation loads (exact widening) and stores (one RN rounding of the values
the fp32 kernels store), so on fp16-valued inputs they reproduce the fp32 kernels bit for bit. DCN offsets stay within
the sampling box (see test_dcn_bf16_gpu.py)."""
import copy

import numpy as np
import pytest
import torch

import kpn_train_oracle as KO
import test_kpn_train_gpu as TG
from conftest import rel_err
from test_dcn_bf16_gpu import FALLBACKS, TC_SHAPES, _box_path, _forward, _fwd_bwd, _module, _rel_l2
from test_kpn_gpu import PIPELINE_SHAPES as KPN_PIPELINE_SHAPES
from test_kpn_gpu import SHAPES as KPN_SHAPES
from test_kpn_gpu import _case as _kpn_case

pytestmark = pytest.mark.gpu
F16 = torch.float16
F16_TOL = 2.0 ** -11        # one fp16 rounding, relative to max|ref|
SLOPE = 0.01


def _dev():
    return torch.device("cuda:0")


def _h(t):
    return t.half().to(_dev())


@pytest.fixture(scope="module")
def ext():
    from ebfi_be_b200.shims import _ext
    return _ext


@pytest.fixture(scope="module")
def mod():
    from ebfi_be_b200 import modification
    return modification


def _dcn_case(shape, seed, packed=False, obound=4.0):
    """fp16 activations, fp32 parameters. shape = (B, C, Co, H, W, k, (sh, sw), pad, dil, dg)."""
    B, C, Co, H, W, k, (sh, sw), p, d, dg = shape
    g = torch.Generator().manual_seed(seed)
    Ho, Wo = (H + 2 * p - (d * (k - 1) + 1)) // sh + 1, (W + 2 * p - (d * (k - 1) + 1)) // sw + 1
    nt = dg * k * k
    x = _h(torch.randn(B, C, H, W, generator=g))
    off = _h((torch.rand(B, 2 * nt, Ho, Wo, generator=g) * 2 - 1) * obound)
    if packed:
        acts = (x, torch.cat([off, _h(torch.randn(B, nt, Ho, Wo, generator=g))], 1))
    else:
        acts = (x, off, _h(torch.rand(B, nt, Ho, Wo, generator=g)))
    w = (torch.randn(Co, C, k, k, generator=g) / (C * k * k) ** 0.5).to(_dev())
    b = torch.randn(Co, generator=g).to(_dev())
    go = _h(torch.randn(B, Co, Ho, Wo, generator=g))
    return acts, w, b, go, (k, k, sh, sw, p, p, d, d, dg)


# ---------------------------------------------------------------- 1. bit-identity with the fp32 kernels
@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("shape", TC_SHAPES)
def test_dcn_bit_identical_to_fp32_kernels(ext, shape, packed):
    acts, w, b, go, ints = _dcn_case(shape, 11, packed, obound=4.0 if shape[6] == (1, 1) else 2.0)
    assert _box_path(ints, shape)
    out, grads = _fwd_bwd(ext, acts, w, b, go, ints, packed)
    out32, grads32 = _fwd_bwd(ext, [a.float() for a in acts], w, b, go.float(), ints, packed)
    assert out.dtype == F16 and torch.equal(out, out32.half())
    for i, (g, g32) in enumerate(zip(grads, grads32)):
        if i < len(acts):
            assert g.dtype == F16 and torch.equal(g, g32.half()), i
        else:
            assert g.dtype == torch.float32 and torch.equal(g, g32), i


def _fac(x, ker, go, K):
    from ebfi_be_b200 import kernelconv2d
    xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
    out = kernelconv2d.KernelConv2DFunction.apply(xg, kg, K)
    out.backward(go)
    return out.detach(), xg.grad, kg.grad


def _fac_case(shape, seed):
    B, C, K, H, W = shape
    g = torch.Generator().manual_seed(seed)
    return (_h(torch.randn(B, C, H + K - 1, W + K - 1, generator=g)), _h(torch.randn(B, C * K * K, H, W, generator=g)),
            _h(torch.randn(B, C, H, W, generator=g)))


# (B, C, K, H, W): one row segment per plane (H <= 16), vector and scalar column paths, odd widths
FAC_SHAPES = [(2, 3, 5, 16, 64), (1, 2, 5, 13, 23), (2, 2, 3, 16, 36), (1, 3, 3, 9, 7), (1, 2, 1, 12, 16),
              (1, 2, 1, 7, 5), (1, 1, 5, 16, 300)]


@pytest.mark.parametrize("shape", FAC_SHAPES)
def test_fac_bit_identical_to_fp32_kernels(shape):
    K = shape[2]
    x, ker, go = _fac_case(shape, sum(shape))
    got = _fac(x, ker, go, K)
    want = _fac(x.float(), ker.float(), go.float(), K)
    for name, a, b in zip(("out", "grad_input", "grad_kernel"), got, want):
        assert a.dtype == F16 and torch.equal(a, b.half()), name


def test_fac_row_segments_round_the_seam_rows_twice():
    """With several row segments per plane, the K-1 grad_input rows at each segment seam are the sum of one segment's
    stored (already rounded) partial and the other's fp32 overhang, rounded again, as in the bf16 variant: there the
    result is within two fp16 roundings (2^-10 of max|grad_input|) of the fp32 result; everywhere else it is the fp32
    result rounded once."""
    B, C, K, H, W = 1, 2, 5, 40, 64
    x, ker, go = _fac_case((B, C, K, H, W), 5)
    got = _fac(x, ker, go, K)
    want = _fac(x.float(), ker.float(), go.float(), K)
    assert torch.equal(got[0], want[0].half()) and torch.equal(got[2], want[2].half())
    gi, gi32 = got[1].float(), want[1].half().float()
    seams = torch.zeros(H + K - 1, dtype=torch.bool)
    for yb in range(16, H, 16):
        seams[yb:yb + K - 1] = True
    assert torch.equal(gi[:, :, ~seams], gi32[:, :, ~seams])
    assert float((gi - want[1]).abs().max()) <= 2.0 ** -10 * float(want[1].abs().max())


@pytest.mark.parametrize("shape", KPN_SHAPES + KPN_PIPELINE_SHAPES)
def test_kpn_bit_identical_to_fp32_kernels(mod, shape):
    from gpu_util import t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b = _kpn_case(np.random.default_rng(sum(shape)), *shape)
    G = np.random.default_rng(sum(shape) + 1).standard_normal(ev.shape).astype(np.float32)
    evh, frh, wt, bt, Gh = t(ev).half(), t(fr).half(), t(w), t(b), t(G).half()
    with torch.no_grad():
        out = mod._fused_forward(evh, frh, wt, bt, K, SLOPE)
        assert out.dtype == F16
        assert torch.equal(out, mod._fused_forward(evh.float(), frh.float(), wt, bt, K, SLOPE).half())
        pub = mod.kernelconv_fac_fused(evh, frh, wt.half(), bt.half(), K, SLOPE)      # a .half() model
        assert torch.equal(pub, mod._fused_forward(evh.float(), frh.float(), wt.half().float(), bt.half().float(), K,
                                                   SLOPE).half())
    got = mod.kernelconv_fac_fused_backward_bf16(evh, frh, wt, bt, K, SLOPE, Gh)
    assert [x.dtype for x in got] == [F16, torch.float32, torch.float32]
    want = mod.kernelconv_fac_fused_backward(evh.float(), frh.float(), wt, bt, K, SLOPE, Gh.float())
    assert torch.equal(got[0], want[0].half())
    assert torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])


# ---------------------------------------------------------------- 2. precision against the fp64 oracle
def test_dcn_precision_against_fp64_oracle(ext, oracle):
    """Each result within one fp16 rounding (2^-11 of its max) of the fp64 oracle, on top of the fp32 kernels' own
    error on the same values."""
    shape = (1, 64, 64, 20, 24, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _dcn_case(shape, 15, obound=2.0)
    out, grads = _fwd_bwd(ext, (x, off, m), w, b, go, ints, False)
    out32, grads32 = _fwd_bwd(ext, (x.float(), off.float(), m.float()), w, b, go.float(), ints, False)
    f = lambda t: t.float().cpu().numpy()
    want = [oracle.dcn_forward(f(x), f(off), f(m), f(w), f(b), 1, 1, 1, 8)]
    want += list(oracle.dcn_backward(f(x), f(off), f(m), f(w), f(b), f(go), 1, 1, 1, 8))
    for i, (g, g32, r) in enumerate(zip([out] + list(grads), [out32] + list(grads32), want)):
        e16, e32 = rel_err(f(g), r), rel_err(f(g32), r)
        print(i, "rel err fp16 %.3g fp32 %.3g" % (e16, e32))
        assert e16 <= F16_TOL + e32, i


def test_fac_precision_against_fp64_oracle(oracle):
    K = 5
    x, ker, go = _fac_case((2, 3, K, 16, 64), 16)
    got = _fac(x, ker, go, K)
    got32 = _fac(x.float(), ker.float(), go.float(), K)
    f = lambda t: t.float().cpu().numpy()
    want = [oracle.fac_forward(f(x), f(ker), K)] + list(oracle.fac_backward(f(x), f(ker), f(go), K))
    for i, (g, g32, r) in enumerate(zip(got, got32, want)):
        assert rel_err(f(g), r) <= F16_TOL + rel_err(f(g32), r), i


def test_kpn_precision_against_fp64_oracle(mod, oracle, monkeypatch):
    """The fused kernels on fp16 inputs against the fp64 block with bf16 conv operands (the kernels' own operands):
    one fp16 rounding on top of the fp32 kernels' error on the same values."""
    from gpu_util import n, t
    shape = (1, 64, 64, 16, 8, 5)
    K = shape[-1]

    def rounded_case(rng, *s):
        ev, fr, w, b = _kpn_case(rng, *s)
        return (ev.astype(np.float16).astype(np.float32), fr.astype(np.float16).astype(np.float32), w, b)
    monkeypatch.setattr(TG, "_case", rounded_case)
    ev, fr, w, b, G = TG._separated_case(shape)
    G = G.astype(np.float16).astype(np.float32)
    want_out, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, SLOPE, bf16_operands=True)
    gev_fac, _, _, gbias, gpre, _ = KO.backward_parts(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    with torch.no_grad():
        out = mod._fused_forward(t(ev).half(), t(fr).half(), t(w), t(b), K, SLOPE)
        out32 = mod._fused_forward(t(ev), t(fr), t(w), t(b), K, SLOPE)
    got = mod.kernelconv_fac_fused_backward_bf16(t(ev).half(), t(fr).half(), t(w), t(b), K, SLOPE, t(G).half())
    got32 = mod.kernelconv_fac_fused_backward(t(ev), t(fr), t(w), t(b), K, SLOPE, t(G))
    for name, g, g32, r in (("out", out, out32, want_out), ("grad_pre", got[0], got32[0], gpre),
                            ("grad_event_fac", got[1], got32[1], gev_fac), ("grad_bias", got[2], got32[2], gbias)):
        assert rel_err(n(g.float()), r) <= F16_TOL + rel_err(n(g32), r), name


# ---------------------------------------------------------------- 3. overflow
def test_overflow_gives_inf(ext):
    """fp16 results beyond 65504 are +-inf (what tensor.half() gives and GradScaler looks for), not a saturated finite
    value and not NaN: a DCN output channel with a huge bias, a FAC grad_kernel of large factors."""
    shape = (1, 64, 64, 24, 24, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _dcn_case(shape, 17)
    b = b.clone()
    b[3], b[5] = 1e5, -1e5
    out = ext.dcn_v2_forward(x, w, b, off, m, *ints)
    assert bool(torch.isposinf(out[:, 3]).all()) and bool(torch.isneginf(out[:, 5]).all())
    keep = [c for c in range(64) if c not in (3, 5)]
    assert bool(torch.isfinite(out[:, keep]).all())
    assert torch.equal(out, ext.dcn_v2_forward(x.float(), w, b, off.float(), m.float(), *ints).half())

    K = 3
    x, ker, go = _fac_case((1, 2, K, 12, 16), 18)
    x[0, 0] = 300.0
    go[0, 0] = 300.0
    _, _, gk = _fac(x, ker, go, K)
    assert bool(torch.isposinf(gk[0, :K * K]).all())               # 90000 per element
    assert bool(torch.isfinite(gk[0, K * K:]).all())


def test_grad_scaler_backs_off_then_trains():
    """DCN_sep under fp16 autocast with a GradScaler whose initial scale overflows the fp16 gradients: the first step
    is skipped (parameters unchanged) and the scale backs off; the loop then trains to finite parameters and a loss
    well below the start."""
    from ebfi_be_b200 import dcn_v2
    torch.manual_seed(41)
    teacher = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
    with torch.no_grad():
        teacher.conv_offset_mask.weight.normal_(0, 0.05)
    g = torch.Generator().manual_seed(42)
    data = [(torch.randn(2, 64, 24, 24, generator=g).to(_dev()), torch.randn(2, 64, 24, 24, generator=g).to(_dev()))
            for _ in range(4)]
    with torch.no_grad():
        targets = [teacher(x, f) for x, f in data]
    s = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
    opt = torch.optim.Adam(s.parameters(), lr=2e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40)
    losses, skipped = [], 0
    for it in range(150):
        x, f = data[it % 4]
        with torch.autocast("cuda"):
            out = s(x, f)
            assert out.dtype == F16
            loss = torch.nn.functional.mse_loss(out.float(), targets[it % 4])
        opt.zero_grad()
        before = [p.detach().clone() for p in s.parameters()]
        scale = scaler.get_scale()
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        if scaler.get_scale() < scale:
            skipped += 1
            assert all(torch.equal(p, q) for p, q in zip(s.parameters(), before))
        if it == 0:
            assert scaler.get_scale() == 2.0 ** 39
        losses.append(float(loss))
    s.flush_offset_warnings()
    print("GradScaler: skipped", skipped, "final scale", scaler.get_scale(), "loss", losses[0], losses[-1])
    assert skipped >= 1
    assert all(bool(torch.isfinite(p).all()) for p in s.parameters())
    assert np.mean(losses[-4:]) < 0.5 * np.mean(losses[:4])


# ---------------------------------------------------------------- 4. modules under torch.autocast("cuda")
KINDS = ["DCNv2", "DCN", "DCN_sep", "DCN_sep_unfused"]
# relative L2 against the fp32 module, the bounds of the bf16 tests (fp16 keeps 3 more mantissa bits)
REL_L2_DCN, REL_L2_OFFSET_PATH = 0.01, 0.1


@pytest.mark.parametrize("in_dtype", [torch.float32, F16])
@pytest.mark.parametrize("kind", KINDS)
def test_dcn_modules_under_autocast(kind, in_dtype):
    m = _module(kind, 21)
    g = torch.Generator().manual_seed(22)
    x0 = torch.randn(2, 64, 24, 32, generator=g).to(_dev())
    f0 = torch.randn(2, 64, 24, 32, generator=g).to(_dev())
    go = torch.randn(2, 64, 24, 32, generator=g).to(_dev())

    def run(autocast):
        m.zero_grad(set_to_none=True)
        x = x0.clone().to(in_dtype).requires_grad_()
        fea = f0.clone().to(in_dtype).requires_grad_()
        with torch.autocast("cuda", enabled=autocast):
            out = _forward(kind, m, x, fea)
        out.backward(go.to(out.dtype))
        return out, x.grad, fea.grad, {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}

    out, gx, gf, gp = run(True)
    assert out.dtype == F16
    assert gx.dtype == in_dtype and (gf is None or gf.dtype == in_dtype)
    assert gp and all(v.dtype == torch.float32 for v in gp.values())
    if in_dtype == torch.float32:
        ref_out, ref_gx, ref_gf, ref_gp = run(False)
        errs = {"out": _rel_l2(out.float(), ref_out), "input": _rel_l2(gx, ref_gx)}
        if gf is not None:
            errs["fea"] = _rel_l2(gf, ref_gf)
        errs.update({n: _rel_l2(v, ref_gp[n]) for n, v in gp.items()})
        print(kind, "relative L2 vs fp32:", {k: round(v, 5) for k, v in errs.items()})
        for k, v in errs.items():
            assert v < (REL_L2_DCN if k in ("out", "weight", "bias") else REL_L2_OFFSET_PATH), (k, errs)
    if hasattr(m, "flush_offset_warnings"):
        m.flush_offset_warnings()


def test_kernelconv2d_under_autocast():
    """KernelConv2D fed by 16-bit convolutions under autocast (the reference model's pattern)."""
    from ebfi_be_b200.kernelconv2d import KernelConv2D
    torch.manual_seed(23)
    conv_e = torch.nn.Conv2d(16, 8, 3, 1, 1).to(_dev())
    conv_k = torch.nn.Conv2d(16, 8 * 25, 3, 1, 1).to(_dev())
    kpn = KernelConv2D(5)
    feat0 = torch.randn(2, 16, 24, 20, device=_dev())
    go = torch.randn(2, 8, 24, 20, device=_dev())

    def run(autocast):
        feat = feat0.clone().requires_grad_()
        conv_e.zero_grad(set_to_none=True)
        conv_k.zero_grad(set_to_none=True)
        with torch.autocast("cuda", enabled=autocast):
            out = kpn(conv_e(feat), conv_k(feat))
        out.backward(go.to(out.dtype))
        return out, feat.grad, conv_e.weight.grad.clone(), conv_k.weight.grad.clone()

    got, ref = run(True), run(False)
    assert got[0].dtype == F16 and [g.dtype for g in got[1:]] == [torch.float32] * 3
    for name, a, b in zip(("out", "feat", "conv_e.weight", "conv_k.weight"), got, ref):
        assert _rel_l2(a.float(), b) < REL_L2_DCN, name


def _kpn_grads(m, ev, fr, G, autocast):
    conv = m.KernelConv.conv2d
    m.zero_grad(set_to_none=True)
    e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
    with torch.autocast("cuda", enabled=autocast):
        out = m(e, f)
    out.backward(G.to(out.dtype))
    return out.detach(), e.grad, f.grad, conv.weight.grad.clone(), conv.bias.grad.clone()


def test_kernel_prediction_under_autocast(mod):
    """KernelPrediction(32, 5), fp32 parameters, fp16 event and frame tensors under autocast: the op sequence
    (fused paths off) and fused_backward (KernelConvFACBF16Function, bit-equal to a direct call), with the dtypes
    autocast's op sequence gives; the fused inference path of a .half() model. Relative L2 against the fp32 module on
    the same values."""
    from gpu_util import dev
    torch.manual_seed(24)
    m = mod.KernelPrediction(32, 5).to(dev())
    conv = m.KernelConv.conv2d
    ev = torch.randn(2, 32, 40, 24, device=dev()).half()
    fr = torch.randn(2, 32, 40, 24, device=dev()).half()
    G = torch.randn(2, 32, 40, 24, device=dev()).half()
    m.fused, m.fused_backward = False, False
    ref = _kpn_grads(m, ev.float(), fr.float(), G.float(), False)
    seq = _kpn_grads(m, ev, fr, G, True)
    m.fused_backward = True
    fused = _kpn_grads(m, ev, fr, G, True)
    for got in (seq, fused):
        assert [x.dtype for x in got] == [F16, F16, F16, torch.float32, torch.float32]
    e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
    m.zero_grad(set_to_none=True)
    out = mod.KernelConvFACBF16Function.apply(e, f, conv.weight, conv.bias, 5, m.KernelConv.activation.negative_slope)
    out.backward(G)
    for name, x, y in zip(("out", "event", "frame", "weight", "bias"), fused,
                          (out.detach(), e.grad, f.grad, conv.weight.grad, conv.bias.grad)):
        assert torch.equal(x, y), name
    mh = copy.deepcopy(m).half()
    mh.fused = True
    wh, bh = mh.KernelConv.conv2d.weight, mh.KernelConv.conv2d.bias
    with torch.no_grad(), torch.autocast("cuda"):
        inf = mh(ev, fr)
        assert inf.dtype == F16
        assert torch.equal(inf, mod._fused_forward(ev, fr, wh.float(), bh.float(), 5, SLOPE))
    for label, got in (("sequence", seq), ("fused_backward", fused)):
        errs = [_rel_l2(a.float(), b) for a, b in zip(got, ref)]
        print(label, "relative L2 vs fp32 (out, event, frame, weight, bias):", [round(x, 5) for x in errs])
        assert errs[0] < 0.02 and max(errs[1:]) < 0.1, (label, errs)
    assert _rel_l2(inf.float(), ref[0]) < 0.02


# ---------------------------------------------------------------- 5. training fits with GradScaler
def test_dcn_sep_adam_grad_scaler_fit():
    """A DCN_sep student fitted by Adam under fp16 autocast with a GradScaler reaches the fp32 fit's loss within 10 %."""
    from ebfi_be_b200 import dcn_v2
    torch.manual_seed(31)
    teacher = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
    with torch.no_grad():
        teacher.conv_offset_mask.weight.normal_(0, 0.05)
    g = torch.Generator().manual_seed(32)
    data = [(torch.randn(2, 64, 24, 24, generator=g).to(_dev()), torch.randn(2, 64, 24, 24, generator=g).to(_dev()))
            for _ in range(4)]
    with torch.no_grad():
        targets = [teacher(x, f) for x, f in data]

    def fit(autocast):
        torch.manual_seed(33)
        s = dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8).to(_dev())
        opt = torch.optim.Adam(s.parameters(), lr=2e-3)
        scaler = torch.amp.GradScaler("cuda", enabled=autocast)
        for it in range(120):
            x, f = data[it % 4]
            with torch.autocast("cuda", enabled=autocast):
                loss = torch.nn.functional.mse_loss(s(x, f).float(), targets[it % 4])
            opt.zero_grad()
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        with torch.no_grad():
            return sum(float(torch.nn.functional.mse_loss(s(x, f), t)) for (x, f), t in zip(data, targets)) / 4

    start = sum(float(t.pow(2).mean()) for t in targets) / 4
    l32, l16 = fit(False), fit(True)
    print("Adam + GradScaler fit: start %.5f fp32 %.5f fp16 autocast %.5f" % (start, l32, l16))
    assert l32 < 0.5 * start
    assert l16 < 1.1 * l32 + 1e-3 * start, (l16, l32, start)


def test_kpn_block_adam_grad_scaler_fit(mod):
    """fused_backward student vs op-sequence student, both under fp16 autocast with a GradScaler: same init and data,
    the fused one halves its loss and ends within 10 % of the sequence's."""
    from gpu_util import dev
    torch.manual_seed(11)
    teacher = mod.KernelPrediction(32, 5).to(dev())
    base = mod.KernelPrediction(32, 5).to(dev())
    data = [(torch.randn(2, 32, 32, 32, device=dev()).half(), torch.randn(2, 32, 32, 32, device=dev()).half())
            for _ in range(4)]
    with torch.no_grad(), torch.autocast("cuda"):
        targets = [teacher(e, f).float() for e, f in data]
    losses = {}
    for fused in (False, True):
        student = mod.KernelPrediction(32, 5).to(dev())
        student.load_state_dict(base.state_dict())
        student.fused_backward = fused
        opt = torch.optim.Adam(student.parameters(), lr=1e-3)
        scaler = torch.amp.GradScaler("cuda")
        hist = []
        for step in range(40):
            e, f = data[step % 4]
            with torch.autocast("cuda"):
                loss = torch.nn.functional.mse_loss(student(e, f).float(), targets[step % 4])
            opt.zero_grad()
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
            hist.append(float(loss))
        losses[fused] = hist
    print("loss first/last: sequence", losses[False][0], losses[False][-1], "fused", losses[True][0], losses[True][-1])
    assert losses[True][-1] < 0.5 * losses[True][0]
    assert losses[True][-1] <= 1.1 * losses[False][-1]


# ---------------------------------------------------------------- 6. fallbacks keep the dtypes
@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("name,shape,env,gin_exact", [f for f in FALLBACKS if f[0] in ("cout32", "deterministic", "simt")],
                         ids=["cout32", "deterministic", "simt"])
def test_fallbacks_return_native_dtypes(ext, monkeypatch, name, shape, env, gin_exact, packed):
    """Where the fp16 kernels decline (Cout = 32 backward, EBFI_DCN_DETERMINISTIC, EBFI_DCN_IMPL=simt) the call
    converts at the boundary: the same dtypes as the native path and the bits of _via_fp32 (grad_input of the CUDA-core
    kernel, which adds with float atomics, at the fp16 tolerance)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    acts, w, b, go, ints = _dcn_case(shape, 13, packed)
    out, grads = _fwd_bwd(ext, acts, w, b, go, ints, packed)
    dts = [F16] * len(acts) + [torch.float32] * 2
    if packed:
        ref_out = ext._via_fp32(F16, ext.dcn_v2_forward_packed, (acts[0], w, b, acts[1]), ints)
        ref = ext._via_fp32(F16, ext.dcn_v2_backward_packed, (acts[0], w, b, acts[1], go), ints, dts)
    else:
        ref_out = ext._via_fp32(F16, ext.dcn_v2_forward, (acts[0], w, b, *acts[1:]), ints)
        ref = ext._via_fp32(F16, ext.dcn_v2_backward, (acts[0], w, b, acts[1], acts[2], go), ints, dts)
    assert out.dtype == F16 and torch.equal(out, ref_out)
    assert [g.dtype for g in grads] == dts
    for i, (g, r) in enumerate(zip(grads, ref)):
        if i == 0 and not gin_exact:
            assert rel_err(g.float().cpu().numpy(), r.float().cpu().numpy()) < F16_TOL
        else:
            assert torch.equal(g, r), i


# ---------------------------------------------------------------- 7. errors
def test_errors(ext, mod):
    shape = (1, 64, 64, 16, 16, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _dcn_case(shape, 61)
    for bad in (x.bfloat16(), x.double()):
        with pytest.raises(RuntimeError, match="must be float32"):
            ext.dcn_v2_forward(bad, w, b, off, m, *ints)
        with pytest.raises(RuntimeError, match="must be float32"):
            ext.dcn_v2_backward(x, w, b, off, m, go.to(bad.dtype), *ints)
    with pytest.raises(RuntimeError, match="must be float32"):
        ext.dcn_v2_forward(x, w.bfloat16(), b, off, m, *ints)             # fp16 activations, bf16 weight
    with pytest.raises(RuntimeError, match="float16"):
        _fac(x[:, :2, :12, :12].contiguous(), off[:, :18, :10, :10].bfloat16().contiguous(),
             go[:, :2, :10, :10].contiguous(), 3)
    ev = torch.randn(1, 32, 8, 8, device=_dev()).half()
    fr = torch.randn(1, 32, 8, 8, device=_dev()).half()
    wk = torch.randn(800, 64, 3, 3, device=_dev(), requires_grad=True)
    bk = torch.zeros(800, device=_dev(), requires_grad=True)
    with pytest.raises(RuntimeError, match="float16"):
        mod.KernelConvFACBF16Function.apply(ev, fr.bfloat16(), wk, bk, 5)
    with pytest.raises(RuntimeError, match="float16"):
        mod.KernelConvFACBF16Function.apply(ev.double(), fr.double(), wk, bk, 5)
    with pytest.raises(RuntimeError, match="float32 or torch.float16"):
        mod.KernelConvFACBF16Function.apply(ev, fr, wk.detach().bfloat16(), bk.detach().bfloat16(), 5)
    with pytest.raises(RuntimeError, match="float16"):
        mod.kernelconv_fac_fused(ev, fr.bfloat16(), wk.detach().half(), bk.detach().half(), 5)
