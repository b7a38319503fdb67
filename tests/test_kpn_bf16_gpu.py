"""bf16 activation I/O of the fused KernelConv -> FAC block (csrc/kpn.cu instantiated for __nv_bfloat16:
ebfi_kpn_fused_forward_bf16 / ebfi_kpn_fused_backward_bf16; KernelConvFACBF16Function and KernelPrediction under
torch.autocast). The bf16 instantiations only convert at the loads and round once at the stores, so on bf16-valued
inputs they must equal the fp32 kernel bit for bit; the autograd Function is checked against the float64
restatement in tests/kpn_train_oracle.py and against autocast's op sequence."""
import numpy as np
import pytest
import torch

import kpn_train_oracle as KO
import test_kpn_train_gpu as TG
from conftest import rel_err
from oracle.oracle import _bf16_round
from test_kpn_gpu import PIPELINE_SHAPES, SHAPES, _case

pytestmark = pytest.mark.gpu

SLOPE = 0.01
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def mod():
    from ebfi_be_b200 import modification
    return modification


def _autocast():
    return torch.autocast("cuda", dtype=BF16)


@pytest.mark.parametrize("shape", SHAPES + PIPELINE_SHAPES)
def test_forward_bit_identical_to_fp32_kernel(mod, shape):
    from gpu_util import t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b = _case(np.random.default_rng(sum(shape)), *shape)
    evb, frb, wt, bt = t(ev).to(BF16), t(fr).to(BF16), t(w), t(b)
    with torch.no_grad():
        got = mod._fused_forward(evb, frb, wt, bt, K, SLOPE)
        assert got.dtype == BF16
        assert torch.equal(got, mod._fused_forward(evb.float(), frb.float(), wt, bt, K, SLOPE).to(BF16))
        # public all-bf16 entry (a .bfloat16() model): same as staging every tensor through fp32
        wb, bb = wt.to(BF16), bt.to(BF16)
        pub = mod.kernelconv_fac_fused(evb, frb, wb, bb, K, SLOPE)
        assert pub.dtype == BF16
        assert torch.equal(pub, mod._fused_forward(evb.float(), frb.float(), wb.float(), bb.float(), K, SLOPE).to(BF16))


@pytest.mark.parametrize("shape", SHAPES + PIPELINE_SHAPES)
def test_backward_bit_identical_to_fp32_kernel(mod, shape):
    from gpu_util import t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b = _case(np.random.default_rng(sum(shape)), *shape)
    G = np.random.default_rng(sum(shape) + 1).standard_normal(ev.shape).astype(np.float32)
    evb, frb, wt, bt, Gb = t(ev).to(BF16), t(fr).to(BF16), t(w), t(b), t(G).to(BF16)
    got = mod.kernelconv_fac_fused_backward_bf16(evb, frb, wt, bt, K, SLOPE, Gb)
    assert [x.dtype for x in got] == [BF16, torch.float32, torch.float32]
    gpre, gev, gbias = mod.kernelconv_fac_fused_backward(evb.float(), frb.float(), wt, bt, K, SLOPE, Gb.float())
    assert torch.equal(got[0], gpre.to(BF16))
    assert torch.equal(got[1], gev)
    assert torch.equal(got[2], gbias)
    again = mod.kernelconv_fac_fused_backward_bf16(evb, frb, wt, bt, K, SLOPE, Gb)
    for x, y in zip(got, again):
        assert torch.equal(x, y)


def _bf16_separated_case(shape, monkeypatch):
    """test_kpn_train_gpu._separated_case with event, frame, weight (and G) rounded to bf16 before the bias shift:
    every input but the (fp32) bias is bf16-valued, and no pre-activation lies near zero."""
    def rounded_case(rng, *s):
        ev, fr, w, b = _case(rng, *s)
        return _bf16_round(ev), _bf16_round(fr), _bf16_round(w), b
    monkeypatch.setattr(TG, "_case", rounded_case)
    ev, fr, w, b, G = TG._separated_case(shape)
    return ev, fr, w, b, _bf16_round(G)


@pytest.mark.parametrize("shape", SHAPES)
def test_function_against_oracle(mod, oracle, shape, monkeypatch):
    """fp32 parameters and bf16 activations, as autocast hands them over. Output and dL/dP are rounded once to bf16
    and the conv's gradients come from a bf16 convolution backward, hence the bf16-sized bounds; grad_bias is summed
    in fp32 from the unrounded dL/dP."""
    from gpu_util import n, t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b, G = _bf16_separated_case(shape, monkeypatch)
    want_out, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, SLOPE, bf16_operands=True)
    want = KO.kpn_fused_backward(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    leaves = [t(ev).to(BF16), t(fr).to(BF16), t(w), t(b)]
    leaves = [x.requires_grad_() for x in leaves]
    out = mod.KernelConvFACBF16Function.apply(*leaves, K, SLOPE)
    assert out.dtype == BF16
    assert rel_err(n(out.float()), want_out) <= 2.0 ** -8
    out.backward(t(G).to(BF16))
    assert [x.grad.dtype for x in leaves] == [BF16, BF16, torch.float32, torch.float32]
    assert rel_err(n(leaves[3].grad), want[3]) <= 1e-5                       # grad_bias
    assert rel_err(n(leaves[0].grad.float()), want[0]) <= 2.0 ** -7          # grad_event
    if Cf:
        assert rel_err(n(leaves[1].grad.float()), want[1]) <= 2.0 ** -7      # grad_frame
    assert rel_err(n(leaves[2].grad), want[2]) <= 2.0 ** -7                  # grad_weight


def test_full_size_one_hot_kernels_exact(mod):
    """BASELINE cfg2 size (B=4, C=64, K=5, 256x256), bf16 activations, zero conv weights and a one-hot bias per
    channel (the construction of test_kpn_train_gpu.test_full_size_one_hot_kernels_exact): the output is the
    replication-padded input shifted by the tap, dL/dP is G*Epad on the tap and G*Epad*slope off it (each rounded once
    from fp32), and the FAC part of dL/dEvent is G shifted back by the tap."""
    from gpu_util import dev
    torch.manual_seed(2)
    B, C, K, H, W = 4, 64, 5, 256, 256
    R, KK = 2, 25
    ev = torch.randn(B, C, H, W, device=dev()).to(BF16)
    fr = torch.randn(B, C, H, W, device=dev()).to(BF16)
    G = torch.randn(B, C, H, W, device=dev()).to(BF16)
    w = torch.zeros(C * KK, 2 * C, 3, 3, device=dev())
    bias = torch.zeros(C, KK, device=dev())
    taps = torch.arange(C, device=dev()) % KK
    bias[torch.arange(C, device=dev()), taps] = 1.0
    bias = bias.reshape(-1)
    evp = torch.nn.functional.pad(ev.float(), (R, R, R, R), mode="replicate")
    with torch.no_grad():
        out = mod.kernelconv_fac_fused(ev, fr, w.to(BF16), bias.to(BF16), K, SLOPE)
    for c in (0, 7, 24, 63):
        ky, kx = int(taps[c]) // K, int(taps[c]) % K
        assert torch.equal(out[:, c], evp[:, c, ky:ky + H, kx:kx + W].to(BF16)), c
    del out

    gpre, gev_fac, gbias = mod.kernelconv_fac_fused_backward_bf16(ev, fr, w, bias, K, SLOPE, G)
    Gf = G.float()
    for c in (0, 7, 24, 63):
        tap = int(taps[c])
        for q in (tap, (tap + 1) % KK, (tap + 13) % KK):
            ky, kx = q // K, q % K
            ge = Gf[:, c] * evp[:, c, ky:ky + H, kx:kx + W]            # fp32, exact (bf16 x bf16)
            want = ge if q == tap else ge * SLOPE
            assert torch.equal(gpre[:, c * KK + q], want.to(BF16)), (c, q)
    ev_leaf = ev.float().requires_grad_()
    pad = torch.nn.functional.pad(ev_leaf, (R, R, R, R), mode="replicate")
    ky, kx = taps // K, taps % K
    shifted = torch.stack([pad[:, c, int(ky[c]):int(ky[c]) + H, int(kx[c]):int(kx[c]) + W] for c in range(C)], 1)
    (shifted * Gf).sum().backward()
    inner = (slice(None), slice(None), slice(R, H - R), slice(R, W - R))
    assert torch.equal(gev_fac[inner], ev_leaf.grad[inner])


def _rel_l2(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / np.linalg.norm(want))


def _grads(m, ev, fr, G, fused):
    """forward under autocast, backward outside it: (out, grad_event, grad_frame, grad_weight, grad_bias)"""
    conv = m.KernelConv.conv2d
    m.fused_backward = fused
    m.zero_grad(set_to_none=True)
    e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
    with _autocast():
        out = m(e, f)
    out.backward(G)
    return out.detach(), e.grad, f.grad, conv.weight.grad.clone(), conv.bias.grad.clone()


def test_module_under_autocast(mod):
    """KernelPrediction(64, 5) with fp32 parameters and bf16 activations under autocast. fused_backward = True runs
    KernelConvFACBF16Function (bit-equal to a direct call, whose backward here runs inside autocast: the result must
    not depend on it), with the gradient dtypes autocast's op sequence gives. Each gradient's relative L2 error
    against the unrounded fp64 block is compared with the sequence's (fused_backward = False)."""
    from gpu_util import dev, n
    torch.manual_seed(5)
    m = mod.KernelPrediction(64, 5).to(dev())
    conv = m.KernelConv.conv2d
    ev = torch.randn(2, 64, 40, 32, device=dev()).to(BF16)
    fr = torch.randn(2, 64, 40, 32, device=dev()).to(BF16)
    G = torch.randn(2, 64, 40, 32, device=dev()).to(BF16)
    fused = _grads(m, ev, fr, G, True)
    assert [x.dtype for x in fused] == [BF16, BF16, BF16, torch.float32, torch.float32]

    m.zero_grad(set_to_none=True)
    e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
    with _autocast():
        out = mod.KernelConvFACBF16Function.apply(e, f, conv.weight, conv.bias, 5, m.KernelConv.activation.negative_slope)
        out.backward(G)
    direct = (out.detach(), e.grad, f.grad, conv.weight.grad, conv.bias.grad)
    for name, x, y in zip(("out", "grad_event", "grad_frame", "grad_weight", "grad_bias"), fused, direct):
        assert torch.equal(x, y), name

    seq = _grads(m, ev, fr, G, False)
    assert [x.dtype for x in seq] == [x.dtype for x in fused]
    assert not torch.equal(seq[0], fused[0])                   # the two paths really differ
    want = KO.kpn_fused_backward(n(ev.float()), n(fr.float()), n(conv.weight.detach()), n(conv.bias.detach()), 5,
                                 m.KernelConv.activation.negative_slope, n(G.float()))
    errs = {k: [_rel_l2(n(x.float()), y) for x, y in zip(v[1:], want[:4])] for k, v in (("seq", seq), ("fused", fused))}
    print("rel L2 vs fp64 under autocast (event, frame, weight, bias): sequence", errs["seq"], "fused", errs["fused"])
    for name, s, f in zip(("grad_event", "grad_frame", "grad_weight", "grad_bias"), errs["seq"], errs["fused"]):
        assert f <= 1.25 * s, name


def test_bf16_model_parameters(mod):
    """A .bfloat16() model (bf16 parameters) with fused_backward takes the same Function; its parameter gradients
    come back bf16."""
    from gpu_util import dev
    torch.manual_seed(6)
    m = mod.KernelPrediction(32, 5).to(dev()).to(BF16)
    conv = m.KernelConv.conv2d
    ev = torch.randn(1, 32, 24, 16, device=dev()).to(BF16)
    fr = torch.randn(1, 32, 24, 16, device=dev()).to(BF16)
    G = torch.randn(1, 32, 24, 16, device=dev()).to(BF16)
    got = _grads(m, ev, fr, G, True)
    assert all(x.dtype == BF16 for x in got)
    m.zero_grad(set_to_none=True)
    e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
    out = mod.KernelConvFACBF16Function.apply(e, f, conv.weight, conv.bias, 5, m.KernelConv.activation.negative_slope)
    out.backward(G)
    for x, y in zip(got, (out.detach(), e.grad, f.grad, conv.weight.grad, conv.bias.grad)):
        assert torch.equal(x, y)


def test_adam_fits_a_teacher_under_autocast(mod):
    """40 Adam steps fitting a randomly initialised teacher block under autocast (bf16 activations, fp32 parameters):
    the fused-backward student reaches the autocast sequence student's loss (same init, same data) within 10 %."""
    from gpu_util import dev
    torch.manual_seed(11)
    teacher = mod.KernelPrediction(32, 5).to(dev())
    base = mod.KernelPrediction(32, 5).to(dev())
    data = [(torch.randn(2, 32, 32, 32, device=dev()).to(BF16), torch.randn(2, 32, 32, 32, device=dev()).to(BF16))
            for _ in range(4)]
    with torch.no_grad(), _autocast():
        targets = [teacher(e, f).float() for e, f in data]
    losses = {}
    for fused in (False, True):
        student = mod.KernelPrediction(32, 5).to(dev())
        student.load_state_dict(base.state_dict())
        student.fused_backward = fused
        opt = torch.optim.Adam(student.parameters(), lr=1e-3)
        hist = []
        for step in range(40):
            e, f = data[step % 4]
            with _autocast():
                loss = torch.nn.functional.mse_loss(student(e, f).float(), targets[step % 4])
            opt.zero_grad()
            loss.backward()
            opt.step()
            hist.append(float(loss))
        losses[fused] = hist
    print("loss first/last under autocast: sequence", losses[False][0], losses[False][-1],
          "fused", losses[True][0], losses[True][-1])
    assert losses[True][-1] < 0.5 * losses[True][0]
    assert losses[True][-1] <= 1.1 * losses[False][-1]


def test_memory_below_the_autocast_sequence(mod):
    """Forward + backward at B=2, 64+64 channels, 256x256, K=5 under autocast. Between forward and backward the
    sequence keeps P and the kernel tensor (bf16, B*Ce*K*K*H*W each), the fused path only its inputs: at least two
    such tensors less. The peaks differ by less: the sequence peaks in its FAC backward (P, the kernel tensor and its
    gradient live), the fused path in the bf16 convolution backward of grad_pre, which the sequence runs on its own
    dL/dP as well; cuDNN's workspace there is not the fused path's to save. Measured on a B200: 337 MB lower at this
    size, 0.84 kernel tensors (DESIGN §3); the bound asks for half a tensor."""
    from gpu_util import dev
    torch.manual_seed(7)
    B, C, H, W, K = 2, 64, 256, 256, 5
    m = mod.KernelPrediction(C, K).to(dev())
    ev = torch.randn(B, C, H, W, device=dev()).to(BF16).requires_grad_()
    fr = torch.randn(B, C, H, W, device=dev()).to(BF16).requires_grad_()
    G = torch.randn(B, C, H, W, device=dev()).to(BF16)

    def step(fused, kept=None):
        m.fused_backward = fused
        ev.grad = fr.grad = None
        m.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with _autocast():
            out = m(ev, fr)
        if kept is not None:
            kept[fused] = torch.cuda.memory_allocated() - base
        out.backward(G)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    for fused in (False, True):                                # warm-up: cuDNN algorithm choice and workspaces
        step(fused)
    kept = {}
    peak = {fused: step(fused, kept) for fused in (False, True)}
    kt_bytes = B * C * K * K * H * W * 2
    mb = lambda d: {k: round(v / 2 ** 20, 1) for k, v in d.items()}
    print("MB under autocast (False = sequence, True = fused): kept for backward", mb(kept), "peak", mb(peak),
          "kernel tensor", kt_bytes / 2 ** 20)
    assert kept[True] <= kept[False] - 2 * kt_bytes
    assert peak[True] <= peak[False] - kt_bytes // 2


def test_errors_and_fallbacks(mod):
    from gpu_util import dev
    ev = torch.randn(1, 32, 8, 8, device=dev()).to(BF16)
    fr = torch.randn(1, 32, 8, 8, device=dev()).to(BF16)
    w = torch.randn(800, 64, 3, 3, device=dev(), requires_grad=True)
    b = torch.zeros(800, device=dev(), requires_grad=True)
    with pytest.raises(RuntimeError, match="bfloat16"):
        mod.KernelConvFACBF16Function.apply(ev, fr.float(), w, b, 5)        # bf16 event, fp32 frame
    with pytest.raises(RuntimeError, match="bfloat16"):
        mod.kernelconv_fac_fused_backward_bf16(ev, fr.float(), w.detach(), b.detach(), 5, SLOPE, ev)
    with pytest.raises(RuntimeError, match="bfloat16"):
        mod.KernelConvFACBF16Function.apply(ev.float(), fr.float(), w, b, 5)  # fp32 activations
    with pytest.raises(RuntimeError, match="CUDA"):
        mod.KernelConvFACBF16Function.apply(ev.cpu(), fr.cpu(), w.detach().cpu(), b.detach().cpu(), 5)
    with pytest.raises(RuntimeError, match="multiple of 32"):
        mod.KernelConvFACBF16Function.apply(ev[:, :24], fr[:, :24], torch.randn(600, 48, 3, 3, device=dev()),
                                            torch.zeros(600, device=dev()), 5)

    m = mod.KernelPrediction(24, 5).to(dev())                 # Cin = 48: not supported -> autocast op sequence
    m.fused_backward = True
    e = torch.randn(1, 24, 8, 8, device=dev()).to(BF16).requires_grad_()
    f = torch.randn(1, 24, 8, 8, device=dev()).to(BF16).requires_grad_()
    with _autocast():
        out = m(e, f)
    out.float().sum().backward()
    assert m.KernelConv.conv2d.weight.grad is not None and m.KernelConv.conv2d.weight.grad.dtype == torch.float32
    assert e.grad is not None and e.grad.dtype == BF16
