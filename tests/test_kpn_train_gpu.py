"""Fused backward of the KernelConv -> FAC block (csrc/kpn.cu, ebfi_kpn_fused_backward; KernelConvFACFunction and
KernelPrediction.fused_backward) against the float64 restatement in tests/kpn_train_oracle.py and against torch's
autograd of the reference's op sequence."""
import numpy as np
import pytest
import torch

import kpn_train_oracle as KO
from conftest import rel_err
from test_kpn_gpu import SHAPES, _case

pytestmark = pytest.mark.gpu

SLOPE = 0.01


@pytest.fixture(scope="module")
def mod():
    from ebfi_be_b200 import modification
    return modification


@pytest.fixture
def no_tf32():
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = prev


def _separated_case(shape):
    """_case of test_kpn_gpu with each conv bias shifted so that no pre-activation (bf16 operands, fp64) lies within
    1e-3 * max|P| of zero: there fp32 and fp64 sums could take different LeakyReLU branches. The shift moves zero into
    the widest gap between the middle half of the channel's sorted values, so both branches stay well populated."""
    ev, fr, w, b = _case(np.random.default_rng(sum(shape)), *shape)
    P = KO.pre_activation(ev, fr, w, b, bf16_operands=True)
    N = P.shape[1]
    vals = np.sort(np.moveaxis(P, 1, 0).reshape(N, -1), axis=1)
    n = vals.shape[1]
    mid = vals[:, n // 4: max(n - n // 4, n // 4 + 2)]
    gaps = np.diff(mid, axis=1)
    j = gaps.argmax(1)
    centre = 0.5 * (mid[np.arange(N), j] + mid[np.arange(N), j + 1])
    b = (b - centre).astype(np.float32)
    P = KO.pre_activation(ev, fr, w, b, bf16_operands=True)
    assert np.abs(P).min() >= 1e-3 * np.abs(P).max()
    assert (P > 0).mean() > 0.2 and (P < 0).mean() > 0.2
    G = np.random.default_rng(sum(shape) + 1).standard_normal(ev.shape).astype(np.float32)
    return ev, fr, w, b, G


@pytest.mark.parametrize("shape", SHAPES)
def test_fused_backward_against_oracle(mod, shape, no_tf32):
    from gpu_util import n, t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b, G = _separated_case(shape)
    gev_fac, _, _, gbias, gpre, _ = KO.backward_parts(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    args = [t(a) for a in (ev, fr, w, b)]
    got = mod.kernelconv_fac_fused_backward(*args, K, SLOPE, t(G))
    assert rel_err(n(got[0]), gpre) <= 1e-5
    assert rel_err(n(got[1]), gev_fac) <= 1e-5
    assert rel_err(n(got[2]), gbias) <= 1e-5
    again = mod.kernelconv_fac_fused_backward(*args, K, SLOPE, t(G))
    for x, y in zip(got, again):
        assert torch.equal(x, y)                              # bit-reproducible: no float atomics

    want = KO.kpn_fused_backward(ev, fr, w, b, K, SLOPE, G, bf16_operands=True)
    leaves = [a.clone().requires_grad_() for a in args]
    out = mod.KernelConvFACFunction.apply(*leaves, K, SLOPE)
    assert torch.equal(out.detach(), mod._fused_forward(*args, K, SLOPE))
    out.backward(t(G))
    assert rel_err(n(leaves[0].grad), want[0]) <= 1e-4        # grad_event
    if Cf:
        assert rel_err(n(leaves[1].grad), want[1]) <= 1e-4    # grad_frame
    assert rel_err(n(leaves[2].grad), want[2]) <= 1e-4        # grad_weight
    assert rel_err(n(leaves[3].grad), want[3]) <= 1e-5        # grad_bias


def test_full_size_one_hot_kernels_exact(mod, no_tf32):
    """BASELINE cfg2 size (B=4, C=64, K=5, 256x256) with zero conv weights and a one-hot bias per channel (the
    construction of test_kpn_gpu.test_full_size_one_hot_kernels_shift_the_input): P is exactly 1 on the channel's
    tap and 0 elsewhere, so dL/dP = G*Epad on the tap and G*Epad*slope off it, and the FAC part of dL/dEvent is G
    shifted back by the tap."""
    from gpu_util import dev
    torch.manual_seed(2)
    B, C, K, H, W = 4, 64, 5, 256, 256
    R, KK = 2, 25
    ev, fr = torch.randn(B, C, H, W, device=dev()), torch.randn(B, C, H, W, device=dev())
    G = torch.randn(B, C, H, W, device=dev())
    w = torch.zeros(C * KK, 2 * C, 3, 3, device=dev())
    bias = torch.zeros(C, KK, device=dev())
    taps = torch.arange(C, device=dev()) % KK
    bias[torch.arange(C, device=dev()), taps] = 1.0
    bias = bias.reshape(-1)
    gpre, gev_fac, gbias = mod.kernelconv_fac_fused_backward(ev, fr, w, bias, K, SLOPE, G)
    evp = torch.nn.functional.pad(ev, (R, R, R, R), mode="replicate")
    for c in (0, 7, 24, 63):
        tap = int(taps[c])
        for q in (tap, (tap + 1) % KK, (tap + 13) % KK):
            ky, kx = q // K, q % K
            ge = G[:, c] * evp[:, c, ky:ky + H, kx:kx + W]
            got = gpre[:, c * KK + q]
            if q == tap:
                assert torch.equal(got, ge), (c, q)
            else:
                want = ge * SLOPE
                ulp = torch.abs(torch.nextafter(want, torch.full_like(want, float("inf"))) - want)
                assert bool((torch.abs(got - want) <= ulp).all()), (c, q)
    # FAC part of dL/dEvent: autograd of the replication pad and the tap's shift alone
    ev_leaf = ev.clone().requires_grad_()
    pad = torch.nn.functional.pad(ev_leaf, (R, R, R, R), mode="replicate")
    ky, kx = taps // K, taps % K
    shifted = torch.stack([pad[:, c, int(ky[c]):int(ky[c]) + H, int(kx[c]):int(kx[c]) + W] for c in range(C)], 1)
    (shifted * G).sum().backward()
    want = ev_leaf.grad
    inner = (slice(None), slice(None), slice(R, H - R), slice(R, W - R))
    assert torch.equal(gev_fac[inner], want[inner])
    border = torch.ones(H, W, dtype=torch.bool, device=dev())
    border[R:H - R, R:W - R] = False
    d = torch.abs(gev_fac - want)[:, :, border]
    assert float(d.max()) <= 1e-6 * float(torch.abs(want[:, :, border]).max())

    # weight / bias / event gradients vs autograd through the reference sequence (Conv2d -> LeakyReLU -> FAC)
    from ebfi_be_b200.kernelconv2d import KernelConv2D
    leaves = [x.clone().requires_grad_() for x in (ev, fr, w, bias)]
    P = torch.nn.functional.conv2d(torch.cat(leaves[:2], 1), leaves[2], leaves[3], padding=1)
    KernelConv2D(K)(leaves[0], torch.nn.functional.leaky_relu(P, SLOPE)).backward(G)
    ref = [x.grad for x in leaves]
    del P
    fused = [x.clone().requires_grad_() for x in (ev, fr, w, bias)]
    mod.KernelConvFACFunction.apply(*fused, K, SLOPE).backward(G)
    for i, name in ((0, "grad_event"), (2, "grad_weight"), (3, "grad_bias")):
        assert rel_err(fused[i].grad.cpu().numpy(), ref[i].cpu().numpy()) <= 1e-5, name
    assert rel_err(fused[3].grad.cpu().numpy(), gbias.cpu().numpy()) == 0.0


def _rel_l2(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / np.linalg.norm(want))


def test_module_gradients_vs_reference_training_precision(mod):
    """KernelPrediction(64, 5), default init, default torch settings (cuDNN TF32). Each gradient of the fused-backward
    path and of the reference's op sequence is compared with the unrounded fp64 block by relative L2. bf16 conv
    operands flip more LeakyReLU branches than TF32 does, so the fused error is larger: measured on a B200, the
    sequence 0.7-1.2 %, the fused path 2.2-3.8 %, a ratio of 3.0-3.1 for each of the four gradients (DESIGN §3).
    The bounds keep about a factor of two of margin."""
    from gpu_util import dev, n
    torch.manual_seed(5)
    m = mod.KernelPrediction(64, 5).to(dev())
    ev, fr = torch.randn(2, 64, 40, 32, device=dev()), torch.randn(2, 64, 40, 32, device=dev())
    G = torch.randn(2, 64, 40, 32, device=dev())
    conv = m.KernelConv.conv2d
    want = KO.kpn_fused_backward(n(ev), n(fr), n(conv.weight.detach()), n(conv.bias.detach()), 5,
                                 m.KernelConv.activation.negative_slope, n(G))
    errs = {}
    for fused in (False, True):
        m.fused_backward = fused
        m.zero_grad()
        e, f = ev.clone().requires_grad_(), fr.clone().requires_grad_()
        m(e, f).backward(G)
        got = (e.grad, f.grad, conv.weight.grad, conv.bias.grad)
        errs[fused] = [_rel_l2(n(x), y) for x, y in zip(got, want[:4])]
    print("rel L2 vs fp64 (event, frame, weight, bias): sequence", errs[False], "fused", errs[True])
    for name, s, f in zip(("grad_event", "grad_frame", "grad_weight", "grad_bias"), errs[False], errs[True]):
        assert f <= 0.08, name
        assert f <= 6 * s, name


def test_adam_fits_a_teacher_like_the_reference_sequence(mod):
    """Capability: 40 Adam steps fitting a randomly initialised teacher block. The fused-backward student reaches the
    same loss as the reference-sequence student (same init, same data) within 10 %."""
    from gpu_util import dev
    torch.manual_seed(11)
    teacher = mod.KernelPrediction(32, 5).to(dev())
    base = mod.KernelPrediction(32, 5).to(dev())
    data = [(torch.randn(2, 32, 32, 32, device=dev()), torch.randn(2, 32, 32, 32, device=dev())) for _ in range(4)]
    with torch.no_grad():
        targets = [teacher(e, f) for e, f in data]
    losses = {}
    for fused in (False, True):
        student = mod.KernelPrediction(32, 5).to(dev())
        student.load_state_dict(base.state_dict())
        student.fused_backward = fused
        opt = torch.optim.Adam(student.parameters(), lr=1e-3)
        hist = []
        for step in range(40):
            e, f = data[step % 4]
            loss = torch.nn.functional.mse_loss(student(e, f), targets[step % 4])
            opt.zero_grad()
            loss.backward()
            opt.step()
            hist.append(float(loss))
        losses[fused] = hist
    print("loss first/last: sequence", losses[False][0], losses[False][-1], "fused", losses[True][0], losses[True][-1])
    assert losses[True][-1] < 0.5 * losses[True][0]
    assert losses[True][-1] <= 1.1 * losses[False][-1]


def test_errors(mod):
    from gpu_util import dev
    m = mod.KernelPrediction(24, 5).to(dev())                 # Cin = 48: not supported -> reference sequence
    m.fused_backward = True
    ev, fr = torch.randn(1, 24, 8, 8, device=dev()), torch.randn(1, 24, 8, 8, device=dev())
    m(ev, fr).sum().backward()
    assert m.KernelConv.conv2d.weight.grad is not None
    w = torch.randn(600, 48, 3, 3, device=dev(), requires_grad=True)
    with pytest.raises(RuntimeError, match="multiple of 32"):
        mod.KernelConvFACFunction.apply(ev, fr, w, torch.zeros(600, device=dev()), 5, 0.01)
    ev, fr = torch.randn(1, 32, 8, 8, device=dev()), torch.randn(1, 32, 8, 8, device=dev())
    wb = torch.randn(800, 64, 3, 3, device=dev()).bfloat16().requires_grad_()
    with pytest.raises(RuntimeError, match="float32"):
        mod.KernelConvFACFunction.apply(ev.bfloat16(), fr.bfloat16(), wb, torch.zeros(800, device=dev()).bfloat16(), 5)
