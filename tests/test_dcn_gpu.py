"""GPU parity of DCNv2: CUDA path (through the C ABI / autograd Function) vs the CPU oracle, the
reference-generated golden vectors and the stored results of the reference's own CUDA kernels (tests/golden/ref_dcn_*).
Gates (BASELINE.json north_star): forward 1e-5, gradients 1e-4, relative to max|ref| per tensor."""
import numpy as np
import pytest
import torch

from conftest import DCN_CASES, FWD_TOL, GRAD_TOL, load_golden, rel_err

pytestmark = pytest.mark.gpu
GRADS = ["grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias"]


@pytest.fixture(scope="module")
def dcn():
    from ebfi_be_b200 import dcn_v2
    return dcn_v2


def _run(dcn, x, off, msk, w, b, go, stride, pad, dil, dg):
    from gpu_util import n, t
    ts = [t(a).requires_grad_() for a in (x, off, msk, w, b)]
    out = dcn.dcn_v2_conv(*ts, stride, pad, dil, dg)
    out.backward(t(go))
    return n(out), [n(v.grad) for v in ts]


def _geom(g):
    kh, kw, sh, sw, ph, pw, dh, dw, dg = (int(v) for v in g["geom"])
    return (sh, sw), (ph, pw), (dh, dw), dg


@pytest.mark.parametrize("case", DCN_CASES)
def test_golden_vectors(dcn, case):
    g = load_golden(case)
    s, p, d, dg = _geom(g)
    out, grads = _run(dcn, g["input"], g["offset"], g["mask"], g["weight"], g["bias"], g["grad_output"], s, p, d, dg)
    assert rel_err(out, g["output"]) < FWD_TOL
    order = ["grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias"]
    for name, got in zip(order, grads):
        assert rel_err(got, g[name]) < GRAD_TOL, name


def test_zero_offset_known_answer(dcn):
    # reference fixture testcuda.py:32-67: identity weights, zero offsets, mask 0.5 => 2*out == input
    from gpu_util import n, t
    g = load_golden("dcn_zero_offset")
    out = dcn.dcn_v2_conv(t(g["input"]), t(g["offset"]), t(g["mask"]), t(g["weight"]), t(g["bias"]), 1, 1, 1, 1)
    assert np.abs(2 * n(out) - g["input"]).max() < 1e-10


# (B, C, Co, H, W, k, stride, pad, dil, dg, offset scale)
SHAPES = [(1, 64, 64, 32, 32, 3, 1, 1, 1, 8, 2.0),      # benchmark geometry, small image
          (2, 16, 24, 19, 23, 3, 1, 1, 1, 4, 2.0),      # ragged pixels, Cout not a multiple of 4
          (1, 8, 70, 12, 12, 3, 1, 1, 1, 2, 2.0),       # two Cout tiles
          (1, 6, 5, 14, 9, 3, 2, 1, 1, 3, 1.0),         # stride 2
          (1, 4, 4, 11, 13, 3, 1, 2, 2, 1, 10.0),       # dilation 2, large offsets (far out of window)
          (2, 4, 6, 8, 8, 1, 1, 0, 1, 2, 1.5),          # 1x1 kernel
          (1, 2, 3, 9, 9, 5, 1, 2, 1, 1, 2.0),          # 5x5 kernel
          (1, 24, 8, 10, 10, 3, 1, 1, 1, 2, 2.0)]       # 12 channels/group * 9 taps > slab: two chunks


@pytest.mark.parametrize("shape", SHAPES)
def test_against_oracle(dcn, oracle, shape):
    B, C, Co, H, W, k, s, p, d, dg, osc = shape
    rng = np.random.default_rng(abs(hash(shape)) % (2 ** 32))
    Ho = (H + 2 * p - (d * (k - 1) + 1)) // s + 1
    Wo = (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = (rng.random((Co, C, k, k), dtype=np.float32) * 2 - 1) / np.sqrt(C * k * k)
    b = rng.standard_normal(Co, dtype=np.float32)
    off = (rng.standard_normal((B, 2 * dg * k * k, Ho, Wo)) * osc).astype(np.float32)
    msk = (1 / (1 + np.exp(-rng.standard_normal((B, dg * k * k, Ho, Wo))))).astype(np.float32)
    go = rng.standard_normal((B, Co, Ho, Wo), dtype=np.float32)
    out, grads = _run(dcn, x, off, msk, w, b, go, s, p, d, dg)
    assert rel_err(out, oracle.dcn_forward(x, off, msk, w, b, s, p, d, dg)) < FWD_TOL
    want = oracle.dcn_backward(x, off, msk, w, b, go, s, p, d, dg)
    for name, got, ref in zip(GRADS, grads, want):
        assert rel_err(got, ref) < GRAD_TOL, name


def test_window_edges_match_oracle(dcn, oracle):
    """Samples exactly on -1, 0, H-1, H and integer coordinates: the (-1, H) window, per-corner
    bounds and zero-weight corners of im2col_cuda.cu:38-48,180."""
    B, C, Co, H, W, dg = 1, 4, 4, 6, 7, 2
    rng = np.random.default_rng(1)
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = rng.standard_normal((Co, C, 3, 3), dtype=np.float32) * 0.2
    b = np.zeros(Co, np.float32)
    off = rng.choice(np.array([-2.0, -1.0, -0.5, 0.0, 0.5, 1.0, 2.0, 5.0, -7.0], np.float32), (B, 2 * dg * 9, H, W))
    msk = np.ones((B, dg * 9, H, W), np.float32)
    go = rng.standard_normal((B, Co, H, W), dtype=np.float32)
    out, grads = _run(dcn, x, off, msk, w, b, go, 1, 1, 1, dg)
    assert rel_err(out, oracle.dcn_forward(x, off, msk, w, b, 1, 1, 1, dg)) < FWD_TOL
    for name, got, ref in zip(GRADS, grads, oracle.dcn_backward(x, off, msk, w, b, go, 1, 1, 1, dg)):
        assert rel_err(got, ref) < GRAD_TOL, name


# (B, H, W, pad_h, pad_w, offset sigma, stride, dilation): shapes of the box backward (dcn_bwd_box.cu: C = Cout = 64, 8 channels per group)
BOX_SHAPES = [(1, 40, 56, 1, 1, 2.0, 1, 1),        # ragged tiles (40 = 5 x 8 rows, 56 = 3.5 x 16 pixels)
              (2, 33, 47, 1, 1, 1.0, 1, 1),        # odd sizes: offsets / masks read without TMA (row stride not 16-byte)
              (1, 48, 64, 1, 1, 12.0, 1, 1),       # most samples leave the 24 x 30 box: global gather / red.add fall-back
              (1, 32, 48, 2, 1, 2.0, 1, 1),        # pad_h != pad_w: the scatter's x uses pad_h (im2col_cuda.cu:368)
              (3, 24, 16, 1, 1, 3.0, 1, 1),        # one tile column, three samples
              (1, 50, 70, 1, 1, 1.5, 2, 1),        # stride 2: a tile's footprint is 17 x 33 input pixels (wider than the box: SIMT path)
              (1, 50, 36, 1, 1, 1.5, (2, 1), 1),   # stride 2 in y only: footprint 17 x 18 fits, box pitch in tiles = 16 rows
              (2, 36, 52, 2, 2, 1.5, 1, 2),        # dilation 2: footprint 12 x 20
              (1, 36, 40, 0, 0, 2.0, 1, 1)]        # no padding


# (C, dg): more than 8 channels per deformable group on the tensor-core path — the reference's own example
# DCN(64, 64, 3, deformable_groups=2) (testcuda.py:169-180) has 32; grad_offset / grad_mask sum over the group's units
@pytest.mark.parametrize("C,dg", [(64, 2), (64, 4), (32, 1), (16, 1), (96, 3)])
def test_box_backward_channels_per_group(dcn, oracle, C, dg):
    B, H, W, Co, k = 2, 36, 44, 64, 3
    rng = np.random.default_rng(C * 10 + dg)
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = (rng.random((Co, C, k, k), dtype=np.float32) * 2 - 1) / np.sqrt(C * 9)
    b = rng.standard_normal(Co, dtype=np.float32)
    off = (np.round(rng.standard_normal((B, 2 * dg * k * k, H, W)) * 2.0 * 64) / 64 + 1 / 128).astype(np.float32)
    msk = (1 / (1 + np.exp(-rng.standard_normal((B, dg * k * k, H, W))))).astype(np.float32)
    go = rng.standard_normal((B, Co, H, W), dtype=np.float32)
    out, grads = _run(dcn, x, off, msk, w, b, go, 1, 1, 1, dg)
    assert rel_err(out, oracle.dcn_forward(x, off, msk, w, b, 1, 1, 1, dg)) < FWD_TOL
    for name, got, ref in zip(GRADS, grads, oracle.dcn_backward(x, off, msk, w, b, go, 1, 1, 1, dg)):
        assert rel_err(got, ref) < GRAD_TOL, name
    out2, grads2 = _run(dcn, x, off, msk, w, b, go, 1, 1, 1, dg)              # and bit-reproducible
    for a, c in zip(grads, grads2):
        assert np.array_equal(a, c)


@pytest.mark.parametrize("shape", BOX_SHAPES)
def test_box_backward_against_oracle(dcn, oracle, shape):
    B, H, W, ph, pw, osc, stride, dil = shape
    C = Co = 64; dg = 8; k = 3
    rng = np.random.default_rng(abs(hash(shape)) % (2 ** 32))
    sh, sw = (stride, stride) if isinstance(stride, int) else stride
    Ho = (H + 2 * ph - (dil * (k - 1) + 1)) // sh + 1
    Wo = (W + 2 * pw - (dil * (k - 1) + 1)) // sw + 1
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = (rng.random((Co, C, k, k), dtype=np.float32) * 2 - 1) / 24
    b = rng.standard_normal(Co, dtype=np.float32)
    # offsets on the grid k/64 + 1/128: sampling coordinates are exact in fp32 and never integers, where grad_offset jumps
    # (a coordinate that rounds to an integer in fp32 but not in the oracle's fp64 would compare two different branches)
    off = (np.round(rng.standard_normal((B, 2 * dg * k * k, Ho, Wo)) * osc * 64) / 64 + 1 / 128).astype(np.float32)
    msk = (1 / (1 + np.exp(-rng.standard_normal((B, dg * k * k, Ho, Wo))))).astype(np.float32)
    go = rng.standard_normal((B, Co, Ho, Wo), dtype=np.float32)
    out, grads = _run(dcn, x, off, msk, w, b, go, (sh, sw), (ph, pw), dil, dg)
    assert rel_err(out, oracle.dcn_forward(x, off, msk, w, b, (sh, sw), (ph, pw), dil, dg)) < FWD_TOL
    for name, got, ref in zip(GRADS, grads, oracle.dcn_backward(x, off, msk, w, b, go, (sh, sw), (ph, pw), dil, dg)):
        assert rel_err(got, ref) < GRAD_TOL, name


def test_grad_input_is_bit_reproducible_by_default(dcn):
    """Default mode, no flag: samples inside the staged box accumulate in shared-memory fixed point and the per-tile boxes
    are summed in a fixed order, so ALL five gradients are bit-identical run to run (512 tiles: 7 per CTA)."""
    from gpu_util import dev
    torch.manual_seed(4)
    B, C, H, W, dg = 1, 64, 256, 256, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    go = torch.randn(B, 64, H, W, device=dev())
    runs = []
    for i in range(3):
        ts = [v.clone().requires_grad_() for v in (x, off, msk, w, b)]
        dcn.dcn_v2_conv(*ts, 1, 1, 1, dg).backward(go)
        runs.append([v.grad.clone() for v in ts])
        torch.zeros(64 << 20, device=dev())                  # perturb the cache / timing state between runs
    for r in runs[1:]:
        for i in range(5):
            assert torch.equal(r[i], runs[0][i]), GRADS[i]


def test_grad_input_scale_invariance(dcn):
    """The fixed-point scale follows the data: gradients 1e-12 .. 1e12 keep the same relative accuracy."""
    from gpu_util import dev
    torch.manual_seed(6)
    B, C, H, W, dg = 1, 64, 32, 48, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    go = torch.randn(B, 64, H, W, device=dev())
    ref = None
    for sc in (1.0, 2.0 ** -20, 2.0 ** 20, 2.0 ** -100, 2.0 ** 90, 1e-12, 1e12):
        xi = x.clone().requires_grad_()
        dcn.dcn_v2_conv(xi, off, msk, w, b, 1, 1, 1, dg).backward(go * sc)
        g = xi.grad.double() / sc
        if ref is None:
            ref = g
        elif sc in (1e-12, 1e12):       # go * sc rounds: the bf16 hi/lo operand splits change, at the GEMM's 2^-16 level
            assert float((g - ref).abs().max() / ref.abs().max()) < 3e-5, sc
        else:                            # power-of-two scalings are exact all the way through
            assert torch.equal(g, ref), sc


def test_nonfinite_grad_output_reaches_grad_input(dcn):
    """An Inf / NaN in grad_output must surface in grad_input (AMP GradScaler's overflow check), not vanish in the
    fixed-point conversion."""
    from gpu_util import dev
    torch.manual_seed(7)
    B, C, H, W, dg = 1, 64, 24, 32, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    for bad in (float("inf"), float("nan")):
        go = torch.randn(B, 64, H, W, device=dev())
        go[0, 3, 10, 17] = bad
        xi = x.clone().requires_grad_()
        dcn.dcn_v2_conv(xi, off, msk, w, b, 1, 1, 1, dg).backward(go)
        assert not bool(torch.isfinite(xi.grad).all()), bad
        assert bool(torch.isfinite(xi.grad[0, :, 20:, :8]).all())      # far from the bad pixel: untouched


def test_backward_reuses_the_forwards_blocked_input(dcn, monkeypatch):
    """The forward's group-blocked input copy is handed to the backward of the same tensor (EBFI_DCN_INPUT_BLOCKED):
    identical results, and any change of the tensor (version counter) or a different tensor misses the cache."""
    from gpu_util import dev
    from ebfi_be_b200.shims import _ext
    torch.manual_seed(9)
    B, C, H, W, dg = 2, 64, 40, 48, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    go = torch.randn(B, 64, H, W, device=dev())
    geom = (3, 3, 1, 1, 1, 1, 1, 1, dg)
    monkeypatch.setenv("EBFI_DCN_NO_BLOCKED_REUSE", "1")
    _ext._blocked_cache.clear()
    _ext.dcn_v2_forward(x, w, b, off, msk, *geom)
    assert not _ext._blocked_cache
    plain = _ext.dcn_v2_backward(x, w, b, off, msk, go, *geom)
    monkeypatch.delenv("EBFI_DCN_NO_BLOCKED_REUSE")
    _ext.dcn_v2_forward(x, w, b, off, msk, *geom)
    assert _ext._blocked_cache[dev().index][0] == _ext._blocked_key(x, _ext._geom(x, w, *geom)[0])
    reused = _ext.dcn_v2_backward(x, w, b, off, msk, go, *geom)
    for a, c in zip(reused, plain):
        assert torch.equal(a, c)
    x.mul_(2.0)                                  # version bump: the cached copy is stale and must not be used
    want = _ext.dcn_v2_backward(x.clone(), w, b, off, msk, go, *geom)      # a different tensor: cache miss
    got = _ext.dcn_v2_backward(x, w, b, off, msk, go, *geom)
    for a, c in zip(got, want):
        assert torch.equal(a, c)


def test_blocked_copy_only_goes_to_the_box_backward(monkeypatch):
    """The CUDA-core kernels (EBFI_DCN_IMPL=simt, for the forward and backward or only for the backward) and a grad_output
    that is not 16-byte aligned run backwards that read the NCHW input: they get it, not a forward's blocked copy, and
    give the results of the same backward on a tensor no forward has seen (grad_input to the order of its float atomics)."""
    from gpu_util import dev
    from ebfi_be_b200.shims import _ext
    torch.manual_seed(10)
    B, C, H, W, dg = 2, 64, 24, 40, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    go = torch.randn(B, 64, H, W, device=dev())
    go_mis = torch.empty(go.numel() + 1, device=dev())[1:].view(go.shape).copy_(go)
    geom = (3, 3, 1, 1, 1, 1, 1, 1, dg)
    for fwd_env, bwd_env, g in ((None, None, go_mis), ("simt", "simt", go), (None, "simt", go)):
        for name, env in (("fwd", fwd_env), ("bwd", bwd_env)):
            if env:
                monkeypatch.setenv("EBFI_DCN_IMPL", env)
            else:
                monkeypatch.delenv("EBFI_DCN_IMPL", raising=False)
            if name == "fwd":
                _ext.dcn_v2_forward(x, w, b, off, msk, *geom)
        want = _ext.dcn_v2_backward(x.clone(), w, b, off, msk, g, *geom)
        got = _ext.dcn_v2_backward(x, w, b, off, msk, g, *geom)
        assert rel_err(got[0].cpu().numpy(), want[0].cpu().numpy()) < 1e-6, (fwd_env, bwd_env)
        for a, c in zip(got[1:], want[1:]):
            assert torch.equal(a, c), (fwd_env, bwd_env)


def test_reductions_are_bit_reproducible(dcn):
    """grad_offset / grad_mask / grad_weight / grad_bias use fixed-order reductions."""
    from gpu_util import dev
    torch.manual_seed(1)
    B, C, H, W, dg = 2, 64, 48, 48, 8
    x = torch.randn(B, C, H, W, device=dev())
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    w = torch.randn(64, C, 3, 3, device=dev()) / 24
    b = torch.randn(64, device=dev())
    go = torch.randn(B, 64, H, W, device=dev())
    runs = []
    for _ in range(3):
        ts = [v.clone().requires_grad_() for v in (x, off, msk, w, b)]
        dcn.dcn_v2_conv(*ts, 1, 1, 1, dg).backward(go)
        runs.append([v.grad.clone() for v in ts])
    for r in runs[1:]:
        for i in (1, 2, 3, 4):
            assert torch.equal(r[i], runs[0][i]), GRADS[i]
        assert rel_err(r[0].cpu().numpy(), runs[0][0].cpu().numpy()) < 1e-5


def test_matches_reference_cuda_kernels(dcn):
    """The reference's own dcn_v2_im2col_cuda.cu kernels compiled unmodified for sm_100a, through their stored
    results (tests/golden/ref_dcn_b2_40x40.npz, see make_golden_ref.py)."""
    from gpu_util import RefGolden, ref_dcn_inputs
    d = ref_dcn_inputs()
    ref = RefGolden("ref_dcn_b2_40x40", d)
    ts = [d[k].clone().requires_grad_() for k in ("x", "off", "msk", "w", "b")]
    out = dcn.dcn_v2_conv(*ts, 1, 1, 1, 8)
    out.backward(d["go"])
    assert ref.rel_err("out", out) < FWD_TOL
    for name, v in zip(GRADS, ts):
        assert ref.rel_err(name, v.grad) < GRAD_TOL, name


def test_modules_forward_backward(dcn):
    """example_dconv of the reference (testcuda.py:169-180): DCN(64,64,3,pad 1,dg 2) on 2x64x128x128."""
    from gpu_util import dev
    torch.manual_seed(0)
    m = dcn.DCN(64, 64, kernel_size=(3, 3), stride=1, padding=1, deformable_groups=2).to(dev())
    x = torch.randn(2, 64, 128, 128, device=dev())
    out = m(x)
    assert out.shape == x.shape
    out.norm().backward()
    assert m.weight.grad.shape == m.weight.shape and torch.isfinite(m.weight.grad).all()
    # zero-initialised offset conv => plain 3x3 convolution with mask 0.5
    want = 0.5 * torch.nn.functional.conv2d(x.double(), m.weight.double(), None, 1, 1) + m.bias.double().view(1, -1, 1, 1)
    assert rel_err(out.detach().cpu().numpy(), want.detach().cpu().numpy()) < FWD_TOL
    sep = dcn.DCN_sep(64, 64, 3, stride=1, padding=1, deformable_groups=8).to(dev())
    assert sep(x, torch.randn_like(x)).shape == x.shape


def test_full_size_properties(dcn):
    """BASELINE config 1 (B=1, C=64->64, 3x3, dg=8, 256x256). Size-independent properties:
    zero offsets + unit mask == ordinary convolution; the op is linear in input and in weight,
    so <gO, out - bias> == <grad_input, input> == <grad_weight, weight>; grad_bias == sum gO."""
    from gpu_util import dev, dot
    torch.manual_seed(0)
    B, C, H, W, dg = 1, 64, 256, 256, 8
    x = torch.randn(B, C, H, W, device=dev())
    w = (torch.rand(64, C, 3, 3, device=dev()) * 2 - 1) / 24
    b = torch.randn(64, device=dev())
    out0 = dcn.dcn_v2_conv(x, torch.zeros(B, 2 * dg * 9, H, W, device=dev()),
                           torch.ones(B, dg * 9, H, W, device=dev()), w, b, 1, 1, 1, dg)
    want = torch.nn.functional.conv2d(x.double(), w.double(), b.double(), 1, 1)
    assert rel_err(out0.cpu().numpy(), want.cpu().numpy()) < FWD_TOL
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev())
    msk = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev()))
    go = torch.randn(B, 64, H, W, device=dev())
    ts = [v.clone().requires_grad_() for v in (x, off, msk, w, b)]
    out = dcn.dcn_v2_conv(*ts, 1, 1, 1, dg)
    out.backward(go)
    a = dot(go, out.detach() - b.view(1, -1, 1, 1))
    assert abs(a - dot(ts[0].grad, x)) <= 1e-4 * abs(a)
    assert abs(a - dot(ts[3].grad, w)) <= 1e-4 * abs(a)
    assert abs(a - dot(ts[2].grad, msk)) <= 1e-4 * abs(a)          # linear in mask, too
    assert rel_err(ts[4].grad.cpu().numpy(), go.double().sum((0, 2, 3)).cpu().numpy()) < GRAD_TOL


def test_reference_gradcheck_recipe(dcn):
    """check_gradient_dconv of the reference (testcuda.py:69-97): torch.autograd.gradcheck on dcn_v2_conv in
    fp32 with eps=1e-3, atol=1e-4, rtol=1e-2, N=2, C=2, 4x4, dg=1, input rand*0.01, offset ~ randn*2,
    mask sigmoid(rand). Bilinear sampling is only piecewise differentiable, so (unlike the reference's
    script, which just prints the verdict) the fractional parts of the offsets are kept in [0.2, 0.8]:
    no sample sits within eps of a pixel boundary. grad_input uses fp32 reductions whose order is not
    fixed -> nondet_tol."""
    from gpu_util import dev
    torch.manual_seed(0)
    N, inC, outC, inH, inW, kH, kW, dg = 2, 2, 2, 4, 4, 3, 3, 1
    input = (torch.rand(N, inC, inH, inW, device=dev()) * 0.01).requires_grad_()
    offset = torch.randn(N, dg * 2 * kW * kH, inH, inW, device=dev()) * 2
    offset = (offset.floor() + 0.2 + 0.6 * torch.rand_like(offset)).requires_grad_()
    mask = torch.sigmoid(torch.rand(N, dg * kW * kH, inH, inW, device=dev())).detach().requires_grad_()
    weight = torch.randn(outC, inC, kH, kW, device=dev()).requires_grad_()
    bias = torch.rand(outC, device=dev()).requires_grad_()
    assert torch.autograd.gradcheck(dcn.dcn_v2_conv, (input, offset, mask, weight, bias, 1, 1, 1, dg),
                                    eps=1e-3, atol=1e-4, rtol=1e-2, nondet_tol=1e-5)


def test_bf16_tensors_stated_tolerance(dcn, oracle):
    """bf16 at the boundary (new capability): fp32 arithmetic on the exactly converted values, one rounding
    to bf16 per result -> |err| <= 2^-8 * max|ref| per tensor against the oracle run on the same bf16 inputs."""
    from gpu_util import dev
    torch.manual_seed(3)
    B, C, Co, H, W, dg = 1, 64, 64, 20, 24, 8
    mk = lambda *s: torch.randn(*s).bfloat16()
    x, off, msk = mk(B, C, H, W), (2 * torch.randn(B, 2 * dg * 9, H, W)).bfloat16(), torch.sigmoid(torch.randn(B, dg * 9, H, W)).bfloat16()
    w, b, go = (torch.randn(Co, C, 3, 3) / 24).bfloat16(), mk(Co), mk(B, Co, H, W)
    ts = [t.to(dev()).requires_grad_() for t in (x, off, msk, w, b)]
    out = dcn.dcn_v2_conv(*ts, 1, 1, 1, dg)
    assert out.dtype == torch.bfloat16
    out.backward(go.to(dev()))
    f = lambda t: t.float().numpy()
    tol = 2.0 ** -8
    assert rel_err(out.detach().float().cpu().numpy(), oracle.dcn_forward(f(x), f(off), f(msk), f(w), f(b), 1, 1, 1, dg)) < tol
    want = oracle.dcn_backward(f(x), f(off), f(msk), f(w), f(b), f(go), 1, 1, 1, dg)
    for name, t, r in zip(GRADS, ts, want):
        assert rel_err(t.grad.float().cpu().numpy(), r) < tol, name


# ---- packed entry points: raw conv_offset_mask output in, chunk/cat/sigmoid folded into the kernels ----
def _packed_case(rng, shape):
    B, C, Co, H, W, k, s, p, d, dg, osc = shape
    Ho = (H + 2 * p - (d * (k - 1) + 1)) // s + 1
    Wo = (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    n_t = dg * k * k
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = (rng.random((Co, C, k, k), dtype=np.float32) * 2 - 1) / np.sqrt(C * k * k)
    b = rng.standard_normal(Co, dtype=np.float32)
    om = rng.standard_normal((B, 3 * n_t, Ho, Wo)).astype(np.float32)
    om[:, :2 * n_t] *= osc
    om[:, 2 * n_t:] *= 2.0                         # logits in about (-6, 6)
    go = rng.standard_normal((B, Co, Ho, Wo), dtype=np.float32)
    return x, w, b, om, go, n_t


def _packed_expected(oracle, x, w, b, om, go, n_t, s, p, d, dg):
    """The reference's op sequence (dcn_v2.py:217-227) in float64 around the CPU oracle."""
    off = np.ascontiguousarray(om[:, :2 * n_t])
    m = 1.0 / (1.0 + np.exp(-om[:, 2 * n_t:].astype(np.float64)))
    msk = m.astype(np.float32)
    out = oracle.dcn_forward(x, off, msk, w, b, s, p, d, dg)
    g_in, g_off, g_msk, g_w, g_b = oracle.dcn_backward(x, off, msk, w, b, go, s, p, d, dg)
    g_om = np.concatenate([g_off, g_msk * m * (1.0 - m)], axis=1)
    return out, [g_in, g_om, g_w, g_b], off


@pytest.mark.parametrize("shape", [SHAPES[0], SHAPES[1], SHAPES[3], SHAPES[7]])
def test_packed_offset_mask_against_oracle(dcn, oracle, shape):
    from gpu_util import dev, n, t
    rng = np.random.default_rng(7 + len(str(shape)))
    s, p, d, dg = shape[6], shape[7], shape[8], shape[9]
    x, w, b, om, go, n_t = _packed_case(rng, shape)
    want_out, want_grads, off = _packed_expected(oracle, x, w, b, om, go, n_t, s, p, d, dg)
    ts = [t(a).requires_grad_() for a in (x, om, w, b)]
    stat = torch.full((1,), -1.0, device=dev())
    out = dcn.dcn_v2_conv_packed(*ts, s, p, d, dg, stat)
    out.backward(t(go))
    assert rel_err(n(out), want_out) < FWD_TOL
    for name, v, ref in zip(["grad_input", "grad_offset_mask", "grad_weight", "grad_bias"], ts, want_grads):
        assert rel_err(n(v.grad), ref) < GRAD_TOL, name
    # the statistic behind the `offset_mean > 100` warning (dcn_v2.py:221-223)
    assert abs(float(stat) / off.size - np.abs(off.astype(np.float64)).mean()) < 1e-4 * np.abs(off).mean()


def test_packed_equals_unpacked_sequence(dcn):
    """Same kernels, two addressings: packed == chunk -> cat -> sigmoid -> dcn_v2_conv through autograd, to
    rounding of the sigmoid (torch's vs the in-kernel one)."""
    from gpu_util import dev
    torch.manual_seed(3)
    B, C, H, W, dg = 2, 64, 40, 56, 8
    x = torch.randn(B, C, H, W, device=dev(), requires_grad=True)
    om = (torch.randn(B, 3 * dg * 9, H, W, device=dev()) * 2).requires_grad_()
    w = (torch.randn(C, C, 3, 3, device=dev()) / 24).requires_grad_()
    b = torch.randn(C, device=dev(), requires_grad=True)
    go = torch.randn(B, C, H, W, device=dev())
    o1, o2, mask = torch.chunk(om, 3, dim=1)
    ref = dcn.dcn_v2_conv(x, torch.cat((o1, o2), 1), torch.sigmoid(mask), w, b, 1, 1, 1, dg)
    ref.backward(go)
    want = [v.grad.clone() for v in (x, om, w, b)]
    for v in (x, om, w, b):
        v.grad = None
    got = dcn.dcn_v2_conv_packed(x, om, w, b, 1, 1, 1, dg)
    got.backward(go)
    assert rel_err(got.detach().cpu().numpy(), ref.detach().cpu().numpy()) < FWD_TOL
    for name, v, r in zip(["grad_input", "grad_offset_mask", "grad_weight", "grad_bias"], (x, om, w, b), want):
        assert rel_err(v.grad.cpu().numpy(), r.cpu().numpy()) < GRAD_TOL, name


def test_fused_modules_match_reference_sequence(dcn, caplog):
    """DCN / DCN_sep with fused=True (packed kernels, deferred warning) vs fused=False (the reference's op
    sequence with its host sync), same parameters."""
    import logging
    from gpu_util import dev
    torch.manual_seed(5)
    x = torch.randn(1, 64, 48, 64, device=dev())
    fea = torch.randn_like(x)
    for cls, args in ((dcn.DCN, (x,)), (dcn.DCN_sep, (x, fea))):
        m = cls(64, 64, 3, stride=1, padding=1, deformable_groups=8).to(dev())
        with torch.no_grad():
            m.conv_offset_mask.weight.normal_(0, 0.05)
            m.conv_offset_mask.bias.normal_(0, 0.5)
        outs, grads = [], []
        for fused in (True, False):
            m.fused = fused
            m.zero_grad()
            out = m(*args)
            out.square().sum().backward()
            outs.append(out.detach().cpu().numpy())
            grads.append({k: v.grad.cpu().numpy().copy() for k, v in m.named_parameters()})
        assert rel_err(outs[0], outs[1]) < FWD_TOL
        for k in grads[0]:
            assert rel_err(grads[0][k], grads[1][k]) < GRAD_TOL, k
    # the warning: offsets with mean |.| > 100 are reported (late, at the latest on flush)
    sep = dcn.DCN_sep(64, 64, 3, stride=1, padding=1, deformable_groups=8).to(dev())
    with torch.no_grad():
        sep.conv_offset_mask.bias[:144] = 500.0
    with caplog.at_level(logging.WARNING, logger="base"):
        sep(x, fea)
        sep.flush_offset_warnings()
    assert any("larger than 100" in r.getMessage() for r in caplog.records)
    caplog.clear()
    with torch.no_grad():
        sep.conv_offset_mask.bias.zero_()
    with caplog.at_level(logging.WARNING, logger="base"):
        sep(x, fea)
        sep.flush_offset_warnings()
    assert not caplog.records


def test_packed_rejects_wrong_channel_count(dcn):
    from gpu_util import dev
    x = torch.randn(1, 16, 8, 8, device=dev())
    w = torch.randn(16, 16, 3, 3, device=dev())
    with pytest.raises(RuntimeError, match="offset_mask shape"):
        dcn.dcn_v2_conv_packed(x, torch.randn(1, 2 * 2 * 9, 8, 8, device=dev()), w, torch.zeros(16, device=dev()), 1, 1, 1, 2)


# ---- deterministic mode: the determinism gate of SURVEY 8(d) for ALL five gradients ----
@pytest.mark.parametrize("shape", [(2, 64, 64, 48, 48, 8), (2, 16, 24, 19, 23, 4)])   # tensor-core / CUDA-core path
@pytest.mark.parametrize("scale", [1.0, 3.0e4, 2.0e-6])
def test_deterministic_mode_bit_identical_and_in_tolerance(dcn, oracle, shape, scale, monkeypatch):
    """EBFI_DCN_DETERMINISTIC: grad_input accumulated in int64 fixed point -> every gradient bit-identical run to
    run (the reference's float atomicAdd col2im, im2col_cuda.cu:249, is not), still inside the 1e-4 gate, for
    large and tiny gradient magnitudes (the fixed-point scale adapts on the device)."""
    from gpu_util import dev, n, t
    monkeypatch.setenv("EBFI_DCN_DETERMINISTIC", "1")
    B, C, Co, H, W, dg = shape
    rng = np.random.default_rng(5)
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    off = (2 * rng.standard_normal((B, 2 * dg * 9, H, W))).astype(np.float32)
    msk = (1 / (1 + np.exp(-rng.standard_normal((B, dg * 9, H, W))))).astype(np.float32)
    w = ((rng.random((Co, C, 3, 3), dtype=np.float32) * 2 - 1) / np.sqrt(C * 9)).astype(np.float32)
    b = rng.standard_normal(Co, dtype=np.float32)
    go = (scale * rng.standard_normal((B, Co, H, W))).astype(np.float32)
    runs = []
    for _ in range(3):
        ts = [t(a).requires_grad_() for a in (x, off, msk, w, b)]
        dcn.dcn_v2_conv(*ts, 1, 1, 1, dg).backward(t(go))
        runs.append([v.grad.clone() for v in ts])
    for r in runs[1:]:
        for i in range(5):
            assert torch.equal(r[i], runs[0][i]), GRADS[i]
    want = oracle.dcn_backward(x, off, msk, w, b, go, 1, 1, 1, dg)
    for name, got, ref in zip(GRADS, runs[0], want):
        assert rel_err(n(got), ref) < GRAD_TOL, name


def test_deterministic_follows_torch_switch(dcn):
    from gpu_util import dev
    torch.manual_seed(9)
    x = torch.randn(1, 64, 32, 32, device=dev())
    off = 2 * torch.randn(1, 144, 32, 32, device=dev())
    msk = torch.rand(1, 72, 32, 32, device=dev())
    w = torch.randn(64, 64, 3, 3, device=dev()) / 24
    go = torch.randn(1, 64, 32, 32, device=dev())
    torch.use_deterministic_algorithms(True)
    try:
        outs = []
        for _ in range(2):
            xi = x.clone().requires_grad_()
            dcn.dcn_v2_conv(xi, off, msk, w, torch.zeros(64, device=dev()), 1, 1, 1, 8).backward(go)
            outs.append(xi.grad.clone())
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(outs[0], outs[1])


def test_backward_with_misaligned_offset_views(dcn, oracle):
    """offset / mask tensors whose storage starts 4 bytes off a 16-byte boundary (contiguous views of a larger buffer):
    the TMA staging of the backward cannot be used; the kernel must fall back to direct loads, not fail."""
    from gpu_util import dev, n, t
    rng = np.random.default_rng(17)
    B, C, H, W, dg = 1, 64, 16, 16, 8
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = ((rng.random((64, C, 3, 3), dtype=np.float32) * 2 - 1) / 24).astype(np.float32)
    b = rng.standard_normal(64, dtype=np.float32)
    off = (2 * rng.standard_normal((B, 2 * dg * 9, H, W))).astype(np.float32)
    msk = rng.random((B, dg * 9, H, W), dtype=np.float32)
    go = rng.standard_normal((B, 64, H, W), dtype=np.float32)

    def shifted(a):
        buf = torch.empty(a.size + 1, device=dev())
        v = buf[1:].view(a.shape)
        v.copy_(t(a))
        assert v.is_contiguous() and v.data_ptr() % 16 == 4
        return v

    from ebfi_be_b200.shims import _ext
    want = oracle.dcn_backward(x, off, msk, w, b, go, 1, 1, 1, dg)
    grads = _ext.dcn_v2_backward(t(x), t(w), t(b), shifted(off), shifted(msk), t(go), 3, 3, 1, 1, 1, 1, 1, 1, dg)
    for name, got, ref in zip(GRADS, grads, want):
        assert rel_err(n(got), ref) < GRAD_TOL, name
    # every tensor shifted, grad_output included (its 128-bit staging loads are not usable either)
    grads = _ext.dcn_v2_backward(shifted(x), shifted(w), shifted(b), shifted(off), shifted(msk), shifted(go),
                                 3, 3, 1, 1, 1, 1, 1, 1, dg)
    for name, got, ref in zip(GRADS, grads, want):
        assert rel_err(n(got), ref) < GRAD_TOL, name
    out = _ext.dcn_v2_forward(shifted(x), shifted(w), shifted(b), shifted(off), shifted(msk), 3, 3, 1, 1, 1, 1, 1, 1, dg)
    assert rel_err(n(out), oracle.dcn_forward(x, off, msk, w, b, 1, 1, 1, dg)) < FWD_TOL
