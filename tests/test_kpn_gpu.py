"""KernelConv producer -> FAC fused forward (csrc/kpn.cu) vs the float64 restatement of the reference's op sequence
(models/Ours/model_singleframe.py:145-146,159-162). Tolerances: 1e-5 of max|out| against the sequence with
bf16-rounded conv operands (isolates indexing from precision), 1e-2 against the unrounded fp64 sequence."""
import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mod():
    from ebfi_be_b200 import modification
    return modification


def _case(rng, B, Ce, Cf, H, W, K):
    ev = rng.standard_normal((B, Ce, H, W), dtype=np.float32)
    fr = rng.standard_normal((B, Cf, H, W), dtype=np.float32)
    w = (rng.standard_normal((Ce * K * K, Ce + Cf, 3, 3)) * 0.1 / np.sqrt(9 * (Ce + Cf))).astype(np.float32) * 10
    b = (0.1 * rng.standard_normal(Ce * K * K)).astype(np.float32)
    return ev, fr, w, b


# (B, Ce, Cf, H, W, K)
SHAPES = [(1, 64, 64, 16, 8, 5),      # exactly one tile
          (2, 64, 64, 19, 13, 5),     # ragged tiles, two samples
          (1, 64, 64, 40, 24, 3),     # K = 3
          (1, 32, 32, 33, 17, 5),     # 64 input channels, 11 slices (last one 2 channels)
          (1, 16, 16, 20, 20, 5),     # 32 input channels; last slice has a single channel
          (1, 64, 0, 18, 10, 1)]      # no frame features, 1x1 FAC

# Shapes at which a CTA of the persistent kernel walks several items: its accumulator and halo-part barrier phases
# wrap, parts are refilled while others compute, its range crosses weight slices and samples. Comments give Cin / 32
# halo parts, channels in the last weight slice and items per CTA at 148 SMs (kpn_work_split; the coverage is
# asserted at the device's SM count in test_kpn_pipeline_gpu.py).
PIPELINE_SHAPES = [(2, 48, 48, 21, 33, 5),    # 3 parts, last slice full, 3 items per CTA, crosses slice and sample
                   (3, 96, 0, 33, 20, 3),     # 3 parts, K = 3, 6 items, no frame features
                   (2, 32, 64, 29, 43, 1),    # 3 parts, K = 1
                   (2, 64, 32, 64, 64, 5),    # 3 parts, 10 items
                   (2, 33, 31, 40, 40, 5),    # odd Ce: an 8-channel input chunk mixes event and frame channels
                   (1, 128, 0, 17, 9, 5),     # 4 parts, no frame features, H % 16 = 1
                   (2, 64, 64, 17, 25, 1),    # 4 parts, K = 1, W % 8 = 1
                   (2, 64, 64, 17, 29, 5),    # 4 parts, 3 items, crosses slice and sample
                   (2, 16, 16, 49, 49, 5),    # 1 part, 3 items
                   (2, 32, 32, 80, 56, 3),    # 2 parts, 6 items
                   (3, 32, 32, 3, 70, 5),     # H < K: a window reaches past both image borders
                   (4, 16, 16, 7, 5, 3),      # W < 8, H < 16: a single partial tile per sample
                   (2, 32, 0, 1, 1, 5),       # H = W = 1: the whole replication pad folds onto one pixel
                   (5, 64, 64, 2, 2, 5),      # 4 parts, 2 x 2 images
                   (2, 96, 32, 36, 50, 3)]    # 4 parts, last slice full, 10 items


def kpn_work_split(shape, sms, backward=False):
    """The work split of csrc/kpn.cu (`fill` and the launch arithmetic of kpn_forward / kpn_backward) for
    shape = (B, Ce, Cf, H, W, K) on `sms` SMs. Items are (weight slice of 3 FAC channels, 16 x 8 pixel tile) in
    slice-major order, tiles in (sample, tile row, tile column) order; CTA k walks items [k * per, (k + 1) * per).
    Returns npart (halo parts = Cin / 32), last (FAC channels in the last slice), tiles_x, tiles_y, ntile (tiles per
    slice), nslice, per, ctas, crosses_slice / crosses_sample (some CTA's range holds items of two slices / two
    samples)."""
    B, Ce, Cf, H, W, K = shape
    nslice = -(-Ce // 3)
    tiles_x, tiles_y = -(-W // 8), -(-H // 16)
    tiles_per_sample = tiles_x * tiles_y
    ntile = B * tiles_per_sample
    total = nslice * ntile
    grid = min(total, sms, 1024) if backward else min(total, sms)      # 1024: BWD_MAX_GRID
    per = -(-total // grid)
    ctas = -(-total // per)
    first = np.arange(ctas) * per
    last = np.minimum(first + per, total) - 1
    return dict(npart=(Ce + Cf) // 32, last=Ce - 3 * (nslice - 1), tiles_x=tiles_x, tiles_y=tiles_y, ntile=ntile,
                nslice=nslice, per=per, ctas=ctas,
                crosses_slice=bool((first // ntile != last // ntile).any()),
                crosses_sample=B > 1 and bool((first // tiles_per_sample != last // tiles_per_sample).any()))


@pytest.mark.parametrize("shape", SHAPES + PIPELINE_SHAPES)
def test_fused_against_oracle(mod, oracle, shape):
    from gpu_util import n, t
    B, Ce, Cf, H, W, K = shape
    ev, fr, w, b = _case(np.random.default_rng(sum(shape)), *shape)
    with torch.no_grad():
        got = n(mod.kernelconv_fac_fused(t(ev), t(fr), t(w), t(b), K, 0.01))
    want_bf16, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, 0.01, bf16_operands=True)
    want, _ = oracle.kpn_fused_forward(ev, fr, w, b, K, 0.01)
    assert rel_err(got, want_bf16) < 1e-5
    assert rel_err(got, want) < 1e-2


def test_module_matches_unfused_sequence_and_falls_back_under_autograd(mod):
    from gpu_util import dev
    torch.manual_seed(0)
    m = mod.KernelPrediction(64, 5).to(dev())
    ev, fr = torch.randn(2, 64, 48, 40, device=dev()), torch.randn(2, 64, 48, 40, device=dev())
    with torch.no_grad():
        fused = m(ev, fr)
        ref = m.KPN(ev, m.KernelConv(torch.cat([ev, fr], 1)))
    assert rel_err(fused.cpu().numpy(), ref.cpu().numpy()) < 1e-2
    out = m(ev, fr)                                   # parameters require grad -> reference op sequence
    out.mean().backward()
    assert m.KernelConv.conv2d.weight.grad is not None and rel_err(out.detach().cpu().numpy(), ref.cpu().numpy()) < 1e-3
    with pytest.raises(RuntimeError, match="forward-only"):
        mod.kernelconv_fac_fused(ev, fr, m.KernelConv.conv2d.weight, m.KernelConv.conv2d.bias, 5)


def test_full_size_one_hot_kernels_shift_the_input(mod):
    """BASELINE cfg2 size (B=4, C=64, K=5, 256x256). Zero conv weights and a bias that is one-hot per channel make
    the predicted kernel a constant one-hot tap (LeakyReLU(1) = 1, LeakyReLU(0) = 0), so the output is the
    replication-padded input shifted by that tap — exact, at full size."""
    from gpu_util import dev
    torch.manual_seed(1)
    B, C, K, H, W = 4, 64, 5, 256, 256
    ev, fr = torch.randn(B, C, H, W, device=dev()), torch.randn(B, C, H, W, device=dev())
    w = torch.zeros(C * K * K, 2 * C, 3, 3, device=dev())
    bias = torch.zeros(C, K * K, device=dev())
    taps = torch.arange(C, device=dev()) % (K * K)
    bias[torch.arange(C, device=dev()), taps] = 1.0
    with torch.no_grad():
        out = mod.kernelconv_fac_fused(ev, fr, w, bias.reshape(-1), K)
    evp = torch.nn.functional.pad(ev, (2, 2, 2, 2), mode="replicate")
    for c in (0, 7, 24, 63):
        ky, kx = int(taps[c]) // K, int(taps[c]) % K
        assert torch.equal(out[:, c], evp[:, c, ky:ky + H, kx:kx + W]), c


def test_unsupported_channel_count_raises(mod):
    from gpu_util import dev
    ev = torch.randn(1, 24, 8, 8, device=dev())
    with pytest.raises(RuntimeError, match="multiple of 32"):
        mod.kernelconv_fac_fused(ev, ev, torch.randn(24 * 25, 48, 3, 3, device=dev()), torch.zeros(600, device=dev()), 5)


def test_bf16_tensors_stated_tolerance(mod, oracle):
    """bfloat16 tensors (BASELINE config 4 runs the model in bf16; the reference is fp32-only): the conv operands are the
    bf16 values themselves, accumulation and FAC are fp32, the output is rounded once to bf16. Stated tolerance
    (SURVEY 8d): max-abs error <= 2^-7 of max|out| against the float64 op sequence on the same bf16-valued inputs."""
    from gpu_util import n, t
    rng = np.random.default_rng(3)
    B, Ce, Cf, H, W, K = 1, 64, 64, 24, 16, 5
    ev, fr, w, b = _case(rng, B, Ce, Cf, H, W, K)
    tb = [t(a).bfloat16() for a in (ev, fr, w, b)]
    with torch.no_grad():
        got = mod.kernelconv_fac_fused(*tb, K, 0.01)
    assert got.dtype == torch.bfloat16
    ev_r, fr_r, w_r, b_r = (n(x.float()) for x in tb)
    want, _ = oracle.kpn_fused_forward(ev_r, fr_r, w_r, b_r, K, 0.01)
    assert rel_err(n(got.float()), want) < 2.0 ** -7
    with pytest.raises(RuntimeError, match="all tensors must be"):
        mod.kernelconv_fac_fused(tb[0], tb[1].float(), tb[2], tb[3], K)
