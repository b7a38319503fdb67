"""The DCNv2 tensor-core kernels (csrc/dcn_fwd_box.cu, csrc/dcn_bwd_box.cu) at sizes where each persistent CTA walks
several tiles, compared EXACTLY with float64: second and later waves, ragged last waves, walks that cross a sample,
partial right / bottom tiles, 1, 3 and 4 taps per thread row, 1, 2 and 4 units per deformable group and 1-4 CTA rows
of the backward (PIPELINE_SHAPES, chosen with dcn_work_split). The inputs lie on the dyadic lattice of _lattice_case,
on which DCNv2's fp32 arithmetic does not round, so a wrong tile stride, a stale box or offset plane, a skipped seam in
dcn_gin_collect or a partial slot summed twice fails the comparison, however few elements it touches.
The second half measures the two long fp32 accumulation chains against float64 on random data, at the stated gates:
the forward's hi*hi chain where Cout > 64 leaves fewer than three accumulators, and the backward's grad_weight chain
over a whole CTA walk at the training size."""
import numpy as np
import pytest
import torch

from conftest import FWD_TOL, GRAD_TOL, rel_err

BF16, F16 = torch.bfloat16, torch.float16
GRADS = ("grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias")


@pytest.fixture(scope="module")
def dcn():
    from ebfi_be_b200 import dcn_v2
    return dcn_v2


@pytest.fixture(scope="module")
def ext():
    from ebfi_be_b200.shims import _ext
    return _ext


def _pair(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def _ceil(a, b):
    return -(-a // b)


def _geom(shape):
    """(B, C, Co, H, W, dg, k, stride, pad, dil) -> (the nine geometry ints of _ext, Ho, Wo)."""
    B, C, Co, H, W, dg, k, s, p, dl = shape
    (kh, kw), (sh, sw), (ph, pw), (dh, dw) = (_pair(v) for v in (k, s, p, dl))
    Ho = (H + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    Wo = (W + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    return (kh, kw, sh, sw, ph, pw, dh, dw, dg), Ho, Wo


# ---------------------------------------------------------------- the work split, restated
def dcn_work_split(shape, sms):
    """The launch arithmetic of the two tensor-core kernels for `shape` on `sms` SMs.

    Forward (dcn_fwd_box.cu make_plan / forward_tc): 8 x 16-pixel tiles, grid = min(sms, B * ntiles), CTA i walks the
    tiles i, i + grid, ...; TPR taps per thread row, nacc hi*hi accumulators, offsets / masks by TMA when an fp32 row
    is a whole number of 16-byte words; `fwd_tc` = make_plan accepts the fp32 call (its shared memory fits), else the
    CUDA-core kernel runs.
    Backward (dcn_bwd_box.cu make_plan / box_splits): units = C / 8 eight-channel units, ncs of them per deformable
    group, GPC per CTA, NH CTA rows; CTA (s, h) walks the tiles s, s + grid_x, ... for units [h * GPC, h * GPC + GPC);
    `box` = make_plan accepts the fp32 call.
    For both: the largest number of tiles a CTA walks, whether the last wave is ragged and whether some CTA's walk
    crosses from one sample into the next."""
    B, C, Co, H, W, dg = shape[:6]
    (kh, kw, sh, sw, ph, pw, dh, dw, _), Ho, Wo = _geom(shape)
    KK = kh * kw
    tiles_x, tiles_y = _ceil(Wo, 16), _ceil(Ho, 8)
    ntiles = tiles_x * tiles_y
    total = B * ntiles

    def walk(grid):
        return dict(per=_ceil(total, grid), ragged=total % grid != 0,
                    crosses_sample=any(c // ntiles != (c + (_ceil(total - c, grid) - 1) * grid) // ntiles
                                       for c in range(min(grid, total))))

    TPR, nacc = _ceil(KK, 3), min(3, 256 // Co - 1)
    unit_bytes = TPR * 2 * Co * 24 * 4
    fwd_smem = 3 * 2 * 128 * 24 * 4 + 2 * unit_bytes + 2 * 24 * 30 * 32 + 2 * 3 * KK * 128 * 4
    fwd_tc = Co % 16 == 0 and Co <= 128 and (C // dg) % 8 == 0 and nacc >= 1 and TPR <= 4 and fwd_smem <= 225 * 1024
    grid = min(sms, total)
    fwd = dict(grid=grid, TPR=TPR, nacc=nacc, om_tma=Wo % 4 == 0, fwd_tc=fwd_tc, **walk(grid))

    units, ncs = C // 8, C // dg // 8
    Kc = 8 * KK
    N1, N3 = _ceil(Kc, 16) * 16, _ceil(Kc + 1, 16) * 16
    GPC = max(1, min(4, units, (512 - 2 * N1) // N3))
    NH = _ceil(units, GPC)
    grid_x = max(1, min(total, sms // NH))
    bwd_smem = 2 * 2 * N1 * 64 * 2 + 2 * 64 * 128 * 2 + 2 * N3 * 128 * 2 + 3 * 24 * 30 * 32 + 2 * 2944 + 2 * 3 * KK * 128 * 4
    fh, fw = 7 * sh + (kh - 1) * dh + 1, 15 * sw + (kw - 1) * dw + 1
    box = ((C // dg) % 8 == 0 and Co == 64 and ncs & (ncs - 1) == 0 and KK <= 15 and (512 - 2 * N1) // N3 >= 1
           and N3 <= 256 and GPC % ncs == 0 and fh <= 23 and fw <= 29 and bwd_smem <= 226 * 1024)
    bwd = dict(units=units, ncs=ncs, TPR=TPR, GPC=GPC, NH=NH, grid_x=grid_x, box=box, **walk(grid_x))
    return dict(Ho=Ho, Wo=Wo, tiles_x=tiles_x, tiles_y=tiles_y, ntiles=ntiles, KK=KK, fwd=fwd, bwd=bwd)


# (B, C, Co, H, W, dg, kernel, stride, pad, dilation); at 148 SMs (see SPLIT_AT_148):
PIPELINE_SHAPES = [
    (1, 64, 64, 256, 256, 8, 3, 1, 1, 1),           # cfg1: 4 forward / 7 backward tiles per CTA
    (2, 64, 64, 200, 152, 8, 3, 1, 1, 1),           # two samples: walks cross from one into the other
    (4, 32, 64, 200, 152, 1, 3, 1, 1, 1),           # 32 channels per group (ncs 4), one CTA row: 7 tiles per CTA
    (2, 96, 64, 128, 96, 3, 3, 1, 1, 1),            # three CTA rows of four units
    (2, 64, 64, 160, 160, 4, 3, 1, 2, 2),           # dilation 2, 16 channels per group
    (1, 128, 64, 96, 120, 4, 3, 1, 1, 1),           # four CTA rows of four units
    (3, 64, 64, 64, 72, 8, 1, 1, 0, 1),             # 1x1 kernel (TPR 1), no padding
    (2, 64, 64, 130, 99, 8, 3, (2, 1), 1, 1),       # stride (2, 1); Wo = 99: offsets / masks read without TMA
    # TPR 4 (10-12 taps) and Cout = 64 do not fit one CTA's shared memory in the fp32 forward, so the two kernels get
    # a shape each: 2x5 for the box backward (forward on CUDA cores), 3x4 at Cout = 48 for the forward (backward on
    # CUDA cores). Ho = 89 / 90, Wo = 110 / 109: partial bottom and right tiles; pad_h != pad_w (the collect's x uses
    # pad_h, as the reference's col2im does).
    (2, 64, 64, 90, 110, 8, (2, 5), 1, (0, 2), 1),
    (2, 64, 48, 90, 110, 4, (3, 4), 1, 1, 1),
]

# per shape: (forward tiles per CTA, ragged, crosses a sample), (backward NH, tiles per CTA, ragged, crosses a sample);
# None where the other kernel runs
SPLIT_AT_148 = [((4, True, False), (2, 7, True, False)), ((4, True, True), (2, 7, True, True)),
                ((7, True, True), (1, 7, True, True)), ((2, True, True), (3, 4, True, True)),
                ((3, True, True), (2, 6, True, True)), ((1, False, False), (4, 3, True, False)),
                ((1, False, False), (2, 2, True, True)), ((1, False, False), (2, 2, True, True)),
                (None, (3, 4, True, True)), ((2, True, True), None)]


def _check_coverage(sms):
    splits = [dcn_work_split(s, sms) for s in PIPELINE_SHAPES]
    fwd = [x["fwd"] for x in splits if x["fwd"]["fwd_tc"]]
    bwd = [x["bwd"] for x in splits if x["bwd"]["box"]]
    for walks in (fwd, bwd):
        assert any(w["per"] >= 3 for w in walks) and any(w["per"] >= 6 for w in walks)
        assert any(w["ragged"] for w in walks)
        assert any(w["crosses_sample"] and w["per"] >= 3 for w in walks)
        assert {w["TPR"] for w in walks} == {1, 3, 4}
    assert len(fwd) == len(bwd) == len(splits) - 1
    assert any(x["Wo"] % 16 for x in splits) and any(x["Ho"] % 8 for x in splits)          # partial right / bottom tiles
    assert {w["ncs"] for w in bwd} == {1, 2, 4}
    assert {w["NH"] for w in bwd} == {1, 2, 3, 4}
    assert {w["om_tma"] for w in fwd} == {True, False}                                   # Wo % 4 zero and non-zero
    assert any(_pair(s[7]) == (2, 1) for s in PIPELINE_SHAPES)
    assert any(s[9] == 2 for s in PIPELINE_SHAPES) and any(s[8] == 0 for s in PIPELINE_SHAPES)


def _library_plans(shape):
    """(the library runs this fp32 shape on the tensor-core forward, on it AND the box backward)."""
    from ebfi_be_b200 import _lib as L
    B, C, Co, H, W = shape[:5]
    ints, _, _ = _geom(shape)
    g = L.DcnGeom(B, C, H, W, Co, *ints, 0)
    return L.load().ebfi_dcnv2_forward_workspace_bytes(g) > 256, L.load().ebfi_dcnv2_blocked_input_offset(g) != 0


def test_pipeline_shapes_cover_the_work_split_at_148_sms():
    for shape, (f, b) in zip(PIPELINE_SHAPES, SPLIT_AT_148, strict=True):
        x = dcn_work_split(shape, 148)
        assert (f is not None) == x["fwd"]["fwd_tc"] and (b is not None) == x["bwd"]["box"], shape
        assert f is None or (x["fwd"]["per"], x["fwd"]["ragged"], x["fwd"]["crosses_sample"]) == f, shape
        assert b is None or (x["bwd"]["NH"], x["bwd"]["per"], x["bwd"]["ragged"], x["bwd"]["crosses_sample"]) == b, shape
        assert shape[0] * x["Ho"] * x["Wo"] <= 2 ** 18, shape           # grad_weight stays exact (_lattice_case)
        # the restated plans agree with the library's
        assert _library_plans(shape) == (f is not None, f is not None and b is not None), shape
    train = dcn_work_split((8, 64, 64, 256, 256, 8, 3, 1, 1, 1), 148)
    assert (train["fwd"]["per"], train["bwd"]["per"]) == (28, 56)
    _check_coverage(148)


@pytest.mark.gpu
def test_pipeline_shapes_cover_the_work_split_on_this_device():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for shape in PIPELINE_SHAPES:
        print(sms, "SMs", shape, dcn_work_split(shape, sms))
    _check_coverage(sms)


# ---------------------------------------------------------------- the lattice
def _lattice_case(rng, shape, far=1 / 8):
    """(x, offset, mask, weight, bias, grad_output) float32 on which every DCNv2 result is exact in fp32: input integers
    in [-2, 2], weight and grad_output in {-1, 0, 1}, bias an integer + 1/2, mask in {0, 1/2, 1}, offsets k/2 + 1/4 with
    |offset| <= 1.75, except a share `far` that reach +-12.25: those samples leave the 24 x 30 box (the global gather
    and red.global.add fall-back) and the image.

    - Every sampling coordinate has fractional part 1/4 or 3/4: no sample lies on a pixel boundary or on -1 / H, so
      fp32 and float64 take the same branches.
    - Corner weights are multiples of 1/16, so a column entry mask * v is a multiple of 1/32 with |.| <= 2: exact in
      the TF32 hi part (lo = 0) and in bf16 hi (lo = 0).
    - out is below 2^18 units of 1/32 for C * KK <= 2304, so the tensor core's round-toward-zero accumulate never
      rounds; + bias is exact.
    - colgrad (grad_output . weight) is an integer with |.| <= 64.
    - grad_input contributions colgrad * mask * corner weight are multiples of 1/32; they convert exactly at the box's
      power-of-two fixed-point scale (>= 2^13 for n <= 2^11 contributions per cell and M <= 64), and a pixel's total
      stays far below 2^24 units, so the boxes, their collect and the far-sample float red.add are exact in any order.
    - grad_offset (multiples of 1/8), grad_mask (1/16) and grad_bias (integers) stay far below 2^24 units.
    - grad_weight (multiples of 1/32, |.| <= 2 per pixel) is exact while B * Ho * Wo <= 2^18; beyond that it can only
      be compared at GRAD_TOL.
    Every value is also exact in bf16 and fp16, so the 16-bit entries see the same inputs."""
    B, C, Co, H, W, dg = shape[:6]
    (kh, kw, *_), Ho, Wo = _geom(shape)
    KK = kh * kw

    def ints(lo, hi, size):
        return rng.integers(lo, hi + 1, size).astype(np.float32)
    x = ints(-2, 2, (B, C, H, W))
    w = ints(-1, 1, (Co, C, kh, kw))
    b = ints(-8, 7, Co) + np.float32(0.5)
    go = ints(-1, 1, (B, Co, Ho, Wo))
    msk = ints(0, 2, (B, dg * KK, Ho, Wo)) / 2
    k = np.where(rng.random((B, 2 * dg * KK, Ho, Wo)) < far, rng.integers(-25, 25, (B, 2 * dg * KK, Ho, Wo)),
                 rng.integers(-4, 4, (B, 2 * dg * KK, Ho, Wo)))
    off = (k / 2 + 0.25).astype(np.float32)
    return x, off, msk.astype(np.float32), w, b, go


@pytest.mark.parametrize("shape", [(2, 16, 8, 11, 13, 2, 3, (2, 1), 1, 2), (1, 24, 16, 9, 20, 3, (3, 4), 1, 0, 1)])
def test_oracle_is_exact_in_fp32_on_the_lattice(oracle, shape):
    """The argument of _lattice_case checked on the oracle itself: its fp32 build (the reference's arithmetic) gives the
    float64 build's results bit for bit; the first shape has offsets beyond the box and the image at every tap."""
    x, off, msk, w, b, go = _lattice_case(np.random.default_rng(3), shape, far=1 / 2 if shape[0] == 2 else 1 / 8)
    ints, _, _ = _geom(shape)
    s, p, d, dg = ints[2:4], ints[4:6], ints[6:8], ints[8]
    assert (np.abs(off) > 7).mean() > 0.2 or shape[0] == 1
    f32 = oracle.dcn_forward(x, off, msk, w, b, s, p, d, dg, precision="f32")
    assert np.array_equal(f32, oracle.dcn_forward(x, off, msk, w, b, s, p, d, dg))
    for name, a, c in zip(GRADS, oracle.dcn_backward(x, off, msk, w, b, go, s, p, d, dg, precision="f32"),
                          oracle.dcn_backward(x, off, msk, w, b, go, s, p, d, dg)):
        assert np.array_equal(a, c), name


# ---------------------------------------------------------------- failure messages
def _where(name, idx, shape, sp):
    """Where element idx of result `name` is computed: tile and CTA of dcn_work_split."""
    B, C, Co, H, W, dg = shape[:6]
    (kh, kw, sh, sw, ph, pw, *_), Ho, Wo = _geom(shape)
    KK, f, bw = sp["KK"], sp["fwd"], sp["bwd"]

    def tile(b, y, x):
        return b * sp["ntiles"] + (y // 8) * sp["tiles_x"] + x // 16

    if name == "out":
        if not f["fwd_tc"]:
            return "CUDA-core forward"
        b, _, y, x = idx
        t = tile(b, y, x)
        return f"tile {t}, forward CTA {t % f['grid']} (step {t // f['grid']} of its walk)"
    if not bw["box"]:
        return "CUDA-core backward"
    if name in ("grad_weight", "grad_bias"):
        row = idx[1] // 8 // bw["GPC"] if name == "grad_weight" else 0
        return f"GEMM3 of the CTAs in row {row} (all their tiles), dcn_box_reduce_partials"
    b, ch, y, x = idx
    if name == "grad_input":
        # the tile whose undeformed footprint holds (y, x); dcn_gin_collect adds its box, up to five neighbouring
        # boxes and the far samples of any tile within reach of the offsets
        unit = ch // 8
        y, x = min(max((y + ph) // sh, 0), Ho - 1), min(max((x + pw) // sw, 0), Wo - 1)
        prefix = "boxes around "
    else:                                 # grad_offset / grad_mask / grad_offset_mask: output-pixel resolution
        per_group = 2 * KK if name == "grad_offset" or (name == "grad_offset_mask" and ch < 2 * dg * KK) else KK
        g = ch // per_group if name != "grad_offset_mask" or ch < 2 * dg * KK else (ch - 2 * dg * KK) // KK
        unit = g * bw["ncs"]
        prefix = ""
    t = tile(b, y, x)
    return (f"{prefix}tile {t}, backward CTA ({t % bw['grid_x']}, {unit // bw['GPC']}) "
            f"(step {t // bw['grid_x']} of its walk)")


def _mismatch(name, got, want, shape):
    """Failure message of an exact comparison: how many elements differ and, for the first few, their index, values,
    tile and the CTA that dcn_work_split assigns them."""
    got, want = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    bad = torch.nonzero(got != want).tolist()
    sp = dcn_work_split(shape, torch.cuda.get_device_properties(0).multi_processor_count)
    where = [f"{tuple(i)}: {float(got[tuple(i)])} != {float(want[tuple(i)])}, {_where(name, i, shape, sp)}"
             for i in bad[:6]]
    return f"{name}: {len(bad)} of {want.numel()} elements differ at {shape}; " + "; ".join(where)


# ---------------------------------------------------------------- exact comparisons at PIPELINE_SHAPES
_EXPECTED = {}


def _expected(oracle, shape, packed=False):
    """(inputs, float64 oracle results) of the lattice case of `shape`, cached for the module. packed: the mask is the
    sigmoid of logits 0, i.e. 1/2 everywhere."""
    key = (shape, packed)
    if key not in _EXPECTED:
        x, off, msk, w, b, go = _lattice_case(np.random.default_rng(sum(shape[:6])), shape)
        if packed:
            msk = np.full_like(msk, 0.5)
        ints, _, _ = _geom(shape)
        s, p, d, dg = ints[2:4], ints[4:6], ints[6:8], ints[8]
        want = [oracle.dcn_forward(x, off, msk, w, b, s, p, d, dg), *oracle.dcn_backward(x, off, msk, w, b, go, s, p, d, dg)]
        _EXPECTED[key] = ((x, off, msk, w, b, go), want)
    return _EXPECTED[key]


def _check_all(shape, got, want, dtype=torch.float32):
    """out and the three activation gradients equal the float64 values rounded once to `dtype`; grad_weight and
    grad_bias (fp32 in every entry) equal them exactly."""
    from gpu_util import t
    for name, g, r in zip(("out",) + GRADS, got, want):
        r = t(r, torch.float64).to(dtype if name not in ("grad_weight", "grad_bias") else torch.float32)
        assert g.dtype == r.dtype, name
        assert torch.equal(g, r), _mismatch(name, g, r, shape)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PIPELINE_SHAPES)
def test_fp32_exact_on_the_lattice(dcn, ext, oracle, shape):
    """dcn_v2_conv forward + backward through autograd: the backward reads the forward's blocked input copy."""
    from gpu_util import t
    (x, off, msk, w, b, go), want = _expected(oracle, shape)
    ints, _, _ = _geom(shape)
    ts = [t(a).requires_grad_() for a in (x, off, msk, w, b)]
    out = dcn.dcn_v2_conv(*ts, ints[2:4], ints[4:6], ints[6:8], ints[8])
    if _library_plans(shape)[1]:
        assert ext._blocked_cache[0][0] == ext._blocked_key(ts[0], ext._geom(ts[0], ts[3], *ints)[0])
    out.backward(t(go))
    _check_all(shape, [out.detach()] + [v.grad for v in ts], want)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PIPELINE_SHAPES)
def test_packed_exact_on_the_lattice(ext, oracle, shape):
    """The packed entries with mask logits 0: the in-kernel sigmoid gives 1/2 exactly, the logit gradient is
    grad_mask * 1/4."""
    from gpu_util import t
    (x, off, _, w, b, go), want = _expected(oracle, shape, packed=True)
    ints, _, _ = _geom(shape)
    om = t(np.concatenate([off, np.zeros((off.shape[0], off.shape[1] // 2) + off.shape[2:], np.float32)], 1))
    xt, wt, bt = t(x), t(w), t(b)
    out = ext.dcn_v2_forward_packed(xt, wt, bt, om, *ints)
    g_in, g_om, g_w, g_b = ext.dcn_v2_backward_packed(xt, wt, bt, om, t(go), *ints)
    out_w, gi_w, goff_w, gm_w, gw_w, gb_w = want
    _check_all(shape, [out, g_in, g_om, g_w, g_b], [out_w, gi_w, np.concatenate([goff_w, gm_w / 4], 1), gw_w, gb_w])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("shape", PIPELINE_SHAPES)
def test_16bit_exact_on_the_lattice(ext, oracle, shape, dtype):
    """The _bf16 / _fp16 entries (native 16-bit activation I/O) on the same inputs, exact in both types: each 16-bit
    result is the float64 value rounded once, grad_weight / grad_bias (fp32) are exact."""
    from gpu_util import t
    (x, off, msk, w, b, go), want = _expected(oracle, shape)
    ints, _, _ = _geom(shape)
    xt, offt, mt, got = (t(a).to(dtype) for a in (x, off, msk, go))
    out = ext.dcn_v2_forward(xt, t(w), t(b), offt, mt, *ints)
    grads = ext.dcn_v2_backward(xt, t(w), t(b), offt, mt, got, *ints)
    _check_all(shape, [out, *grads], want, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("env,shape", [("EBFI_DCN_DETERMINISTIC", PIPELINE_SHAPES[1]),
                                       ("EBFI_DCN_IMPL", PIPELINE_SHAPES[6])], ids=["deterministic", "simt"])
def test_other_backwards_exact_on_the_lattice(ext, oracle, monkeypatch, env, shape):
    """The deterministic backward (dcn_bwd_tc.cu, int64 fixed-point grad_input) and the CUDA-core kernels
    (EBFI_DCN_IMPL=simt, forward too) give the same bits as float64, hence as the box backward."""
    from gpu_util import t
    monkeypatch.setenv(env, "1" if env == "EBFI_DCN_DETERMINISTIC" else "simt")
    (x, off, msk, w, b, go), want = _expected(oracle, shape)
    ints, _, _ = _geom(shape)
    xt, offt, mt, wt, bt = (t(a) for a in (x, off, msk, w, b))
    out = ext.dcn_v2_forward(xt, wt, bt, offt, mt, *ints)
    grads = ext.dcn_v2_backward(xt, wt, bt, offt, mt, t(go), *ints)
    _check_all(shape, [out, *grads], want)


# ---------------------------------------------------------------- long accumulation chains (random data)
def column_weight_grads(x, off, msk, go, ints, chunk=1 << 16):
    """grad_weight and grad_bias of DCNv2 in float64 with torch, on the device of the arguments: the column tensor
    (bilinear sampling with the reference's window and per-corner bounds, im2col_cuda.cu:25-54, :180) one sample and
    `chunk` output pixels at a time, contracted with grad_output by a float64 matmul."""
    kh, kw, sh, sw, ph, pw, dh, dw, dg = ints
    B, C, H, W = x.shape
    Co, Ho, Wo = go.shape[1:]
    KK, cpg = kh * kw, C // dg
    F = torch.nn.functional
    dev = x.device
    gw = torch.zeros(Co, C * KK, dtype=torch.float64, device=dev)
    ho, wo = torch.meshgrid(torch.arange(Ho, device=dev), torch.arange(Wo, device=dev), indexing="ij")
    ho, wo = ho.reshape(-1).double(), wo.reshape(-1).double()
    for b in range(B):
        xp = F.pad(x[b].double(), (1, 1, 1, 1)).reshape(dg, cpg, (H + 2) * (W + 2))     # zero border: per-corner bounds
        o = off[b].double().reshape(dg, KK, 2, Ho * Wo)
        m = msk[b].double().reshape(dg, KK, Ho * Wo)
        g = go[b].double().reshape(Co, Ho * Wo)
        for p0 in range(0, Ho * Wo, chunk):
            sl = slice(p0, p0 + chunk)
            col = torch.empty(dg, cpg, KK, ho[sl].numel(), dtype=torch.float64, device=dev)
            for t in range(KK):
                i, j = divmod(t, kw)
                y = ho[sl] * sh - ph + i * dh + o[:, t, 0, sl]
                xx = wo[sl] * sw - pw + j * dw + o[:, t, 1, sl]
                inside = (y > -1) & (xx > -1) & (y < H) & (xx < W)
                y0, x0 = torch.floor(y), torch.floor(xx)
                ly, lx = y - y0, xx - x0
                y0 = y0.clamp(-1, H - 1).long() + 1
                x0 = x0.clamp(-1, W - 1).long() + 1
                v = 0
                for dy, dx, wt in ((0, 0, (1 - ly) * (1 - lx)), (0, 1, (1 - ly) * lx), (1, 0, ly * (1 - lx)), (1, 1, ly * lx)):
                    idx = ((y0 + dy) * (W + 2) + x0 + dx)[:, None, :].expand(dg, cpg, -1)
                    v = v + xp.gather(2, idx) * (wt * inside)[:, None, :]
                col[:, :, t] = v * m[:, t, None, sl]
            gw += g[:, sl] @ col.reshape(C * KK, -1).T
    return gw.reshape(Co, C, kh, kw), go.double().sum((0, 2, 3))


def _random_case(rng, shape, one_signed=False):
    B, C, Co, H, W, dg = shape[:6]
    (kh, kw, *_), Ho, Wo = _geom(shape)
    x = rng.standard_normal((B, C, H, W), dtype=np.float32)
    w = rng.standard_normal((Co, C, kh, kw), dtype=np.float32)
    b = rng.standard_normal(Co, dtype=np.float32)
    off = (2 * rng.standard_normal((B, 2 * dg * kh * kw, Ho, Wo))).astype(np.float32)
    msk = (1 / (1 + np.exp(-rng.standard_normal((B, dg * kh * kw, Ho, Wo))))).astype(np.float32)
    go = rng.standard_normal((B, Co, Ho, Wo), dtype=np.float32)
    if one_signed:
        x, go = np.abs(x), np.abs(go)
    return x, off, msk, w, b, go


def test_column_restatement_matches_the_oracle(oracle):
    shape = (2, 16, 8, 11, 13, 2, 3, (2, 1), 1, 2)
    x, off, msk, w, b, go = _random_case(np.random.default_rng(5), shape)
    off *= 3                                             # far samples, out of the image too
    ints, _, _ = _geom(shape)
    gw, gb = column_weight_grads(*(torch.from_numpy(a) for a in (x, off, msk, go)), ints, chunk=50)
    want = oracle.dcn_backward(x, off, msk, w, b, go, ints[2:4], ints[4:6], ints[6:8], ints[8])
    assert rel_err(gw.numpy(), want[3]) < 1e-6 and rel_err(gb.numpy(), want[4]) < 1e-6


# (Cout, C) with a 2x2 kernel, dg = 8: nacc = 2 at Cout = 80, 1 at 96 and 128. With 3x3 the fp32 plan of Cout > 64
# does not fit shared memory (the CUDA-core kernel runs), so the short hi*hi chains are reached by kernels of <= 6 taps;
# (128, 576) is the longest chain the forward accepts at K = C * KK = 2304.
CHAIN_SHAPES = [(co, c) for co in (80, 96, 128) for c in (64, 128, 256)] + [(128, 576)]


def _chain_shape(co, c):
    return (1, c, co, 32, 48, 8, 2, 1, 0, 1)


def test_chain_shapes_take_the_tensor_core_forward():
    from ebfi_be_b200 import _lib as L
    for co, c in CHAIN_SHAPES:
        shape = _chain_shape(co, c)
        sp = dcn_work_split(shape, 148)
        assert sp["fwd"]["fwd_tc"] and sp["fwd"]["nacc"] == {80: 2, 96: 1, 128: 1}[co], shape
        ints, _, _ = _geom(shape)
        assert L.load().ebfi_dcnv2_forward_workspace_bytes(L.DcnGeom(1, c, 32, 48, co, *ints, 0)) > 256, shape
    assert not dcn_work_split((1, 64, 80, 32, 48, 8, 3, 1, 1, 1), 148)["fwd"]["fwd_tc"]


@pytest.mark.gpu
@pytest.mark.parametrize("co,c", CHAIN_SHAPES)
def test_forward_chain_against_fp64(ext, oracle, co, c):
    from gpu_util import n, t
    shape = _chain_shape(co, c)
    x, off, msk, w, b, _ = _random_case(np.random.default_rng(co + c), shape)
    ints, _, _ = _geom(shape)
    out = n(ext.dcn_v2_forward(t(x), t(w), t(b), t(off), t(msk), *ints))
    err = rel_err(out, oracle.dcn_forward(x, off, msk, w, b, ints[2:4], ints[4:6], ints[6:8], ints[8]))
    sp = dcn_work_split(shape, 148)["fwd"]
    steps = c // 8 * sp["TPR"] * 3
    print(f"forward Cout {co} C {c} K {c * 4}: {steps} hi*hi MMA steps over {sp['nacc']} accumulator(s), "
          f"{_ceil(steps, sp['nacc'])} per accumulator: rel err {err:.2e}")
    assert err < FWD_TOL


TRAIN = (8, 64, 64, 256, 256, 8, 3, 1, 1, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("one_signed", [False, True], ids=["random", "one_signed"])
def test_backward_weight_chain_at_the_training_size(ext, one_signed):
    """B = 8, 256 x 256 (56 tiles per CTA column at 148 SMs): GEMM3 accumulates grad_weight in TMEM over every tile of
    a CTA's walk. One-signed data (input >= 0, grad_output >= 0) makes every term of grad_bias and most of grad_weight
    the same sign, the worst case of the round-toward-zero accumulate."""
    from gpu_util import t
    x, off, msk, w, b, go = (t(a) for a in _random_case(np.random.default_rng(8), TRAIN, one_signed))
    ints, _, _ = _geom(TRAIN)
    grads = ext.dcn_v2_backward(x, w, b, off, msk, go, *ints)
    want_w, want_b = column_weight_grads(x, off, msk, go, ints)
    ew = rel_err(grads[3].cpu().numpy(), want_w.cpu().numpy())
    eb = rel_err(grads[4].cpu().numpy(), want_b.cpu().numpy())
    print(f"backward B=8 256x256 {'one-signed' if one_signed else 'random'}: "
          f"{dcn_work_split(TRAIN, torch.cuda.get_device_properties(0).multi_processor_count)['bwd']['per']} tiles per "
          f"CTA column, grad_weight rel err {ew:.2e}, grad_bias {eb:.2e}")
    assert ew < GRAD_TOL and eb < GRAD_TOL
