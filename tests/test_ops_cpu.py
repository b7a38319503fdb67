"""torch.ops.ebfi_b200: schemas, fakes and fake-mode traces, without a GPU (FakeTensorMode builds fake CUDA tensors on
a CPU-only machine). The GPU side (opcheck, compiled bits, export) is tests/test_ops_gpu.py."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import ebfi_be_b200  # noqa: F401  (registers the ops)
from ebfi_be_b200 import dcn_v2, frame_ops, kernelconv2d, modification

OPS = {
    "dcn_v2_forward": "(Tensor input, Tensor weight, Tensor bias, Tensor offset, Tensor mask, SymInt kernel_h, "
                      "SymInt kernel_w, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, "
                      "SymInt dilation_h, SymInt dilation_w, SymInt deformable_group) -> Tensor",
    "dcn_v2_backward": "(Tensor input, Tensor weight, Tensor bias, Tensor offset, Tensor mask, Tensor grad_output, "
                       "SymInt kernel_h, SymInt kernel_w, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, "
                       "SymInt dilation_h, SymInt dilation_w, SymInt deformable_group) "
                       "-> (Tensor, Tensor, Tensor, Tensor, Tensor)",
    "dcn_v2_forward_packed": "(Tensor input, Tensor weight, Tensor bias, Tensor offset_mask, SymInt kernel_h, "
                             "SymInt kernel_w, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, "
                             "SymInt dilation_h, SymInt dilation_w, SymInt deformable_group, "
                             "Tensor(a13!)? abs_offset_sum) -> Tensor",
    "dcn_v2_backward_packed": "(Tensor input, Tensor weight, Tensor bias, Tensor offset_mask, Tensor grad_output, "
                              "SymInt kernel_h, SymInt kernel_w, SymInt stride_h, SymInt stride_w, SymInt pad_h, "
                              "SymInt pad_w, SymInt dilation_h, SymInt dilation_w, SymInt deformable_group) "
                              "-> (Tensor, Tensor, Tensor, Tensor)",
    "fac_forward": "(Tensor input, Tensor kernel, SymInt kernel_size, Tensor(a3!) output) -> ()",
    "fac_backward": "(Tensor input, Tensor kernel, SymInt kernel_size, Tensor grad_output, Tensor(a4!) grad_input, "
                    "Tensor(a5!) grad_kernel) -> ()",
    "fac_replpad_forward": "(Tensor input, Tensor kernel, SymInt kernel_size) -> Tensor",
    "fac_replpad_backward": "(Tensor input, Tensor kernel, SymInt kernel_size, Tensor grad_output) -> (Tensor, Tensor)",
    "kpn_fused_forward": "(Tensor event_feat, Tensor frame_feat, Tensor conv_weight, Tensor conv_bias, "
                         "SymInt kernel_size, float negative_slope) -> Tensor",
    "kpn_fused_backward": "(Tensor event_feat, Tensor frame_feat, Tensor conv_weight, Tensor conv_bias, "
                          "SymInt kernel_size, float negative_slope, Tensor grad_output) -> (Tensor, Tensor, Tensor)",
    "frame_to_lap": "(Tensor ims) -> Tensor",
    "frame_to_dcp": "(Tensor ims, SymInt sz=35) -> Tensor",
}

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
CUDA = torch.device("cuda")
DCN_INTS = (3, 3, 1, 1, 1, 1, 1, 1, 8)


def op(name):
    return getattr(torch.ops.ebfi_b200, name).default


@pytest.fixture
def fake():
    with FakeTensorMode(allow_non_fake_inputs=False) as mode:
        yield mode


def e(*shape, dtype=F32):
    return torch.empty(shape, dtype=dtype, device=CUDA)


def cuda_module(cls, *args, **kwargs):
    """An eval-mode module with fake CUDA parameters (inside the `fake` fixture)."""
    with torch.device(CUDA):
        return cls(*args, **kwargs).eval()


@pytest.mark.parametrize("name", sorted(OPS))
def test_registered_with_schema(name):
    assert str(op(name)._schema) == f"ebfi_b200::{name}{OPS[name]}"


# (activation dtype of input / offset / mask / grad_output, parameter dtype) -> output dtype, as shims/_ext.py
DCN_DTYPES = [((F32, F32, F32), F32, F32), ((BF16, BF16, BF16), BF16, BF16), ((F16, F16, F16), F16, F16),
              ((BF16, F32, F32), F32, BF16), ((F32, F16, F16), F32, F16), ((BF16, BF16, BF16), F32, BF16),
              ((F16, F32, F16), F16, F16)]


@pytest.mark.parametrize("acts,param,out", DCN_DTYPES)
@pytest.mark.parametrize("geom", [(2, 64, 20, 24, 32, 3, 3, 1, 1, 1, 1, 1, 1, 8),
                                  (1, 16, 17, 9, 8, 3, 3, 2, 1, 1, 0, 2, 1, 4),
                                  (1, 8, 5, 5, 8, 1, 1, 1, 1, 0, 0, 1, 1, 1)])
def test_dcn_fakes(fake, acts, param, out, geom):
    B, C, H, W, Co, kh, kw, sh, sw, ph, pw, dh, dw, dg = geom
    ints = geom[5:]
    Ho = (H + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    Wo = (W + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    taps = dg * kh * kw
    x, off, msk = e(B, C, H, W, dtype=acts[0]), e(B, 2 * taps, Ho, Wo, dtype=acts[1]), e(B, taps, Ho, Wo, dtype=acts[2])
    w, b, go = e(Co, C, kh, kw, dtype=param), e(Co, dtype=param), e(B, Co, Ho, Wo, dtype=acts[0])
    y = op("dcn_v2_forward")(x, w, b, off, msk, *ints)
    assert (y.shape, y.dtype, y.device.type) == ((B, Co, Ho, Wo), out, "cuda")
    grads = op("dcn_v2_backward")(x, w, b, off, msk, go, *ints)
    want = [out] * 3 + ([param] * 2 if out != F32 else [F32] * 2)
    assert [(g.shape, g.dtype) for g in grads] == [(t.shape, d) for t, d in zip((x, off, msk, w, b), want)]
    om = e(B, 3 * taps, Ho, Wo, dtype=acts[1])
    stat = e(1)
    for s in (None, stat):
        y = op("dcn_v2_forward_packed")(x, w, b, om, *ints, s)
        assert (y.shape, y.dtype) == ((B, Co, Ho, Wo), out)
    grads = op("dcn_v2_backward_packed")(x, w, b, om, go, *ints)
    assert [(g.shape, g.dtype) for g in grads] == [(t.shape, d) for t, d in zip((x, om, w, b), [out] * 2 + want[3:])]


def test_dcn_fakes_raise_as_eager(fake):
    x, w, b = e(1, 64, 16, 16), e(32, 64, 3, 3), e(32)
    off, msk, go = e(1, 144, 16, 16), e(1, 72, 16, 16), e(1, 32, 16, 16)
    fwd, bwd = op("dcn_v2_forward"), op("dcn_v2_backward")
    fwd(x, w, b, off, msk, *DCN_INTS)
    with pytest.raises(RuntimeError, match="all tensors must be float32"):       # bf16 with fp16
        fwd(x.bfloat16(), w, b, off.half(), msk, *DCN_INTS)
    with pytest.raises(RuntimeError, match="all tensors must be float32"):       # fp32 activations, bf16 weight
        fwd(x, w.bfloat16(), b, off, msk, *DCN_INTS)
    with pytest.raises(RuntimeError, match="kernel channels"):
        fwd(e(1, 32, 16, 16), w, b, off, msk, *DCN_INTS)
    with pytest.raises(RuntimeError, match="kernel shape"):
        fwd(x, w, b, off, msk, 1, 1, *DCN_INTS[2:])
    with pytest.raises(RuntimeError, match="offset/mask shapes"):
        fwd(x, w, b, off[:, :100], msk, *DCN_INTS)
    with pytest.raises(RuntimeError, match="not divisible"):
        fwd(x, w, b, off, msk, *DCN_INTS[:-1], 7)
    with pytest.raises(RuntimeError, match="empty output"):
        fwd(e(1, 64, 2, 16), w, b, off, msk, 3, 3, 1, 1, 0, 1, 1, 1, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        fwd(x, w, b, off, torch.empty(1, 72, 16, 16), *DCN_INTS)
    with pytest.raises(RuntimeError, match="grad_output has the wrong shape"):
        bwd(x, w, b, off, msk, go[:, :16], *DCN_INTS)
    with pytest.raises(RuntimeError, match="input tensor has to be contiguous"):
        bwd(x.transpose(2, 3), w, b, off, msk, go, *DCN_INTS)
    with pytest.raises(RuntimeError, match="offset_mask shape"):
        op("dcn_v2_forward_packed")(x, w, b, off, *DCN_INTS, None)
    with pytest.raises(RuntimeError, match="abs_offset_sum"):
        op("dcn_v2_forward_packed")(x, w, b, e(1, 216, 16, 16), *DCN_INTS, e(2))


def test_dcn_output_size_matches_the_library():
    """The fakes' size formula against ebfi_dcnv2_output_size, where the library is built."""
    from ebfi_be_b200 import _lib as L
    from ebfi_be_b200.ops import _out_len
    try:
        lib = L.load()
    except (RuntimeError, OSError) as err:
        pytest.skip(str(err))
    for n in (1, 2, 3, 7, 16):
        for k, s, p, d in [(3, 1, 1, 1), (3, 2, 0, 1), (5, 3, 0, 2), (1, 2, 0, 1), (3, 3, 1, 2), (4, 2, 1, 1)]:
            g = L.DcnGeom(1, 8, n, n, 8, k, k, s, s, p, p, d, d, 1, 0)
            ho, wo = L.c_int(), L.c_int()
            rc = lib.ebfi_dcnv2_output_size(g, ho, wo)
            want = _out_len(n, k, s, p, d)
            assert (rc == 0) == (want > 0), (n, k, s, p, d)
            if rc == 0:
                assert ho.value == want


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
@pytest.mark.parametrize("K", [1, 3, 5])
def test_fac_fakes(fake, dtype, K):
    B, C, H, W = 2, 4, 9, 13
    xp, ker = e(B, C, H + K - 1, W + K - 1, dtype=dtype), e(B, C * K * K, H, W, dtype=dtype)
    out, go = e(B, C, H, W, dtype=dtype), e(B, C, H, W, dtype=dtype)
    assert op("fac_forward")(xp, ker, K, out) is None
    assert op("fac_backward")(xp, ker, K, go, torch.empty_like(xp), torch.empty_like(ker)) is None
    x = e(B, C, H, W, dtype=dtype)
    y = op("fac_replpad_forward")(x, ker, K)
    assert (y.shape, y.dtype) == (x.shape, dtype)
    gi, gk = op("fac_replpad_backward")(x, ker, K, go)
    assert (gi.shape, gi.dtype, gk.shape, gk.dtype) == (x.shape, dtype, ker.shape, dtype)
    with pytest.raises(RuntimeError, match="do not fit kernel_size"):
        op("fac_forward")(x, ker, K + 2, out)
    with pytest.raises(RuntimeError, match="output must be"):
        op("fac_forward")(xp, ker, K, out[:, :2])
    with pytest.raises(RuntimeError, match="both"):
        op("fac_replpad_forward")(x, ker.float() if dtype != F32 else ker.half(), K)
    with pytest.raises(RuntimeError, match="grad_output"):
        op("fac_replpad_backward")(x, ker, K, go.double())
    with pytest.raises(RuntimeError, match="grad_input / grad_kernel"):
        op("fac_backward")(xp, ker, K, go, torch.empty_like(xp[:1]), torch.empty_like(ker))


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
@pytest.mark.parametrize("Ce,Cf,K", [(64, 64, 5), (32, 0, 3), (16, 16, 1)])
def test_kpn_fakes(fake, dtype, Ce, Cf, K):
    B, H, W = 2, 11, 7
    ev, fr, go = e(B, Ce, H, W, dtype=dtype), e(B, Cf, H, W, dtype=dtype), e(B, Ce, H, W, dtype=dtype)
    w, b = e(Ce * K * K, Ce + Cf, 3, 3), e(Ce * K * K)
    y = op("kpn_fused_forward")(ev, fr, w, b, K, 0.01)
    assert (y.shape, y.dtype) == (ev.shape, dtype)
    gp, ge, gb = op("kpn_fused_backward")(ev, fr, w, b, K, 0.01, go)
    assert [(t.shape, t.dtype) for t in (gp, ge, gb)] == [((B, Ce * K * K, H, W), dtype), (ev.shape, F32),
                                                            ((Ce * K * K,), F32)]
    with pytest.raises(RuntimeError, match="conv_weight / conv_bias float32"):
        op("kpn_fused_forward")(ev, fr, w.to(BF16), b, K, 0.01)
    with pytest.raises(RuntimeError, match="all float32"):
        op("kpn_fused_backward")(ev, fr, w, b, K, 0.01, go.double())
    with pytest.raises(RuntimeError, match="shapes do not match"):
        op("kpn_fused_forward")(ev, fr, w, b, K + 2, 0.01)
    with pytest.raises(RuntimeError, match="supports"):      # Ce + Cf = 24 is not a multiple of 32
        op("kpn_fused_forward")(ev[:, :12], e(B, 12, H, W, dtype=dtype), e(12 * K * K, 24, 3, 3), e(12 * K * K), K,
                                0.01)


@pytest.mark.parametrize("dtype", [F32, BF16, F16, torch.uint8])
def test_frame_map_fakes(fake, dtype):
    ims = e(2, 3, 37, 21, dtype=dtype)
    for y in (op("frame_to_lap")(ims), op("frame_to_dcp")(ims, 35), op("frame_to_dcp")(ims)):
        assert (y.shape, y.dtype) == ((2, 1, 37, 21), F32)
    with pytest.raises(RuntimeError, match="expected a"):
        op("frame_to_lap")(e(2, 4, 8, 8))


def test_dcn_fake_is_symbolic(fake):
    """The DCN fakes size their outputs by SymInt arithmetic: an export with dynamic H and W keeps them symbolic
    through stride 2."""
    dcn = cuda_module(dcn_v2.DCN_sep, 64, 64, 3, 2, 1, deformable_groups=8)
    H, W = torch.export.Dim("H", min=8, max=512), torch.export.Dim("W", min=8, max=512)
    spec = {2: H, 3: W}
    ep = torch.export.export(dcn, (e(1, 64, 40, 24), e(1, 64, 40, 24)), dynamic_shapes=(spec, spec))
    node, = [n for n in ep.graph.nodes if n.target is op("dcn_v2_forward_packed")]
    out = node.meta["val"].shape
    assert not isinstance(out[2], int) and not isinstance(out[3], int), out
    assert [int(str(v)) if str(v).isdigit() else None for v in out[:2]] == [1, 64]


# ------------------------------------------------------------------- fake-mode export of the modules that call them
def _export_ops(mod, *args):
    ep = torch.export.export(mod, args)
    return {n.target.__name__.split(".")[0] for n in ep.graph.nodes
            if n.op == "call_function" and getattr(n.target, "namespace", None) == "ebfi_b200"}


def test_export_on_fake_inputs_contains_the_ops(fake):
    dcn = cuda_module(dcn_v2.DCN_sep, 64, 64, 3, 1, 1, deformable_groups=8)
    assert _export_ops(dcn, e(1, 64, 24, 24), e(1, 64, 24, 24)) == {"dcn_v2_forward_packed"}
    plain = cuda_module(dcn_v2.DCNv2, 64, 64, 3, 1, 1, deformable_groups=8)
    assert _export_ops(plain, e(1, 64, 24, 24), e(1, 144, 24, 24), e(1, 72, 24, 24)) == {"dcn_v2_forward"}
    assert _export_ops(kernelconv2d.KernelConv2D(5), e(1, 8, 24, 24), e(1, 200, 24, 24)) == {"fac_replpad_forward"}
    kpn = cuda_module(modification.KernelPrediction, 32, 5).requires_grad_(False)   # inference: the fused forward
    assert _export_ops(kpn, e(1, 32, 24, 24), e(1, 32, 24, 24)) == {"kpn_fused_forward"}

    class Maps(torch.nn.Module):
        def forward(self, ims):
            return frame_ops.Frame2Lap(ims), frame_ops.Frame2DCP(ims)
    assert _export_ops(Maps(), e(1, 3, 24, 24)) == {"frame_to_lap", "frame_to_dcp"}


def test_export_padded_kernelconv2d_function(fake):
    class Padded(torch.nn.Module):
        def forward(self, x, k):
            return kernelconv2d.KernelConv2DFunction.apply(x, k, 3)
    assert _export_ops(Padded(), e(1, 4, 10, 10), e(1, 36, 8, 8)) == {"fac_forward"}
