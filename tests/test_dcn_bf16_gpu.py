"""DCNv2 with bf16 activations (mixed precision): the *_bf16 entry points of the tensor-core kernels, the boundary
conversion everywhere else, and the modules under torch.autocast.

The bf16 kernels change only the activation loads and stores, so on bf16-valued inputs they must reproduce the fp32
kernels bit for bit: activations rounded once to bf16, grad_weight / grad_bias equal. Offsets stay within |o| <= 4 px so
that every sample is inside its box: outside it, grad_input takes float red.global.add in both dtypes, whose order
varies run to run."""
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu
BF16_TOL = 2.0 ** -8        # one bf16 rounding per result, relative to max|ref| (test_dcn_gpu.py's bf16 tolerance)


@pytest.fixture(scope="module")
def ext():
    from ebfi_be_b200.shims import _ext
    return _ext


def _dev():
    return torch.device("cuda:0")


def _bf(t):
    return t.bfloat16().to(_dev())


def _case(shape, seed, packed=False, obound=4.0):
    """bf16-valued activations (bf16 tensors), fp32 parameters. shape = (B, C, Co, H, W, k, (sh, sw), pad, dil, dg)."""
    B, C, Co, H, W, k, (sh, sw), p, d, dg = shape
    g = torch.Generator().manual_seed(seed)
    Ho, Wo = (H + 2 * p - (d * (k - 1) + 1)) // sh + 1, (W + 2 * p - (d * (k - 1) + 1)) // sw + 1
    nt = dg * k * k
    x = _bf(torch.randn(B, C, H, W, generator=g))
    off = _bf((torch.rand(B, 2 * nt, Ho, Wo, generator=g) * 2 - 1) * obound)
    if packed:
        om = torch.cat([off, _bf(torch.randn(B, nt, Ho, Wo, generator=g))], 1)
        acts = (x, om)
    else:
        acts = (x, off, _bf(torch.rand(B, nt, Ho, Wo, generator=g)))
    w = (torch.randn(Co, C, k, k, generator=g) / (C * k * k) ** 0.5).to(_dev())
    b = torch.randn(Co, generator=g).to(_dev())
    go = _bf(torch.randn(B, Co, Ho, Wo, generator=g))
    ints = (k, k, sh, sw, p, p, d, d, dg)
    return acts, w, b, go, ints


def _fwd_bwd(ext, acts, w, b, go, ints, packed):
    """(output, [gradients]) through the shim; the grads in the order of the backward entry."""
    if packed:
        x, om = acts
        out = ext.dcn_v2_forward_packed(x, w, b, om, *ints)
        return out, ext.dcn_v2_backward_packed(x, w, b, om, go, *ints)
    x, off, m = acts
    out = ext.dcn_v2_forward(x, w, b, off, m, *ints)
    return out, ext.dcn_v2_backward(x, w, b, off, m, go, *ints)


def _box_path(ints, shape):
    """True when this geometry takes the tensor-core forward AND the box backward (the native bf16 backward)."""
    from ebfi_be_b200 import _lib as L
    B, C, Co, H, W = shape[:5]
    g = L.DcnGeom(B, C, H, W, Co, *ints, 0)
    return L.load().ebfi_dcnv2_blocked_input_offset(g) != 0


# (B, C, Co, H, W, k, stride, pad, dil, dg): all take the tensor-core forward and the box backward
TC_SHAPES = [(1, 64, 64, 32, 32, 3, (1, 1), 1, 1, 8),     # the benchmark geometry (cfg1) at 32 x 32
             (1, 64, 64, 24, 40, 3, (1, 1), 1, 1, 2),     # 32 channels per group (running sums), non-square
             (1, 32, 64, 20, 36, 3, (1, 1), 1, 1, 2),     # 16 per group; Wo % 8 != 0: offsets / masks read from global
             (2, 32, 64, 30, 34, 3, (2, 1), 1, 1, 4),     # stride 2 along y, batch 2
             (1, 64, 64, 17, 19, 3, (1, 1), 1, 1, 8)]     # odd sizes: partial tiles, unaligned grad_output rows


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("shape", TC_SHAPES)
def test_bit_identical_to_fp32_kernels(ext, shape, packed):
    acts, w, b, go, ints = _case(shape, 11, packed, obound=4.0 if shape[6] == (1, 1) else 2.0)   # inside the box
    assert _box_path(ints, shape)
    out, grads = _fwd_bwd(ext, acts, w, b, go, ints, packed)
    out32, grads32 = _fwd_bwd(ext, [a.float() for a in acts], w, b, go.float(), ints, packed)
    assert out.dtype == torch.bfloat16 and torch.equal(out, out32.bfloat16())
    n_act = len(acts)
    for i, (g, g32) in enumerate(zip(grads, grads32)):
        if i < n_act:
            assert g.dtype == torch.bfloat16 and torch.equal(g, g32.bfloat16()), i
        else:
            assert g.dtype == torch.float32 and torch.equal(g, g32), i


def test_stride_two_forward_bit_identical(ext):
    """Stride 2 in both directions: the forward is native, the backward (no box path) converts at the boundary."""
    shape = (1, 32, 64, 34, 38, 3, (2, 2), 1, 1, 4)
    acts, w, b, go, ints = _case(shape, 12, obound=2.0)
    assert not _box_path(ints, shape)
    out, grads = _fwd_bwd(ext, acts, w, b, go, ints, False)
    out32, grads32 = _fwd_bwd(ext, [a.float() for a in acts], w, b, go.float(), ints, False)
    assert torch.equal(out, out32.bfloat16())
    assert [g.dtype for g in grads] == [torch.bfloat16] * 3 + [torch.float32] * 2
    for g, g32 in zip(grads, grads32):
        assert rel_err(g.float().cpu().numpy(), g32.float().cpu().numpy()) < BF16_TOL


def _all_bf16(acts, w, b, go):
    return [a.bfloat16() for a in acts], w.bfloat16(), b.bfloat16(), go.bfloat16()


# shapes / settings that the bf16 kernels do not cover (the boundary conversion runs) and one they do
FALLBACKS = [("tc", (1, 64, 64, 24, 24, 3, (1, 1), 1, 1, 8), {}, True),
             ("cout32", (1, 64, 32, 24, 24, 3, (1, 1), 1, 1, 8), {}, False),
             ("cpg4", (1, 16, 64, 24, 24, 3, (1, 1), 1, 1, 4), {}, False),
             ("deterministic", (1, 64, 64, 24, 24, 3, (1, 1), 1, 1, 8), {"EBFI_DCN_DETERMINISTIC": "1"}, True),
             ("simt", (1, 64, 64, 24, 24, 3, (1, 1), 1, 1, 8), {"EBFI_DCN_IMPL": "simt"}, False)]


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("name,shape,env,gin_exact", FALLBACKS, ids=[f[0] for f in FALLBACKS])
def test_all_bf16_unchanged(ext, monkeypatch, name, shape, env, gin_exact, packed):
    """All-bf16 calls give the bits of the boundary conversion (today's path, called directly). grad_input of the
    CUDA-core kernel (float atomics) is order-dependent in both paths: compared at the bf16 tolerance."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    acts, w, b, go, ints = _case(shape, 13, packed)
    acts, w, b, go = _all_bf16(acts, w, b, go)
    out, grads = _fwd_bwd(ext, acts, w, b, go, ints, packed)
    if packed:
        ref_out = ext._bf16_via_fp32(ext.dcn_v2_forward_packed, (acts[0], w, b, acts[1]), ints)
        ref = ext._bf16_via_fp32(ext.dcn_v2_backward_packed, (acts[0], w, b, acts[1], go), ints)
    else:
        ref_out = ext._bf16_via_fp32(ext.dcn_v2_forward, (*acts[:1], w, b, *acts[1:]), ints)
        ref = ext._bf16_via_fp32(ext.dcn_v2_backward, (acts[0], w, b, acts[1], acts[2], go), ints)
    assert torch.equal(out, ref_out)
    for i, (g, r) in enumerate(zip(grads, ref)):
        assert g.dtype == torch.bfloat16
        if i == 0 and not gin_exact:
            assert rel_err(g.float().cpu().numpy(), r.float().cpu().numpy()) < BF16_TOL
        else:
            assert torch.equal(g, r), i
    # the same call with fp32 parameters: the result dtypes of the mixed-precision contract
    w32, b32 = w.float(), b.float()
    grads = (ext.dcn_v2_backward_packed(acts[0], w32, b32, acts[1], go, *ints) if packed else
             ext.dcn_v2_backward(acts[0], w32, b32, acts[1], acts[2], go, *ints))
    assert [g.dtype for g in grads] == [torch.bfloat16] * len(acts) + [torch.float32] * 2


def test_misaligned_grad_output_view_converts(ext):
    """A grad_output that is not 16-byte aligned leaves the bf16 kernels: the call converts (the widened copy is aligned
    again), also right after a native forward whose blocked input copy is still cached."""
    shape = (1, 64, 64, 24, 24, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _case(shape, 14)
    store = torch.empty(go.numel() + 1, dtype=torch.bfloat16, device=_dev())
    go_mis = store[1:].view_as(go)
    go_mis.copy_(go)
    assert go_mis.data_ptr() % 16 != 0
    ext.dcn_v2_forward(x, w, b, off, m, *ints)
    grads = ext.dcn_v2_backward(x, w, b, off, m, go_mis, *ints)
    ref = ext._bf16_via_fp32(ext.dcn_v2_backward, (x, w, b, off, m, go_mis), ints, [torch.bfloat16] * 3 + [torch.float32] * 2)
    assert [g.dtype for g in grads] == [torch.bfloat16] * 3 + [torch.float32] * 2
    for g, r in zip(grads, ref):
        assert torch.equal(g, r)


def test_precision_against_fp64_oracle(ext, oracle):
    """bf16 activations, fp32 parameters: every result within 2^-8 of max|ref| of the fp64 oracle on the same values."""
    shape = (1, 64, 64, 20, 24, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _case(shape, 15, obound=2.0)
    out, grads = _fwd_bwd(ext, (x, off, m), w, b, go, ints, False)
    f = lambda t: t.float().cpu().numpy()
    assert rel_err(f(out), oracle.dcn_forward(f(x), f(off), f(m), f(w), f(b), 1, 1, 1, 8)) < BF16_TOL
    want = oracle.dcn_backward(f(x), f(off), f(m), f(w), f(b), f(go), 1, 1, 1, 8)
    for i, (g, r) in enumerate(zip(grads, want)):
        assert rel_err(f(g), r) < BF16_TOL, i


# ---------------------------------------------------------------- modules under autocast
def _module(kind, seed):
    from ebfi_be_b200 import dcn_v2
    torch.manual_seed(seed)
    if kind == "DCNv2":
        m = dcn_v2.DCNv2(64, 64, 3, 1, 1, deformable_groups=8)
        m.offset_conv = torch.nn.Conv2d(64, 3 * 8 * 9, 3, 1, 1)
        with torch.no_grad():
            m.offset_conv.weight.mul_(0.3)
    else:
        m = (dcn_v2.DCN if kind == "DCN" else dcn_v2.DCN_sep)(64, 64, 3, 1, 1, deformable_groups=8)
        if kind.endswith("unfused"):
            m.fused = False
        with torch.no_grad():              # non-zero offsets, so that their gradients carry signal
            m.conv_offset_mask.weight.normal_(0, 0.02)
    return m.to(_dev())


def _forward(kind, m, x, fea):
    if kind == "DCNv2":
        om = m.offset_conv(fea)
        o1, o2, mask = torch.chunk(om, 3, dim=1)
        return m(x, torch.cat((o1, o2), 1), torch.sigmoid(mask))
    if kind == "DCN":
        return m(x)
    return m(x, fea)


KINDS = ["DCNv2", "DCN", "DCN_sep", "DCN_sep_unfused"]
# relative L2 of the bf16-autocast module against the fp32 module on the same inputs. Measured on a B200: output and
# the DCN's own weight / bias gradients 0.2-0.45 %; the offset conv's parameter gradients, which reach it through
# grad_offset / grad_mask (differences of bf16-rounded neighbouring pixels) and a bf16 convolution backward, 3.8-6.5 %.
REL_L2_DCN, REL_L2_OFFSET_PATH = 0.01, 0.1


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("in_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kind", KINDS)
def test_modules_under_autocast(kind, in_dtype):
    """Each of these raised before bf16 activations could meet fp32 parameters."""
    m = _module(kind, 21)
    g = torch.Generator().manual_seed(22)
    x0 = torch.randn(2, 64, 24, 32, generator=g).to(_dev())
    f0 = torch.randn(2, 64, 24, 32, generator=g).to(_dev())
    go = torch.randn(2, 64, 24, 32, generator=g).to(_dev())

    def run(autocast):
        m.zero_grad(set_to_none=True)
        x = x0.clone().to(in_dtype).requires_grad_()
        fea = f0.clone().to(in_dtype).requires_grad_()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            out = _forward(kind, m, x, fea)
        out.backward(go.to(out.dtype))
        return out, x.grad, fea.grad, {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}

    out, gx, gf, gp = run(True)
    assert out.dtype == torch.bfloat16
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


def test_adam_fit_under_autocast():
    """A DCN_sep student fitted to a teacher by Adam: under autocast it reaches the fp32 fit's loss within 10 %."""
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
        for it in range(120):
            x, f = data[it % 4]
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                loss = torch.nn.functional.mse_loss(s(x, f).float(), targets[it % 4])
            opt.zero_grad()
            loss.backward()
            opt.step()
        with torch.no_grad():
            return sum(float(torch.nn.functional.mse_loss(s(x, f), t)) for (x, f), t in zip(data, targets)) / 4

    start = sum(float(t.pow(2).mean()) for t in targets) / 4
    l32, l16 = fit(False), fit(True)
    print("Adam fit: start %.5f fp32 %.5f autocast %.5f" % (start, l32, l16))
    assert l32 < 0.5 * start
    assert l16 < 1.1 * l32 + 1e-3 * start, (l16, l32, start)


# ---------------------------------------------------------------- reuse, reproducibility, data-parallel, errors
def _autograd_step(x, om, w, b, go):
    from ebfi_be_b200 import dcn_v2
    ts = [t.detach().clone().requires_grad_() for t in (x, om, w, b)]
    out = dcn_v2.dcn_v2_conv_packed(*ts, 1, 1, 1, 8)
    out.backward(go)
    return [out] + [t.grad for t in ts]


def test_blocked_reuse_and_reproducibility(monkeypatch):
    shape = (2, 64, 64, 32, 48, 3, (1, 1), 1, 1, 8)
    (x, om), w, b, go, _ = _case(shape, 41, packed=True)
    a = _autograd_step(x, om, w, b, go)
    a2 = _autograd_step(x, om, w, b, go)
    monkeypatch.setenv("EBFI_DCN_NO_BLOCKED_REUSE", "1")
    c = _autograd_step(x, om, w, b, go)
    for u, v, z in zip(a, a2, c):
        assert torch.equal(u, v) and torch.equal(u, z)


class _SoloComm:
    """world = 1 communicator over a plain device buffer (the pattern of test_dp_gpu.py)."""
    def __init__(self, n):
        from ebfi_be_b200 import _lib as L
        nbytes = int(L.load().ebfi_dp_comm_bytes(n))
        self.buf = torch.zeros(nbytes, dtype=torch.uint8, device=_dev())
        self.struct = L.DpComm(1, 0, (L.c_void * 8)(self.buf.data_ptr()), nbytes)


def test_data_parallel_world_one(ext):
    from ebfi_be_b200 import _lib as L
    shape = (1, 64, 64, 24, 32, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _case(shape, 51)
    comm = _SoloComm(w.numel() + b.numel())
    want = ext.dcn_v2_backward(x, w, b, off, m, go, *ints)
    got = ext.dcn_v2_backward_dp(x, w, b, off, m, go, *ints, comm, defer=True)
    assert got[3].dtype == torch.float32 and got[4].dtype == torch.float32
    L.check(L.load().ebfi_dp_complete(L.stream_ptr(_dev()), comm.struct, L.ptr(got[3]), got[3].numel(),
                                      L.ptr(got[4]), got[4].numel()), "ebfi_dp_complete")
    for a, c in zip(got, want):
        assert torch.equal(a, c)
    got = ext.dcn_v2_backward_dp(x, w, b, off, m, go, *ints, comm)
    for a, c in zip(got, want):
        assert torch.equal(a, c)


def test_errors(ext):
    shape = (1, 64, 64, 16, 16, 3, (1, 1), 1, 1, 8)
    (x, off, m), w, b, go, ints = _case(shape, 61)
    for dt in (torch.float16, torch.float64):
        with pytest.raises(RuntimeError, match="must be float32"):
            ext.dcn_v2_forward(x.to(dt), w, b, off, m, *ints)
        with pytest.raises(RuntimeError, match="must be float32"):
            ext.dcn_v2_backward(x, w, b, off.to(dt), m, go, *ints)
    with pytest.raises(RuntimeError, match="must be float32"):          # fp32 activations need fp32 parameters
        ext.dcn_v2_forward(x.float(), w.bfloat16(), b, off.float(), m.float(), *ints)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        ext.dcn_v2_forward(x.cpu(), w, b, off, m, *ints)

    def shape_errors(x, off, m, go):
        msgs = []
        for call in (lambda: ext.dcn_v2_forward(x, w, b, off[:, :-2], m, *ints),
                     lambda: ext.dcn_v2_backward(x, w, b, off, m, go[:, :, :-1].contiguous(), *ints),
                     lambda: ext.dcn_v2_forward_packed(x, w, b, off, *ints)):
            with pytest.raises(RuntimeError) as e:
                call()
            msgs.append(str(e.value))
        return msgs
    assert shape_errors(x, off, m, go) == shape_errors(x.float(), off.float(), m.float(), go.float())
