"""torch.ops.ebfi_b200 on the GPU: opcheck of every op, zero graph breaks, compiled forward and gradients bit-equal
to eager (aot_eager, inductor, reduce-overhead), dynamic shapes, torch.export, and eager calls that stay off the ops.

Bit-equality needs eager to be reproducible itself: DCN offsets stay small enough that no sample leaves the backward's
staged box (far samples are accumulated with float atomics), and cuDNN runs its deterministic algorithms."""
import contextlib

import pytest
import torch

import ebfi_be_b200  # noqa: F401  (registers the ops)
from ebfi_be_b200 import dcn_v2, frame_ops, kernelconv2d, modification
from ebfi_be_b200.shims import _ext, kernelconv2d_cuda

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
DCN_INTS = (3, 3, 1, 1, 1, 1, 1, 1, 8)
OP_NAMES = ["dcn_v2_forward", "dcn_v2_backward", "dcn_v2_forward_packed", "dcn_v2_backward_packed", "fac_forward",
            "fac_backward", "fac_replpad_forward", "fac_replpad_backward", "kpn_fused_forward", "kpn_fused_backward",
            "frame_to_lap", "frame_to_dcp"]


def rnd(*shape, scale=1.0, dtype=F32, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (scale * torch.randn(*shape, generator=g)).to(dtype).to(DEV)


@contextlib.contextmanager
def deterministic(on):
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(old)


@pytest.fixture(autouse=True)
def _fresh_dynamo():
    torch._dynamo.reset()
    with torch.backends.cudnn.flags(enabled=True, deterministic=True, benchmark=False):
        yield
    torch._dynamo.reset()


# ------------------------------------------------------------------------------------------------------- opcheck
def _dcn_args(acts, param, seed=0):
    B, C, H, W, dg = 2, 64, 20, 24, 8
    x = rnd(B, C, H, W, dtype=acts, seed=seed)
    off, om = rnd(B, 144, H, W, scale=0.5, dtype=acts, seed=seed + 1), rnd(B, 216, H, W, scale=0.5, seed=seed + 2)
    msk = torch.sigmoid(rnd(B, 72, H, W, seed=seed + 3)).to(acts)
    w, b = rnd(64, C, 3, 3, scale=1 / 24, dtype=param, seed=seed + 4), rnd(64, dtype=param, seed=seed + 5)
    go = rnd(B, 64, H, W, dtype=acts, seed=seed + 6)
    return x, w, b, off, msk, om.to(acts), go


def _op_cases(dtype):
    """(op name, args) for every op at activation dtype `dtype`; DCN with fp32 parameters (autocast) too."""
    x, w, b, off, msk, om, go = _dcn_args(dtype, dtype)
    cases = [("dcn_v2_forward", (x, w, b, off, msk, *DCN_INTS)),
             ("dcn_v2_backward", (x, w, b, off, msk, go, *DCN_INTS)),
             ("dcn_v2_forward_packed", (x, w, b, om, *DCN_INTS, None)),
             ("dcn_v2_forward_packed", (x, w, b, om, *DCN_INTS, torch.zeros(1, device=DEV))),
             ("dcn_v2_backward_packed", (x, w, b, om, go, *DCN_INTS))]
    if dtype != F32:
        x, w, b, off, msk, om, go = _dcn_args(dtype, F32)
        cases += [("dcn_v2_forward", (x, w, b, off.float(), msk, *DCN_INTS)),
                  ("dcn_v2_backward", (x, w, b, off, msk.float(), go, *DCN_INTS)),
                  ("dcn_v2_backward_packed", (x, w, b, om.float(), go, *DCN_INTS))]
    for K in (1, 3, 5):
        B, C, H, W = 2, 4, 13, 9
        xp, x = rnd(B, C, H + K - 1, W + K - 1, dtype=dtype), rnd(B, C, H, W, dtype=dtype, seed=1)
        ker, go = rnd(B, C * K * K, H, W, scale=0.1, dtype=dtype, seed=2), rnd(B, C, H, W, dtype=dtype, seed=3)
        cases += [("fac_forward", (xp, ker, K, torch.empty_like(go))),
                  ("fac_backward", (xp, ker, K, go, torch.empty_like(xp), torch.empty_like(ker))),
                  ("fac_replpad_forward", (x, ker, K)),
                  ("fac_replpad_backward", (x, ker, K, go))]
    ev, fr = rnd(1, 32, 19, 13, dtype=dtype), rnd(1, 32, 19, 13, dtype=dtype, seed=1)
    wk, bk = rnd(800, 64, 3, 3, scale=0.05, seed=2), rnd(800, scale=0.1, seed=3)
    cases += [("kpn_fused_forward", (ev, fr, wk, bk, 5, 0.01)),
              ("kpn_fused_backward", (ev, fr, wk, bk, 5, 0.01, rnd(1, 32, 19, 13, dtype=dtype, seed=4)))]
    ims = torch.rand(2, 3, 37, 29, device=DEV).to(dtype)
    cases += [("frame_to_lap", (ims,)), ("frame_to_dcp", (ims, 35)), ("frame_to_dcp", (ims, 7))]
    return cases


@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
def test_opcheck(dtype, det):
    cases = _op_cases(dtype)
    assert {name for name, _ in cases} == set(OP_NAMES)
    with deterministic(det):
        for name, args in cases:
            torch.library.opcheck(getattr(torch.ops.ebfi_b200, name).default, args)


# ------------------------------------------------------------------------------------------- modules under compile
class _Maps(torch.nn.Module):
    def forward(self, ims):
        return frame_ops.Frame2Lap(ims), frame_ops.Frame2DCP(ims)


class _Padded(torch.nn.Module):
    def forward(self, x, kernel):
        return kernelconv2d.KernelConv2DFunction.apply(x, kernel, 5)


def _randomize(mod):
    with torch.no_grad():
        for i, p in enumerate(mod.parameters()):
            p.copy_(rnd(*p.shape, scale=0.02, seed=100 + i))
    return mod


def _case(name, half=None, train=True):
    """(module, inputs). `half`: the dtype activations arrive in under autocast, for the blocks that take them
    as they are (the DCNs get fp32 inputs and mix them with autocast's 16-bit conv output)."""
    act = half or F32
    g = dict(requires_grad=train)
    if name == "DCNv2":
        m = dcn_v2.DCNv2(64, 64, 3, 1, 1, deformable_groups=8)
        args = (rnd(2, 64, 20, 24), rnd(2, 144, 20, 24, scale=0.5, seed=1), torch.sigmoid(rnd(2, 72, 20, 24, seed=2)))
    elif name in ("DCN", "DCN_sep"):
        m = _randomize(getattr(dcn_v2, name)(64, 64, 3, 1, 1, deformable_groups=8))
        args = (rnd(2, 64, 20, 24),) + ((rnd(2, 64, 20, 24, seed=1),) if name == "DCN_sep" else ())
    elif name == "KernelConv2D":
        m = kernelconv2d.KernelConv2D(5)
        args = (rnd(2, 8, 24, 20, dtype=act), rnd(2, 200, 24, 20, scale=0.1, dtype=act, seed=1))
    elif name == "KernelConv2DFunction":
        m = _Padded()
        args = (rnd(2, 8, 28, 24, dtype=act), rnd(2, 200, 24, 20, scale=0.1, dtype=act, seed=1))
    elif name == "KernelPrediction":
        m = _randomize(modification.KernelPrediction(32, 5))
        m.fused_backward = True
        args = (rnd(2, 32, 24, 20, dtype=act), rnd(2, 32, 24, 20, dtype=act, seed=1))
    else:
        m, args = _Maps(), (torch.rand(2, 3, 40, 36, device=DEV),)
        g = dict(requires_grad=False)
    m = m.to(DEV).requires_grad_(train)
    return m, tuple(a.detach().requires_grad_(g["requires_grad"] and a.is_floating_point()) for a in args)


MODULES = ["DCNv2", "DCN", "DCN_sep", "KernelConv2D", "KernelConv2DFunction", "KernelPrediction", "Maps"]


def _step(fn, mod, args, autocast=None):
    """Outputs, then the gradients of every input and parameter that needs one, of sum(out * fixed weights)."""
    for t in (*args, *mod.parameters()):
        t.grad = None
    with torch.autocast("cuda", dtype=autocast) if autocast else contextlib.nullcontext():
        outs = fn(*args)
    outs = outs if isinstance(outs, tuple) else (outs,)
    res = [o.detach().clone() for o in outs]
    if any(o.requires_grad for o in outs):
        loss = sum((o.float() * rnd(*o.shape, seed=7 + i)).sum() for i, o in enumerate(outs))
        loss.backward()
        res += [t.grad.clone() for t in (*args, *mod.parameters()) if t.grad is not None]
        assert len(res) > len(outs)
    return res


def _assert_equal(got, want):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.dtype == b.dtype and a.shape == b.shape, (i, a.dtype, b.dtype, a.shape, b.shape)
        assert torch.equal(a, b), (i, (a.double() - b.double()).abs().max().item())


@pytest.mark.parametrize("name", MODULES)
def test_no_graph_breaks(name):
    m, args = _case(name)
    assert torch._dynamo.explain(m)(*args).graph_break_count == 0
    if name == "KernelPrediction":          # eval: the fused inference kernel
        m, args = _case(name, train=False)
        torch._dynamo.reset()
        ex = torch._dynamo.explain(m.eval())(*args)
        assert ex.graph_break_count == 0
        assert "kpn_fused_forward" in str(ex.graphs[0].graph)


MODES = {"fp32": dict(), "bf16_autocast": dict(half=BF16), "fp16_autocast": dict(half=F16),
         "deterministic": dict(det=True)}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("name", MODULES)
def test_aot_eager_fullgraph_bit_equal(name, mode):
    half, det = MODES[mode].get("half"), MODES[mode].get("det", False)
    m, args = _case(name, half)
    compiled = torch.compile(m, backend="aot_eager", fullgraph=True)
    with deterministic(det):
        want = _step(m, m, args, half)
        _assert_equal(_step(m, m, args, half), want)      # eager reproduces itself
        _assert_equal(_step(compiled, m, args, half), want)


def test_inductor_ops_bit_equal():
    x, w, b, off, msk, om, go = _dcn_args(F32, F32)
    xp, ker = rnd(2, 8, 28, 24), rnd(2, 200, 24, 20, scale=0.1, seed=1)
    xi, gf = rnd(2, 8, 24, 20, seed=2), rnd(2, 8, 24, 20, seed=3)
    ims = torch.rand(2, 3, 40, 36, device=DEV)
    ev, fr = rnd(1, 32, 19, 13), rnd(1, 32, 19, 13, seed=1)
    wk, bk = rnd(800, 64, 3, 3, scale=0.05, seed=2), rnd(800, scale=0.1, seed=3)

    def calls():
        out = [_ext.dcn_v2_forward(x, w, b, off, msk, *DCN_INTS),
               *_ext.dcn_v2_backward(x, w, b, off, msk, go, *DCN_INTS),
               _ext.dcn_v2_forward_packed(x, w, b, om, *DCN_INTS),
               *_ext.dcn_v2_backward_packed(x, w, b, om, go, *DCN_INTS),
               kernelconv2d.KernelConv2D(5)(xi, ker),
               frame_ops.Frame2Lap(ims), frame_ops.Frame2DCP(ims),
               modification._fused_forward(ev, fr, wk, bk, 5, 0.01),
               *modification._fused_backward(ev, fr, wk, bk, 5, 0.01, ev * 0.5, "kpn")]
        o = torch.empty(2, 8, 24, 20, device=DEV)
        gi, gk = torch.empty_like(xp), torch.empty_like(ker)
        kernelconv2d_cuda.forward(xp, ker, 5, o)
        kernelconv2d_cuda.backward(xp, ker, 5, gf, gi, gk)
        return out + [o, gi, gk]

    want = calls()
    got = torch.compile(calls, backend="inductor", fullgraph=True)()
    _assert_equal([t.clone() for t in got], want)


def _assert_close(got, want):
    """The parity gates of the fp32 tests: forward 1e-5, gradients 1e-4 of max |reference|."""
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        err = ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()
        assert err <= (1e-5 if i == 0 else 1e-4), (i, err)


# Inductor runs the modules' own convolutions with cuDNN algorithms of its choice: with TF32 those differ from eager by
# ~5e-5 of max |out| (measured on DCN_sep's offset conv), so these comparisons run the convolutions in fp32.
@pytest.mark.parametrize("name", ["DCN_sep", "KernelConv2D", "KernelPrediction"])
def test_inductor_modules_within_tolerance(name):
    m, args = _case(name)
    with torch.backends.cudnn.flags(enabled=True, deterministic=True, benchmark=False, allow_tf32=False):
        want = _step(m, m, args)
        _assert_close(_step(torch.compile(m, backend="inductor", fullgraph=True), m, args), want)


def test_dynamic_shapes_one_compile():
    from torch._dynamo.testing import CompileCounterWithBackend
    m, _ = _case("DCN_sep")
    cnt = CompileCounterWithBackend("aot_eager")
    compiled = torch.compile(m, backend=cnt, dynamic=True, fullgraph=True)
    for H, W in ((20, 24), (33, 17)):
        args = tuple(rnd(2, 64, H, W, seed=s).requires_grad_() for s in (0, 1))
        want = _step(m, m, args)
        got = _step(compiled, m, args)
        assert got[0].shape == (2, 64, H, W)
        _assert_equal(got, want)
    assert cnt.frame_count == 1


@pytest.mark.parametrize("name", ["DCN_sep", "KernelPrediction", "Maps"])
def test_export(name):
    m, args = _case(name, train=False)
    m.eval()
    ep = torch.export.export(m, args)
    targets = {str(n.target) for n in ep.graph.nodes if n.op == "call_function"}
    assert any(t.startswith("ebfi_b200.") for t in targets), targets
    with torch.no_grad():
        want = m(*args)
        got = ep.module()(*args)
    _assert_equal(got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,))


class _Train(torch.nn.Module):
    """DCNv2 (offsets and masks as inputs) or DCN_sep, then KernelConv2D(5) on its output."""

    def __init__(self, sep):
        super().__init__()
        self.dcn = _randomize((dcn_v2.DCN_sep if sep else dcn_v2.DCNv2)(64, 64, 3, 1, 1, deformable_groups=8))
        self.kpn = kernelconv2d.KernelConv2D(5)

    def forward(self, x, *rest):
        *dcn_in, kernel = rest
        return self.kpn(self.dcn(x, *dcn_in), kernel)


@pytest.mark.parametrize("sep", [False, True], ids=["DCNv2", "DCN_sep"])
def test_reduce_overhead_training_steps(sep):
    """CUDA-graph replays of fwd + bwd on changing inputs. Only our ops: bit-equal to eager. With DCN_sep's offset
    conv, which inductor runs on its own cuDNN algorithm: within the fp32 gates (TF32 off, as above)."""
    m = _Train(sep).to(DEV)
    compiled = torch.compile(m, mode="reduce-overhead", fullgraph=True)
    with torch.backends.cudnn.flags(enabled=True, deterministic=True, benchmark=False, allow_tf32=False):
        for step in range(4):
            s = 10 * step
            dcn_in = ((rnd(1, 64, 24, 20, seed=s + 1),) if sep else
                      (rnd(1, 144, 24, 20, scale=0.5, seed=s + 1), torch.sigmoid(rnd(1, 72, 24, 20, seed=s + 3))))
            args = (rnd(1, 64, 24, 20, seed=s).requires_grad_(), *(t.requires_grad_() for t in dcn_in),
                    rnd(1, 1600, 24, 20, scale=0.1, seed=s + 2).requires_grad_())
            want = _step(m, m, args)
            (_assert_close if sep else _assert_equal)(_step(compiled, m, args), want)


def test_eager_calls_do_not_dispatch_through_the_ops(monkeypatch):
    def boom(*args, **kwargs):
        raise AssertionError("an eager call went through torch.ops.ebfi_b200")
    for name in OP_NAMES:
        getattr(torch.ops.ebfi_b200, name)
        monkeypatch.setattr(torch.ops.ebfi_b200, name, boom)
    for name in MODULES:
        m, args = _case(name)
        _step(m, m, args)
        _step(m, m, args, BF16)
    m, args = _case("KernelPrediction", train=False)
    with torch.no_grad():
        m.eval()(*args)
    x, w, b, off, msk, om, go = _dcn_args(F32, F32)
    _ext.dcn_v2_backward(x, w, b, off, msk, go, *DCN_INTS)
    _ext.dcn_v2_backward_packed(x, w, b, om, go, *DCN_INTS)
