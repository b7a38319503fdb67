"""CPU: the float64 backward restatement of the KernelConv -> FAC block (tests/kpn_train_oracle.py) against torch's
float64 autograd of the literal op sequence, and the host side of ebfi_kpn_fused_backward (no kernel launched)."""
import numpy as np
import pytest
import torch

import kpn_train_oracle as KO
from ebfi_be_b200 import _lib as L


@pytest.mark.parametrize("shape", [(2, 4, 4, 7, 6, 5), (1, 3, 5, 5, 9, 3), (1, 2, 0, 4, 5, 1), (1, 2, 2, 1, 3, 5)])
def test_kpn_backward_oracle_matches_torch_op_sequence(shape):
    """Conv2d -> LeakyReLU -> ReplicationPad2d -> unfold contraction (KernelConv2D's math), float64 autograd."""
    B, Ce, Cf, H, W, K = shape
    rng = np.random.default_rng(sum(shape))
    ev = rng.standard_normal((B, Ce, H, W)).astype(np.float32)
    fr = rng.standard_normal((B, Cf, H, W)).astype(np.float32)
    w = (0.3 * rng.standard_normal((Ce * K * K, Ce + Cf, 3, 3))).astype(np.float32)
    b = (0.1 * rng.standard_normal(Ce * K * K)).astype(np.float32)
    G = rng.standard_normal((B, Ce, H, W))
    slope = 0.01
    got = KO.kpn_fused_backward(ev, fr, w, b, K, slope, G)

    tev, tfr, tw, tb = (torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (ev, fr, w, b))
    R = (K - 1) // 2
    P = torch.nn.functional.conv2d(torch.cat([tev, tfr], 1), tw, tb, padding=1)
    P.retain_grad()
    Kt = torch.nn.functional.leaky_relu(P, slope)
    evp = torch.nn.ReplicationPad2d(R)(tev)
    cols = torch.nn.functional.unfold(evp, K).reshape(B, Ce, K * K, H, W)
    out = (cols * Kt.reshape(B, Ce, K * K, H, W)).sum(2)
    out.backward(torch.tensor(G))
    want = (tev.grad, tfr.grad, tw.grad, tb.grad, P.grad, P.detach())
    for name, g, t in zip(("grad_event", "grad_frame", "grad_weight", "grad_bias", "grad_pre", "P"), got, want):
        t = t.numpy()
        assert g.shape == t.shape, name
        if t.size:
            assert np.abs(g - t).max() <= 1e-12 * max(np.abs(t).max(), 1.0), name


def test_backward_workspace_query_without_a_gpu():
    lib = L.load()
    assert lib.ebfi_kpn_fused_backward_workspace_bytes(4, 64, 64, 256, 256, 5) > \
        lib.ebfi_kpn_fused_workspace_bytes(4, 64, 64, 256, 256, 5)
    assert lib.ebfi_kpn_fused_backward_workspace_bytes(1, 24, 24, 8, 8, 5) == 0       # Cin = 48: unsupported
    assert lib.ebfi_kpn_fused_backward_workspace_bytes(1, 32, 32, 8, 8, 7) == 0       # K = 7


def test_backward_null_pointers_return_invalid_without_a_gpu():
    lib = L.load()
    assert lib.ebfi_kpn_fused_backward(None, None, None, None, None, 0.01, None, None, None, None,
                                       1, 32, 32, 8, 8, 5, None, 0) == -1
    assert b"null pointer" in lib.ebfi_last_error()
    assert lib.ebfi_kpn_fused_backward(None, None, None, None, None, 0.01, None, None, None, None,
                                       1, 24, 24, 8, 8, 5, None, 0) == -4           # EBFI_ERR_UNSUPPORTED
    assert b"multiple of 32" in lib.ebfi_last_error()


def test_function_refuses_cpu_tensors():
    from ebfi_be_b200 import modification
    ev, fr = torch.randn(1, 32, 8, 8), torch.randn(1, 32, 8, 8)
    w, b = torch.randn(800, 64, 3, 3, requires_grad=True), torch.zeros(800, requires_grad=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        modification.KernelConvFACFunction.apply(ev, fr, w, b, 5, 0.01)
    with pytest.raises(RuntimeError, match="no CPU path"):
        modification.kernelconv_fac_fused_backward(ev, fr, w, b, 5, 0.01, torch.randn(1, 32, 8, 8))


def test_module_on_cpu_keeps_the_reference_sequence():
    """fused_backward only affects CUDA tensors: on the CPU the module runs the reference's op sequence, whose FAC
    refuses the CPU as the reference does (KernelConv2D.py:38-39)."""
    from ebfi_be_b200 import modification
    m = modification.KernelPrediction(32, 5)
    m.fused_backward = True
    with pytest.raises(NotImplementedError):
        m(torch.randn(1, 32, 8, 8), torch.randn(1, 32, 8, 8))
