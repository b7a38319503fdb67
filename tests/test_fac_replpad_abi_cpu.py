"""CPU: the folded-pad FAC entries (ebfi_fac_replpad_*) validate their arguments before any CUDA call, and the
KernelConv2D module refuses CPU tensors as the reference does."""
import pytest
import torch

from ebfi_be_b200 import _lib as L

ENTRIES = ["ebfi_fac_replpad_forward", "ebfi_fac_replpad_forward_bf16", "ebfi_fac_replpad_forward_fp16",
           "ebfi_fac_replpad_backward", "ebfi_fac_replpad_backward_bf16", "ebfi_fac_replpad_backward_fp16"]


def _call(lib, name, K, null_at=None):
    fake = [L.c_void(256 * (i + 1)) for i in range(6)]     # never dereferenced: validation comes first
    if null_at is not None:
        fake[null_at] = None
    if "forward" in name:
        return getattr(lib, name)(None, *fake[:3], 1, 2, 8, 8, K)
    return getattr(lib, name)(None, *fake[:5], 1, 2, 8, 8, K, fake[5], 1 << 20)


@pytest.mark.parametrize("name", ENTRIES)
def test_null_pointers_and_even_k_return_invalid(name):
    lib = L.load()
    nptr = 3 if "forward" in name else 5
    for i in range(nptr):
        assert _call(lib, name, 5, null_at=i) == -1
        assert b"null" in lib.ebfi_last_error()
    assert _call(lib, name, 4) == -1
    assert b"odd" in lib.ebfi_last_error()
    assert _call(lib, name, 1, null_at=0) == -1          # K = 1 (no pad) validates the same way


def test_module_refuses_cpu_tensors_and_has_no_state():
    from ebfi_be_b200.kernelconv2d import KernelConv2D, KernelConv2DReplPadFunction
    m = KernelConv2D(5)
    assert m.state_dict() == {} and list(m.buffers()) == [] and list(m.parameters()) == []
    m.load_state_dict({})
    with pytest.raises(NotImplementedError):                         # KernelConv2D.py:38-39
        m(torch.randn(1, 2, 6, 6), torch.randn(1, 50, 6, 6))
    with pytest.raises(NotImplementedError):
        KernelConv2DReplPadFunction.apply(torch.randn(1, 2, 6, 6).bfloat16(), torch.randn(1, 50, 6, 6).bfloat16(), 5)
