"""B200-native event-frame alignment kernels for EBFI-BE (drop-in for its custom ops).

Host side mirrors of the reference's operator interface, all calling the hand-written
sm_100a kernels in lib/libebfi_b200.so through the C ABI of include/ebfi_b200.h:

    ebfi_be_b200.dcn_v2        _DCNv2 / dcn_v2_conv / DCNv2 / DCN / DCN_sep
                               (reference: models/DCNv2/dcn_v2.py)
    ebfi_be_b200.kernelconv2d  KernelConv2DFunction / KernelConv2D
                               (reference: models/FAC/kernelconv2d/KernelConv2D.py)
    ebfi_be_b200.encodings     events_to_image / voxel / stack / channels / mask
                               (reference: dataloader/encodings.py)
    ebfi_be_b200.shims         modules named `_ext` and `kernelconv2d_cuda`, so the reference's
                               own, unmodified wrappers import and run on these kernels
    ebfi_be_b200.parallel      batch sharding + weight-gradient all-reduce helpers
    ebfi_be_b200.ops           the ops a model's forward and backward call, as torch custom operators
                               (torch.ops.ebfi_b200.*) for torch.compile and torch.export

There is no CPU fallback: every op raises if the CUDA library is missing or the tensors are
not on a CUDA device.
"""
from . import _lib  # noqa: F401
from . import ops  # noqa: F401  (registers torch.ops.ebfi_b200.*, which the modules call under torch.compile)

__all__ = ["_lib", "ops", "dcn_v2", "kernelconv2d", "encodings", "shims", "parallel", "install_shims"]


def install_shims():
    """Make `import _ext` and `import kernelconv2d_cuda` resolve to this package's kernels
    (what models/DCNv2/dcn_v2.py:13 and models/FAC/kernelconv2d/KernelConv2D.py:8 import)."""
    import sys
    from .shims import _ext, kernelconv2d_cuda
    sys.modules["_ext"] = _ext
    sys.modules["kernelconv2d_cuda"] = kernelconv2d_cuda
    return _ext, kernelconv2d_cuda


def __getattr__(name):
    if name in ("dcn_v2", "kernelconv2d", "encodings", "shims", "parallel"):
        import importlib
        return importlib.import_module("." + name, __name__)
    raise AttributeError(name)
