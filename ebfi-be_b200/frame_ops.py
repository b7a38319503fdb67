"""Host-side mirror of the two per-frame maps of myutils/utils.py that the model evaluates in every forward
(models/Ours/model_singleframe.py:311-326): `Frame2DCP` (:15-31) and `Frame2Lap` (:34-49). Same names, arguments and
(B, 1, H, W) CUDA results — but the frames never leave the GPU (the reference does `.cpu().numpy()` per sample,
OpenCV on the host, `.cuda()` back: one device synchronisation per forward). Results are bit-identical to OpenCV's.
"""
import torch

from . import _lib as L


def _frames(ims):
    L.require_cuda(ims)
    if ims.dim() != 4 or ims.shape[1] != 3:
        raise RuntimeError(f"expected a (B, 3, H, W) tensor, got {tuple(ims.shape)}")
    return ims.float().contiguous()


def Frame2DCP(ims, sz=35):
    """Dark-channel prior map: min over channels, then a sz x sz minimum filter (cv2.erode). Bx3xHxW -> Bx1xHxW."""
    if torch.compiler.is_compiling():
        return torch.ops.ebfi_b200.frame_to_dcp(ims, int(sz))
    x = _frames(ims)
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        dark = torch.empty((B, 1, H, W), dtype=torch.float32, device=x.device)
        tmp = torch.empty((B, H, W), dtype=torch.float32, device=x.device)
        L.check(L.load().ebfi_frame_to_dcp(L.stream_ptr(x.device), L.ptr(x), L.ptr(dark), L.ptr(tmp), B, H, W, int(sz)),
                "Frame2DCP")
    return dark


def Frame2Lap(ims):
    """Laplacian of the 8-bit gray image (cv2.cvtColor BGR2GRAY + cv2.Laplacian). Bx3xHxW in [0, 1] -> Bx1xHxW."""
    if torch.compiler.is_compiling():
        return torch.ops.ebfi_b200.frame_to_lap(ims)
    x = _frames(ims)
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        lap = torch.empty((B, 1, H, W), dtype=torch.float32, device=x.device)
        L.check(L.load().ebfi_frame_to_lap(L.stream_ptr(x.device), L.ptr(x), L.ptr(lap), B, H, W), "Frame2Lap")
    return lap
