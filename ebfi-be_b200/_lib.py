"""ctypes binding of lib/libebfi_b200.so (the C ABI declared in include/ebfi_b200.h).

Loading is lazy and LOUD: the first op that needs the library raises RuntimeError with the
build command if it is missing — there is no fallback path.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EBFI_LIB_PATH") or os.path.join(_HERE, "lib", "libebfi_b200.so")   # override: A/B a debug build

EBFI_F32, EBFI_F64 = 0, 1
_lib = None

c_int, c_i64, c_size, c_void = ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_void_p


class DcnGeom(ctypes.Structure):
    """`ebfi_dcn_geom`."""
    _fields_ = [(n, c_int) for n in (
        "batch", "channels", "height", "width", "channels_out", "kernel_h", "kernel_w",
        "stride_h", "stride_w", "pad_h", "pad_w", "dilation_h", "dilation_w", "deformable_group", "flags")]


EBFI_DCN_DETERMINISTIC = 1
EBFI_DCN_INPUT_BLOCKED = 2
EBFI_ERR_UNSUPPORTED = -4


class DpComm(ctypes.Structure):
    """`ebfi_dp_comm`: peer mappings of the symmetric all-reduce buffers (parallel.GradComm fills it)."""
    _fields_ = [("world", c_int), ("rank", c_int), ("peer_base", c_void * 8), ("bytes", c_size)]


# name -> (restype, argtypes); must list every symbol include/ebfi_b200.h declares
_GEOM_P = ctypes.POINTER(DcnGeom)
SIGNATURES = {
    "ebfi_abi_version": (c_int, []),
    "ebfi_last_error": (ctypes.c_char_p, []),
    "ebfi_device_arch": (c_int, []),
    "ebfi_dcnv2_output_size": (c_int, [_GEOM_P, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "ebfi_dcnv2_backward_workspace_bytes": (c_size, [_GEOM_P]),
    "ebfi_dcnv2_forward_workspace_bytes": (c_size, [_GEOM_P]),
    "ebfi_dcnv2_blocked_input_offset": (c_size, [_GEOM_P]),
    "ebfi_dcnv2_forward": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size]),
    "ebfi_dcnv2_backward_dp": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size, ctypes.POINTER(DpComm), c_int]),
    "ebfi_dp_comm_bytes": (c_size, [c_size]),
    "ebfi_dp_allreduce_sum": (c_int, [c_void, ctypes.POINTER(DpComm), c_void, c_size, c_void, c_size]),
    "ebfi_dp_publish": (c_int, [c_void, ctypes.POINTER(DpComm), c_void, c_size, c_void, c_size]),
    "ebfi_dp_complete": (c_int, [c_void, ctypes.POINTER(DpComm), c_void, c_size, c_void, c_size]),
    "ebfi_dcnv2_forward_packed": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward_packed": (c_int, [c_void, _GEOM_P] + [c_void] * 9 + [c_void, c_size]),
    "ebfi_dcnv2_forward_bf16": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward_bf16": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size]),
    "ebfi_dcnv2_backward_dp_bf16": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size, ctypes.POINTER(DpComm), c_int]),
    "ebfi_dcnv2_forward_packed_bf16": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward_packed_bf16": (c_int, [c_void, _GEOM_P] + [c_void] * 9 + [c_void, c_size]),
    "ebfi_dcnv2_forward_fp16": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward_fp16": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size]),
    "ebfi_dcnv2_backward_dp_fp16": (c_int, [c_void, _GEOM_P] + [c_void] * 11 + [c_void, c_size, ctypes.POINTER(DpComm), c_int]),
    "ebfi_dcnv2_forward_packed_fp16": (c_int, [c_void, _GEOM_P] + [c_void] * 6 + [c_void, c_size]),
    "ebfi_dcnv2_backward_packed_fp16": (c_int, [c_void, _GEOM_P] + [c_void] * 9 + [c_void, c_size]),
    "ebfi_fac_forward": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_backward_workspace_bytes": (c_size, [c_int] * 5),
    "ebfi_fac_backward": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_fac_forward_bf16": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_backward_bf16": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_fac_forward_fp16": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_backward_fp16": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_fac_replpad_forward": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_replpad_backward": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_fac_replpad_forward_bf16": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_replpad_backward_bf16": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_fac_replpad_forward_fp16": (c_int, [c_void] * 4 + [c_int] * 5),
    "ebfi_fac_replpad_backward_fp16": (c_int, [c_void] * 6 + [c_int] * 5 + [c_void, c_size]),
    "ebfi_kpn_fused_workspace_bytes": (c_size, [c_int] * 6),
    "ebfi_kpn_fused_forward": (c_int, [c_void] * 5 + [ctypes.c_float, c_void] + [c_int] * 6 + [c_void, c_size]),
    "ebfi_kpn_fused_backward_workspace_bytes": (c_size, [c_int] * 6),
    "ebfi_kpn_fused_backward": (c_int, [c_void] * 5 + [ctypes.c_float] + [c_void] * 4 + [c_int] * 6 + [c_void, c_size]),
    "ebfi_kpn_fused_forward_bf16": (c_int, [c_void] * 5 + [ctypes.c_float, c_void] + [c_int] * 6 + [c_void, c_size]),
    "ebfi_kpn_fused_backward_bf16": (c_int, [c_void] * 5 + [ctypes.c_float] + [c_void] * 4 + [c_int] * 6 + [c_void, c_size]),
    "ebfi_kpn_fused_forward_fp16": (c_int, [c_void] * 5 + [ctypes.c_float, c_void] + [c_int] * 6 + [c_void, c_size]),
    "ebfi_kpn_fused_backward_fp16": (c_int, [c_void] * 5 + [ctypes.c_float] + [c_void] * 4 + [c_int] * 6 + [c_void, c_size]),
    "ebfi_events_to_image": (c_int, [c_void] * 4 + [c_int, c_i64, c_int, c_int, c_void, c_int]),
    "ebfi_events_to_mask": (c_int, [c_void] * 4 + [c_int, c_i64, c_int, c_int, c_void, c_void, c_int]),
    "ebfi_events_to_voxel": (c_int, [c_void] * 5 + [c_int, c_i64, c_int, c_int, c_int, c_void, c_int]),
    "ebfi_events_ts_sum_is_zero": (c_int, [c_void, c_void, c_int, c_i64, c_void, c_void]),
    "ebfi_events_to_stack": (c_int, [c_void] * 5 + [c_int, c_i64, c_int, c_int, c_int, c_void, c_void, c_int, c_void]),
    "ebfi_events_raw_to_stack": (c_int, [c_void] * 5 + [c_i64, c_int, c_int, c_int, c_void, c_void, c_int]),
    "ebfi_frame_to_lap": (c_int, [c_void] * 3 + [c_int] * 3),
    "ebfi_frame_to_dcp": (c_int, [c_void] * 4 + [c_int] * 4),
}
# test-only probes: lib/libebfi_b200_selftest.so, include/ebfi_b200_selftest.h
SELFTEST_LIB_PATH = os.path.join(os.path.dirname(LIB_PATH), "libebfi_b200_selftest.so")
SELFTEST_SIGNATURES = {
    "ebfi_selftest_gemm_tf32x3": (c_int, [c_void] * 4 + [c_int] * 4),
    "ebfi_selftest_gemm_bf16x3": (c_int, [c_void] * 4 + [c_int] * 4),
    "ebfi_selftest_mma_rate": (c_int, [c_void, c_void] + [c_int] * 6),
    "ebfi_selftest_umma_probe": (c_int, [c_void, c_void, c_int, c_int, c_int]),
}
_selftest = None


def load():
    """dlopen the kernel library and attach prototypes. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA kernels are not built and there is no fallback. "
            "Run `python ebfi-be_b200/build.py` (nvcc, sm_100a).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header/library mismatch
        fn.restype, fn.argtypes = res, args
    if lib.ebfi_abi_version() != 3:
        raise RuntimeError("libebfi_b200.so ABI version mismatch")
    _lib = lib
    return lib


def load_selftest():
    """dlopen the test-only probe library (after the product library it links against)."""
    global _selftest
    if _selftest is None:
        load()
        if not os.path.exists(SELFTEST_LIB_PATH):
            raise RuntimeError(f"{SELFTEST_LIB_PATH} is missing: run `python ebfi-be_b200/build.py`")
        lib = ctypes.CDLL(SELFTEST_LIB_PATH)
        for name, (res, args) in SELFTEST_SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _selftest = lib
    return _selftest


def check(rc, what):
    if rc != 0:
        msg = load().ebfi_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def stream_ptr(device):
    """cudaStream_t of torch's current stream on `device`, as the void* the C ABI takes."""
    return c_void(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return c_void(t.data_ptr())


def require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError("ebfi_be_b200 ops need CUDA tensors: there is no CPU path "
                               "(got a tensor on %s)" % t.device)


def require_f32(**named):
    for k, t in named.items():
        if t.dtype != torch.float32:
            raise RuntimeError(f"{k} must be float32 (the reference's `using scalar_t = float`), got {t.dtype}")
