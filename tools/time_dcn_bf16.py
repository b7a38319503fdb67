"""DCNv2 with 16-bit activations at BASELINE cfg1 (B=1, C=64 -> 64, 3x3, dg=8, 256x256). Arms, same inputs:
  fp32          fp32 activations and parameters: the fp32 kernels
  <dt>_convert  16-bit activations, fp32 parameters, through the boundary conversion (_ext._via_fp32, the path every
                16-bit call takes where the kernels have no native 16-bit I/O): widen, fp32 kernels, round the results
  <dt>_native   the same 16-bit call through the shim: the *_bf16 / *_fp16 entries of the tensor-core kernels
with <dt> each of --dtypes (bf16, fp16), for the plain entries (offset, mask) and the packed ones (DCN_sep's raw
conv_offset_mask output), each timed as forward, backward and forward + backward. The backward alone runs after an
untimed forward of the same arm, as in training, so the native arms read the forward's blocked input copy. Then the DCN_sep module (offset conv included) forward +
backward under torch.autocast with each dtype against the same module in fp32, with the memory kept from forward to
backward and the peak.

Times: median of CUDA-event times over alternated repetitions, the L2 flushed (512 MB write) before each. The device
name and power limit are read in the same run. Prints one JSON line per table.

    python tools/time_dcn_bf16.py [--reps 25] [--dtypes bf16,fp16]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebfi_be_b200 import dcn_v2  # noqa: E402
from ebfi_be_b200.shims import _ext  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--dtypes", default="bf16", help="comma-separated 16-bit activation dtypes: bf16, fp16")
    args = ap.parse_args()
    dts = {"bf16": torch.bfloat16, "fp16": torch.float16}
    halves = {k: dts[k] for k in args.dtypes.split(",")}
    if not torch.cuda.is_available():
        raise SystemExit("time_dcn_bf16.py needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def timed_once(fn, prep=None):
        if prep is not None:
            prep()
        flush.zero_()
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e)

    def alternated(fns, prep=None):
        for fn in fns.values():            # warm-up: module loads, allocator
            fn(); fn()
        ts = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, fn in fns.items():
                ts[k].append(timed_once(fn, prep[k] if prep else None))
        return {k: round(sorted(v)[len(v) // 2], 4) for k, v in ts.items()}

    info = device_info()
    B, C, H, W, dg = 1, 64, 256, 256, 8
    ints = (3, 3, 1, 1, 1, 1, 1, 1, dg)
    torch.manual_seed(0)
    x = torch.randn(B, C, H, W, device=dev)
    off = 2 * torch.randn(B, 2 * dg * 9, H, W, device=dev)
    mask = torch.sigmoid(torch.randn(B, dg * 9, H, W, device=dev))
    om = torch.cat([off, torch.randn(B, dg * 9, H, W, device=dev)], 1)
    w = torch.randn(C, C, 3, 3, device=dev) / 24
    b = torch.randn(C, device=dev)
    go = torch.randn(B, C, H, W, device=dev)
    f32 = torch.float32

    for layout in ("plain", "packed"):
        if layout == "plain":
            fwd, bwd = _ext.dcn_v2_forward, _ext.dcn_v2_backward
            acts32 = (x, off, mask)
            call_f = lambda f, a: f(a[0], w, b, *a[1:], *ints)
            call_b = lambda f, a, g: f(a[0], w, b, *a[1:], g, *ints)
            conv_f = lambda dt, a: _ext._via_fp32(dt, fwd, (a[0], w, b, *a[1:]), ints)
            conv_b = lambda dt, a, g: _ext._via_fp32(dt, bwd, (a[0], w, b, *a[1:], g), ints, [dt] * 3 + [f32, f32])
        else:
            fwd, bwd = _ext.dcn_v2_forward_packed, _ext.dcn_v2_backward_packed
            acts32 = (x, om)
            call_f = lambda f, a: f(a[0], w, b, a[1], *ints)
            call_b = lambda f, a, g: f(a[0], w, b, a[1], g, *ints)
            conv_f = lambda dt, a: _ext._via_fp32(dt, fwd, (a[0], w, b, a[1]), ints)
            conv_b = lambda dt, a, g: _ext._via_fp32(dt, bwd, (a[0], w, b, a[1], g), ints, [dt] * 2 + [f32, f32])
        arms_f, arms_b = {"fp32": lambda: call_f(fwd, acts32)}, {"fp32": lambda: call_b(bwd, acts32, go)}
        for name, dt in halves.items():
            acts16, go16 = [t.to(dt) for t in acts32], go.to(dt)
            arms_f[name + "_convert"] = lambda dt=dt, a=acts16: conv_f(dt, a)
            arms_f[name + "_native"] = lambda a=acts16: call_f(fwd, a)
            arms_b[name + "_convert"] = lambda dt=dt, a=acts16, g=go16: conv_b(dt, a, g)
            arms_b[name + "_native"] = lambda a=acts16, g=go16: call_b(bwd, a, g)
        arms_fb = {k: (lambda k=k: (arms_f[k](), arms_b[k]())) for k in arms_f}
        res = {"table": f"DCNv2 {layout} entries, cfg1 (B=1, 64->64, 3x3, dg=8, 256x256)", **info,
               "reps": args.reps, "l2_flush": "512 MB write before each timed call"}
        res["fwd_ms"] = alternated(arms_f)
        # the backward alone follows a forward of its input, as in training (the native arms then read the forward's
        # blocked input copy); the forward is not timed
        res["bwd_ms"] = alternated(arms_b, prep=arms_f)
        res["fwd_bwd_ms"] = alternated(arms_fb)
        print(json.dumps(res), flush=True)

    # ---- the DCN_sep module (offset conv + packed kernels) under autocast vs fp32
    torch.manual_seed(1)
    m = dcn_v2.DCN_sep(C, C, 3, 1, 1, deformable_groups=dg).to(dev)
    with torch.no_grad():
        m.conv_offset_mask.weight.normal_(0, 0.02)
    xm = torch.randn(B, C, H, W, device=dev).requires_grad_()
    fea = torch.randn(B, C, H, W, device=dev).requires_grad_()
    mem = {}

    def step(dtype, record=None):
        m.zero_grad(set_to_none=True)
        xm.grad = fea.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with torch.autocast("cuda", dtype=dtype or torch.bfloat16, enabled=dtype is not None):
            out = m(xm, fea)
        kept = torch.cuda.memory_allocated() - base
        out.backward(go.to(out.dtype))
        if record is not None:
            torch.cuda.synchronize()
            mem[record] = {"kept_fwd_to_bwd_mb": round(kept / 2 ** 20, 1),
                           "peak_mb": round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)}

    step(None, "fp32")
    for name, dt in halves.items():
        step(dt, "autocast_" + name)
    arms = {"fp32": lambda: step(None)}
    arms.update({"autocast_" + name: (lambda dt=dt: step(dt)) for name, dt in halves.items()})
    res = {"table": "DCN_sep module (offset conv + DCNv2) fwd+bwd, cfg1, autocast vs fp32, fp32 inputs", **info,
           "reps": args.reps, "l2_flush": "512 MB write before each timed call",
           "fwd_bwd_ms": alternated(arms), "memory": mem}
    m.flush_offset_warnings()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
