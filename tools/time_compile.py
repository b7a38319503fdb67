"""Eager vs torch.compile (default mode and reduce-overhead) on the blocks that call torch.ops.ebfi_b200, the graph
breaks torch._dynamo.explain reports for each, and the host cost of one call through torch.ops.ebfi_b200 against the
direct call (what the eager paths make).

    python tools/time_compile.py [--iters 50] [--only dcn_sep,kernelconv2d,kpn_fp32,kpn_bf16,frame_maps]

Prints one JSON line per measurement. Times are CUDA-event medians over --reps windows of --iters fwd+bwd steps."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ebfi_be_b200  # noqa: E402,F401
from ebfi_be_b200 import dcn_v2, frame_ops, kernelconv2d, modification  # noqa: E402
from ebfi_be_b200.shims import _ext  # noqa: E402

DEV = torch.device("cuda:0")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def rnd(*shape, scale=1.0, dtype=torch.float32):
    return (scale * torch.randn(*shape, device=DEV)).to(dtype)


def cases():
    """name -> (module, inputs, autocast dtype or None)."""
    def train(m):
        return m.to(DEV).train()

    dcn = train(dcn_v2.DCN_sep(64, 64, 3, 1, 1, deformable_groups=8))
    with torch.no_grad():
        dcn.conv_offset_mask.weight.normal_(0, 0.01)
    kpn = train(modification.KernelPrediction(64, 5))
    kpn.fused_backward = True

    class Maps(torch.nn.Module):
        def forward(self, ims):
            return frame_ops.Frame2Lap(ims), frame_ops.Frame2DCP(ims)

    return {
        "dcn_sep": (dcn, (rnd(1, 64, 256, 256).requires_grad_(), rnd(1, 64, 256, 256).requires_grad_()), None),
        "kernelconv2d": (kernelconv2d.KernelConv2D(5), (rnd(4, 64, 256, 256).requires_grad_(),
                                                        rnd(4, 1600, 256, 256, scale=0.1).requires_grad_()), None),
        "kpn_fp32": (kpn, (rnd(4, 64, 256, 256).requires_grad_(), rnd(4, 64, 256, 256).requires_grad_()), None),
        "kpn_bf16": (kpn, (rnd(4, 64, 256, 256, dtype=torch.bfloat16).requires_grad_(),
                           rnd(4, 64, 256, 256, dtype=torch.bfloat16).requires_grad_()), torch.bfloat16),
        "frame_maps": (Maps(), (torch.rand(1, 3, 720, 1280, device=DEV),), None),
    }


def step(fn, args, autocast):
    with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
        out = fn(*args)
    out = out if isinstance(out, tuple) else (out,)
    grads = [o for o in out if o.requires_grad]
    if grads:
        torch.autograd.backward(grads, [torch.ones_like(o) for o in grads])


def timed(fn, args, autocast, iters, reps):
    for _ in range(5):
        step(fn, args, autocast)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            step(fn, args, autocast)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b) / iters)
    return statistics.median(ms), min(ms), max(ms)


def host_cost(n=2000):
    """Per-call wall time of a tiny call (host-bound) through the direct path and through torch.ops.ebfi_b200."""
    x, w, b = rnd(1, 64, 8, 8), rnd(64, 64, 3, 3, scale=0.04), rnd(64)
    off, msk = rnd(1, 144, 8, 8, scale=0.5), torch.rand(1, 72, 8, 8, device=DEV)
    xi, ker = rnd(1, 8, 8, 8), rnd(1, 200, 8, 8)
    ims = torch.rand(1, 3, 8, 8, device=DEV)
    geom = (3, 3, 1, 1, 1, 1, 1, 1, 8)
    pairs = {
        "dcn_v2_forward": (lambda: _ext.dcn_v2_forward(x, w, b, off, msk, *geom),
                           lambda: torch.ops.ebfi_b200.dcn_v2_forward(x, w, b, off, msk, *geom)),
        "fac_replpad_forward": (lambda: kernelconv2d._replpad_forward(xi, ker, 5),
                                lambda: torch.ops.ebfi_b200.fac_replpad_forward(xi, ker, 5)),
        "frame_to_lap": (lambda: frame_ops.Frame2Lap(ims), lambda: torch.ops.ebfi_b200.frame_to_lap(ims)),
    }
    res = {}
    for name, fns in pairs.items():
        us = {}
        for _ in range(3):                        # alternate the two paths
            for label, fn in zip(("direct_us", "op_us"), fns):
                for _ in range(50):
                    fn()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(n):
                    fn()
                torch.cuda.synchronize()
                us.setdefault(label, []).append((time.perf_counter() - t0) / n * 1e6)
        res[name] = {k: round(min(v), 2) for k, v in us.items()}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_compile.py needs a CUDA device")
    print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
    print(json.dumps({"host_cost_per_call": host_cost()}), flush=True)
    for name, (mod, inp, autocast) in cases().items():
        if args.only and name not in args.only.split(","):
            continue
        torch._dynamo.reset()
        with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
            breaks = torch._dynamo.explain(mod)(*inp).graph_break_count
        row = {"case": name, "graph_breaks": breaks}
        for label, fn in (("eager", mod), ("compile_default", torch.compile(mod)),
                          ("compile_reduce_overhead", torch.compile(mod, mode="reduce-overhead"))):
            torch._dynamo.reset()
            med, lo, hi = timed(fn, inp, autocast, args.iters, args.reps)
            row[label + "_ms"] = [round(med, 4), round(lo, 4), round(hi, 4)]
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
