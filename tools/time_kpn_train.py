"""KernelConv producer -> FAC block in training: forward + backward of the reference's op sequence (nn.Conv2d ->
nn.LeakyReLU -> KernelConv2D, torch defaults, i.e. cuDNN TF32) vs KernelPrediction(fused_backward=True) (fused
forward, fused backward kernel + cuDNN dgrad/wgrad of grad_pre). Workloads: the BASELINE cfg2 block (B=4, 64+64
channels, 256x256, K=5) and the cfg5 block shape (B=8, 128x128). Prints one JSON line per workload:
  *_fwd_bwd_ms      median of CUDA-event times over alternated repetitions, L2 flushed (512 MB write) before each
  bwd_breakdown_ms  the fused path's backward pieces, each timed alone the same way
  kpn_kernels_ms    device time per kernel of one fused backward call (torch.profiler)
  *_peak_mb         torch.cuda.max_memory_allocated over forward + backward, above what was allocated before
and the device name and power limit read in the same run.

--dtype bf16 / fp16 times the same two workloads in mixed precision: 16-bit event / frame tensors and fp32
parameters under torch.autocast with that dtype, the autocast op sequence (16-bit cuDNN conv, LeakyReLU and FAC)
against fused_backward=True (KernelConvFACBF16Function: 16-bit fused kernels + 16-bit cuDNN dgrad/wgrad of the 16-bit
grad_pre); the reference_* keys then hold the autocast sequence. --bf16 is short for --dtype bf16.

    python tools/time_kpn_train.py [--reps 15] [--dtype fp32|bf16|fp16]
"""
import argparse
import contextlib
import json
import os
import re
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebfi_be_b200 import modification  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--dtype", choices=("fp32", "bf16", "fp16"), default="fp32",
                    help="activation dtype; bf16 / fp16 run under torch.autocast (mixed precision)")
    ap.add_argument("--bf16", action="store_true", help="same as --dtype bf16")
    args = ap.parse_args()
    if args.bf16:
        args.dtype = "bf16"
    if not torch.cuda.is_available():
        raise SystemExit("time_kpn_train.py needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def timed_once(fn):
        flush.zero_()
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e)

    def median(ts):
        ts = sorted(ts)
        return ts[len(ts) // 2]

    info = device_info()
    act = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    half = act != torch.float32
    amp = (lambda: torch.autocast("cuda", dtype=act)) if half else contextlib.nullcontext
    for (B, H, W) in [(4, 256, 256), (8, 128, 128)]:
        C, K = 64, 5
        torch.manual_seed(0)
        m = modification.KernelPrediction(C, K).to(dev)
        conv = m.KernelConv.conv2d
        ev = torch.randn(B, C, H, W, device=dev).to(act).requires_grad_()
        fr = torch.randn(B, C, H, W, device=dev).to(act).requires_grad_()
        G = torch.randn(B, C, H, W, device=dev).to(act)

        def step(fused):
            m.fused_backward = fused
            ev.grad = fr.grad = None
            m.zero_grad(set_to_none=True)
            with amp():
                out = m(ev, fr)
            out.backward(G)

        for fused in (False, True, False, True):          # warm-up: cuDNN algorithm choice, module loads
            step(fused)
        ts = {False: [], True: []}
        for _ in range(args.reps):
            for fused in (False, True):
                ts[fused].append(timed_once(lambda: step(fused)))

        peak = {}
        for fused in (False, True):
            ev.grad = fr.grad = None
            m.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            step(fused)
            torch.cuda.synchronize()
            peak[fused] = (torch.cuda.max_memory_allocated() - base) / 2 ** 20

        # backward pieces of the fused path, each alone
        # (16-bit: the calls KernelConvFACBF16Function makes — 16-bit activations, fp32 weights for the fused kernels,
        # 16-bit weights for cuDNN's convolution backward)
        evd, frd, w, b = ev.detach(), fr.detach(), conv.weight.detach(), conv.bias.detach()
        x, wc = torch.cat([evd, frd], 1), w.to(act)
        fused_bwd = modification.kernelconv_fac_fused_backward_bf16 if half else \
            modification.kernelconv_fac_fused_backward
        gpre = fused_bwd(evd, frd, w, b, K, 0.01, G)[0]
        pieces = {
            "fused_forward": lambda: modification._fused_forward(evd, frd, w, b, K, 0.01),
            "kpn_fused_backward": lambda: fused_bwd(evd, frd, w, b, K, 0.01, G),
            "cudnn_dgrad": lambda: torch.ops.aten.convolution_backward(gpre, x, wc, None, [1, 1], [1, 1], [1, 1], False,
                                                                       [0, 0], 1, [True, False, False]),
            "cudnn_wgrad": lambda: torch.ops.aten.convolution_backward(gpre, x, wc, None, [1, 1], [1, 1], [1, 1], False,
                                                                       [0, 0], 1, [False, True, False]),
        }
        with torch.no_grad():
            for fn in pieces.values():
                fn()
            breakdown = {k: round(median([timed_once(fn) for _ in range(args.reps)]), 4) for k, fn in pieces.items()}
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                pieces["kpn_fused_backward"]()
                torch.cuda.synchronize()
        kernels = {}
        for ev_ in prof.events():
            if ev_.device_type == torch.autograd.DeviceType.CUDA and "kpn" in ev_.name:
                name = re.search(r"kpn_\w+", ev_.name).group(0)
                kernels[name] = round(kernels.get(name, 0.0) + ev_.device_time_total / 1e3, 4)
        del gpre, x

        res = {"workload": f"B={B} Ce=Cf={C} K={K} {H}x{W}",
               "precision": f"{args.dtype} activations, fp32 parameters, autocast" if half else "fp32",
               "reference_fwd_bwd_ms": round(median(ts[False]), 4), "fused_fwd_bwd_ms": round(median(ts[True]), 4),
               "bwd_breakdown_ms": breakdown, "kpn_kernels_ms": kernels,
               "reference_peak_mb": round(peak[False], 1), "fused_peak_mb": round(peak[True], 1),
               "reps": args.reps, "l2_flush": "512 MB write before each timed call"}
        res["speedup"] = round(res["reference_fwd_bwd_ms"] / res["fused_fwd_bwd_ms"], 3)
        res.update(info)
        print(json.dumps(res), flush=True)
        del m, ev, fr, G


if __name__ == "__main__":
    main()
