"""KernelConv producer -> FAC block in training: forward + backward of the reference's op sequence (nn.Conv2d ->
nn.LeakyReLU -> KernelConv2D, torch defaults, i.e. cuDNN TF32) vs KernelPrediction(fused_backward=True) (fused
forward, fused backward kernel + cuDNN dgrad/wgrad of grad_pre). Workloads: the BASELINE cfg2 block (B=4, 64+64
channels, 256x256, K=5) and the cfg5 block shape (B=8, 128x128). Prints one JSON line per workload:
  *_fwd_bwd_ms      median of CUDA-event times over alternated repetitions, L2 flushed (512 MB write) before each
  bwd_breakdown_ms  the fused path's backward pieces, each timed alone the same way
  kpn_kernels_ms    device time per kernel of one fused backward call (torch.profiler)
  *_peak_mb         torch.cuda.max_memory_allocated over forward + backward, above what was allocated before
and the device name and power limit read in the same run.

    python tools/time_kpn_train.py [--reps 15]
"""
import argparse
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
    args = ap.parse_args()
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
    for (B, H, W) in [(4, 256, 256), (8, 128, 128)]:
        C, K = 64, 5
        torch.manual_seed(0)
        m = modification.KernelPrediction(C, K).to(dev)
        conv = m.KernelConv.conv2d
        ev = torch.randn(B, C, H, W, device=dev, requires_grad=True)
        fr = torch.randn(B, C, H, W, device=dev, requires_grad=True)
        G = torch.randn(B, C, H, W, device=dev)

        def step(fused):
            m.fused_backward = fused
            ev.grad = fr.grad = None
            m.zero_grad(set_to_none=True)
            m(ev, fr).backward(G)

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
        evd, frd, w, b = ev.detach(), fr.detach(), conv.weight.detach(), conv.bias.detach()
        x = torch.cat([evd, frd], 1)
        gpre = modification.kernelconv_fac_fused_backward(evd, frd, w, b, K, 0.01, G)[0]
        pieces = {
            "fused_forward": lambda: modification.kernelconv_fac_fused(evd, frd, w, b, K, 0.01),
            "kpn_fused_backward": lambda: modification.kernelconv_fac_fused_backward(evd, frd, w, b, K, 0.01, G),
            "cudnn_dgrad": lambda: torch.ops.aten.convolution_backward(gpre, x, w, None, [1, 1], [1, 1], [1, 1], False,
                                                                       [0, 0], 1, [True, False, False]),
            "cudnn_wgrad": lambda: torch.ops.aten.convolution_backward(gpre, x, w, None, [1, 1], [1, 1], [1, 1], False,
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
