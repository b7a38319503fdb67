"""FAC KernelConv2D forward and backward at BASELINE cfg2 (B=4, C=64, K=5, 256x256) per storage dtype, with the
HBM bytes each call moves. A 16-bit dtype is timed twice, alternated with the others: native (its own entries) and
convert (widen to fp32, fp32 kernels, round the results: what a 16-bit call costs without native 16-bit I/O).
Median of CUDA-event times, the L2 flushed (512 MB write) before each; the device name and power limit are printed.

    python tools/time_fac_dtypes.py [--dtypes fp32,bf16,fp16] [--reps 10]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebfi_be_b200.shims import kernelconv2d_cuda as kc  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtypes", default="fp32,bf16")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(torch.cuda.get_device_name(0), "|", q.stdout.strip())
    B, C, K, H, W = 4, 64, 5, 256, 256
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)
    x32 = torch.randn(B, C, H + 4, W + 4, device=dev)
    ker32 = torch.randn(B, C * 25, H, W, device=dev)
    go32 = torch.randn(B, C, H, W, device=dev)

    def fac_fwd(x, ker):
        out = torch.empty(B, C, H, W, device=dev, dtype=x.dtype)
        kc.forward(x, ker, K, out)
        return out

    def fac_bwd(x, ker, go):
        gi, gk = torch.empty_like(x), torch.empty_like(ker)
        kc.backward(x, ker, K, go, gi, gk)
        return gi, gk

    arms = {}
    for name in args.dtypes.split(","):
        dt = DTYPES[name]
        x, ker, go = x32.to(dt), ker32.to(dt), go32.to(dt)
        arms[name] = (lambda x=x, ker=ker: fac_fwd(x, ker), lambda x=x, ker=ker, go=go: fac_bwd(x, ker, go),
                      x.element_size())
        if dt != torch.float32:
            arms[name + "_convert"] = (lambda x=x, ker=ker, dt=dt: fac_fwd(x.float(), ker.float()).to(dt),
                                       lambda x=x, ker=ker, go=go, dt=dt: [g.to(dt) for g in
                                                                          fac_bwd(x.float(), ker.float(), go.float())],
                                       None)

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    for f, b_, _ in arms.values():          # warm-up
        f(), b_()
    ts = {k: ([], []) for k in arms}
    for _ in range(args.reps):
        for k, (f, b_, _) in arms.items():
            ts[k][0].append(timed(f))
            ts[k][1].append(timed(b_))
    med = lambda v: sorted(v)[len(v) // 2]
    for k, (f, b_, es) in arms.items():
        tf, tb = med(ts[k][0]), med(ts[k][1])
        line = f"{k:13s} fwd {tf:.4f} ms   bwd {tb:.4f} ms   fwd+bwd {tf + tb:.4f} ms"
        if es:
            fb = es * (x32.numel() + ker32.numel() + go32.numel())
            bb = es * (2 * ker32.numel() + go32.numel() + 2 * x32.numel())
            line += f"   ({fb / tf / 1e6:.0f} / {bb / tb / 1e6:.0f} GB/s)"
        print(line, flush=True)


if __name__ == "__main__":
    main()
