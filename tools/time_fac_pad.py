"""KernelConv2D forward + backward with the ReplicationPad2d folded into the FAC kernels (the module) against
the unfolded sequence nn.ReplicationPad2d + KernelConv2DFunction (padded copy, padded entries, ATen's pad backward).
Shapes: cfg2 (B=4, C=64, K=5, 256x256) and the cfg5 block (B=8, C=64, K=5, 128x128), fp32 / bf16 / fp16, forward +
backward; and the forward alone at the cfg4 FAC shape (B=1, C=64, K=5, 360x640, bf16). The two arms alternate in one
run; median of CUDA-event times, the L2 flushed (512 MB write) before each call; peak memory of one call above the
inputs; the device name and power limit are printed.

    python tools/time_fac_pad.py [--reps 20]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebfi_be_b200.kernelconv2d import KernelConv2D, KernelConv2DFunction  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
CASES = [("cfg2", (4, 64, 5, 256, 256), dt, True) for dt in DTYPES] + \
        [("cfg5", (8, 64, 5, 128, 128), dt, True) for dt in DTYPES] + \
        [("cfg4", (1, 64, 5, 360, 640), "bf16", False)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(torch.cuda.get_device_name(0), "|", q.stdout.strip(), flush=True)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        return (torch.cuda.max_memory_allocated() - base) / 1e6

    med = lambda v: sorted(v)[len(v) // 2]
    for name, (B, C, K, H, W), dname, backward in CASES:
        dt = DTYPES[dname]
        torch.manual_seed(0)
        x = torch.randn(B, C, H, W, device=dev).to(dt)
        ker = (0.1 * torch.randn(B, C * K * K, H, W, device=dev)).to(dt)
        go = torch.randn(B, C, H, W, device=dev).to(dt)
        pad = torch.nn.ReplicationPad2d((K - 1) // 2)
        folded = KernelConv2D(K)
        arms = {"pad+Function": lambda a, b: KernelConv2DFunction.apply(pad(a), b, K), "folded": folded}

        def step(fn):
            if not backward:
                return lambda: fn(x, ker)
            xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()

            def call():
                xg.grad = kg.grad = None         # no gradient accumulation in the timed window
                fn(xg, kg).backward(go)
            return call

        calls = {k: step(f) for k, f in arms.items()}
        for c in calls.values():
            c()
        outs = {}
        with torch.no_grad():
            for k, f in arms.items():
                outs[k] = f(x, ker)
        assert torch.equal(outs["pad+Function"], outs["folded"]), "forward differs"
        del outs
        ts = {k: [] for k in calls}
        for _ in range(args.reps):
            for k, c in calls.items():
                if backward:
                    ts[k].append(timed(c))
                else:
                    with torch.no_grad():
                        ts[k].append(timed(c))
        mems = {}
        for k, f in arms.items():
            if backward:
                xg, kg = x.clone().requires_grad_(), ker.clone().requires_grad_()
                mems[k] = peak(lambda: f(xg, kg).backward(go))
                del xg, kg
            else:
                with torch.no_grad():
                    mems[k] = peak(lambda: f(x, ker))
        what = "fwd+bwd" if backward else "fwd"
        t0, t1 = med(ts["pad+Function"]), med(ts["folded"])
        print(f"{name} {(B, C, K, H, W)} {dname:4s} {what:7s}  pad+Function {t0:.4f} ms  folded {t1:.4f} ms  "
              f"({(t1 / t0 - 1) * 100:+.1f} %)   peak MB {mems['pad+Function']:.1f} -> {mems['folded']:.1f}",
              flush=True)
        del x, ker, go, calls
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
