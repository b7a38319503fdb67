"""DCNv2 backward: default mode vs EBFI_DCN_DETERMINISTIC on the box kernel vs EBFI_DCN_DETERMINISTIC with
EBFI_DCN_BWD_NO_BOX=1 (the deterministic path before the box kernel covered it: dcn_bwd_tc.cu for 8 channels per
group, the CUDA-core kernel otherwise; 16-bit calls convert at the boundary there).

Arms alternate call by call, the L2 is overwritten before each call, medians of CUDA-event times.
    python tools/time_dcn_det.py [--iters 30]"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebfi_be_b200.shims import _ext  # noqa: E402

ARMS = {"default": {}, "det_box": {"EBFI_DCN_DETERMINISTIC": "1"},
        "det_no_box": {"EBFI_DCN_DETERMINISTIC": "1", "EBFI_DCN_BWD_NO_BOX": "1"}}
ENV_KEYS = ("EBFI_DCN_DETERMINISTIC", "EBFI_DCN_BWD_NO_BOX")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                       # noqa: BLE001 - informational only
        return f"{torch.cuda.get_device_name(0)} (power limit unavailable: {e})"


def case(dev, dg, sigma, dtype, packed, seed=0):
    """cfg1 geometry (1 x 64 x 256 x 256 -> 64, 3x3, pad 1) with dg deformable groups, offsets sigma * randn."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(1, 64, 256, 256, generator=g)
    w = torch.randn(64, 64, 3, 3, generator=g) / 24
    b = torch.randn(64, generator=g)
    off = sigma * torch.randn(1, 2 * dg * 9, 256, 256, generator=g)
    m = torch.randn(1, dg * 9, 256, 256, generator=g)
    go = torch.randn(1, 64, 256, 256, generator=g)
    geom = (3, 3, 1, 1, 1, 1, 1, 1, dg)
    x, off, m, go = (t.to(dtype).to(dev) for t in (x, off, m, go))
    w, b = w.to(dev), b.to(dev)
    if packed:
        om = torch.cat([off, m], 1).contiguous()
        _ext.dcn_v2_forward_packed(x, w, b, om, *geom)          # the blocked input copy, as in training
        return lambda: _ext.dcn_v2_backward_packed(x, w, b, om, go, *geom)
    m = torch.sigmoid(m.float()).to(dtype)
    _ext.dcn_v2_forward(x, w, b, off, m, *geom)
    return lambda: _ext.dcn_v2_backward(x, w, b, off, m, go, *geom)


def set_arm(arm):
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update(ARMS[arm])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # twice the 126 MB L2
    print("card, power limit:", card())
    cases = []
    for dtype in (torch.float32, torch.bfloat16):
        for packed in (False, True):
            for sigma in (2.0, 10.0):
                cases.append((f"cfg1 dg8 {str(dtype)[6:]} {'packed' if packed else 'plain'} off {sigma:g}*randn",
                              8, sigma, dtype, packed))
    for sigma in (2.0, 10.0):
        cases.append((f"DCN(64,64,3,dg=2) fp32 plain off {sigma:g}*randn", 2, sigma, torch.float32, False))
    print(f"{'case':48s} " + " ".join(f"{a:>11s}" for a in ARMS) + "   (ms, median)")
    for name, dg, sigma, dtype, packed in cases:
        fn = case(dev, dg, sigma, dtype, packed)
        times = {a: [] for a in ARMS}
        for it in range(args.iters + 3):
            for arm in ARMS:
                set_arm(arm)
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if it >= 3:                                             # warm-up of every arm
                    times[arm].append(e0.elapsed_time(e1))
        med = {a: sorted(v)[len(v) // 2] for a, v in times.items()}
        print(f"{name:48s} " + " ".join(f"{med[a]:11.3f}" for a in ARMS), flush=True)
        del fn
    set_arm("default")


if __name__ == "__main__":
    main()
