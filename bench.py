#!/usr/bin/env python
"""bench.py — DCNv2+FAC fwd+bwd Mpix/s on B200 (BASELINE.json metric), with roofline and CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU path (rank 0)

One "step" = one pass of the alignment hot path over one synthetic GoPro-shaped batch, exactly
BASELINE.json configs[0] + configs[1]:
    DCNv2  3x3, C=64->64, deformable_groups=8, B=1, 256x256, fp32, forward + backward
    FAC    KernelConv2D k=5, C=64,            B=4, 256x256, fp32, forward + backward
Mpix/s = (1 + 4) * 256 * 256 output pixels / step time. Every rank runs the same per-GPU batch
(weak scaling); with N > 1 the DCN weight/bias gradients are all-reduced over NCCL each step.

`value`   : inputs resident in HBM, ops called through the drop-in extension modules (`_ext`,
            `kernelconv2d_cuda` shims -> C ABI), CUDA events on the launching stream.
`e2e`     : same step through the autograd Functions with HOST (pinned) inputs and outputs; the
            H2D copies of every input and the D2H copies of every output/gradient are inside the
            timed region.
`roofline`: the dominant kernel (FAC backward): algorithmic bytes per launch / its average
            CUDA-event duration inside the timed region, against MEASURED_PEAKS.json.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 256
C = 64
DG = 8
B_DCN, B_FAC, K_FAC = 1, 4, 5
MPIX_PER_STEP = (B_DCN + B_FAC) * H * W / 1e6

# Algorithmic bytes (SURVEY.md §8d / DESIGN.md): every tensor of the op read or written once.
_F = 4
DCN_FWD_BYTES = _F * (B_DCN * C * H * W + B_DCN * 2 * DG * 9 * H * W + B_DCN * DG * 9 * H * W + C * C * 9 + C
                      + B_DCN * C * H * W)
DCN_BWD_BYTES = _F * (2 * B_DCN * C * H * W + B_DCN * 3 * DG * 9 * H * W + C * C * 9            # reads
                      + B_DCN * C * H * W + B_DCN * 3 * DG * 9 * H * W + C * C * 9 + C)         # writes
FAC_IN = B_FAC * C * (H + 4) * (W + 4)
FAC_KER = B_FAC * C * 25 * H * W
FAC_OUT = B_FAC * C * H * W
FAC_FWD_BYTES = _F * (FAC_IN + FAC_KER + FAC_OUT)
FAC_BWD_BYTES = _F * (FAC_KER + FAC_OUT + FAC_IN + FAC_IN + FAC_KER)
STEP_BYTES = DCN_FWD_BYTES + DCN_BWD_BYTES + FAC_FWD_BYTES + FAC_BWD_BYTES
# kernels of ours per step (profiles/r2f_launches.txt): DCN forward = dcn_prep_weights + nchw_to_blocked +
# dcn_fwd_box_kernel; DCN backward = dcn_bwd_prep_weights + dcn_bwd_box_kernel + dcn_gin_collect +
# dcn_box_reduce_partials (the forward's blocked input copy is reused: a memset node replaces nchw_to_blocked);
# FAC = fac_fwd_march + fac_bwd_march; N > 1 with the fused exchange: + dp_complete_kernel
LAUNCHES_PER_STEP = 9


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region: NVML (the library
    behind nvidia-smi) polled every 5 ms from a thread of this process, so that even a 100 ms region gets
    samples; `nvidia-smi -lms` as the fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, uuid=None):
        self.rows, self.proc, self.index, self.uuid = [], None, index, uuid
        self.nvml, self.handle, self.stop, self.source = None, None, threading.Event(), None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = (pynvml.nvmlDeviceGetHandleByUUID(self.uuid) if self.uuid
                           else pynvml.nvmlDeviceGetHandleByIndex(self.index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml"
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def _poll(self):
        n = self.nvml
        bits = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown,
                n.nvmlClocksEventReasonSwThermalSlowdown, n.nvmlClocksEventReasonSwPowerCap]
        while not self.stop.is_set():
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                self.rows.append([str(mhz), str(self.max_mhz)] + ["Active" if r & b else "Not Active" for b in bits])
            except Exception:
                pass
            time.sleep(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.nvml:
            self.stop.set()
            self.th.join(timeout=2)
        elif self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.th.join(timeout=2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples (NVML and nvidia-smi unavailable)"]}
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) >= 6 and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": self.source}


def _bind_to_gpu_numa_node(torch, dev):
    """Multi-rank runs: pin this process to the CPUs NVML reports as local to its GPU, so that the pinned host
    buffers of the e2e leg are allocated on the GPU's NUMA node (one process per GPU, all ranks share the host)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByUUID(_gpu_uuid(torch, dev)))
    except Exception:
        pass


def _gpu_uuid(torch, dev):
    try:
        return "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        return None


def make_inputs(torch, dev, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    d = dict(
        x=r(B_DCN, C, H, W), off=2 * r(B_DCN, 2 * DG * 9, H, W), msk=torch.sigmoid(r(B_DCN, DG * 9, H, W)),
        w=(torch.rand(C, C, 3, 3, generator=g) * 2 - 1) / 24, b=r(C), go_d=r(B_DCN, C, H, W),
        xi=r(B_FAC, C, H + 4, W + 4), ker=0.1 * r(B_FAC, C * 25, H, W), go_f=r(B_FAC, C, H, W))
    return d


# --------------------------------------------------------------------- ours ---
def run_ours(args):
    import torch
    import torch.distributed as dist
    import ebfi_be_b200
    from ebfi_be_b200 import dcn_v2, kernelconv2d, parallel
    from ebfi_be_b200.shims import _ext, kernelconv2d_cuda as kc

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL on a high-priority stream: its (tiny) all-reduce kernel is scheduled ahead of the queued FAC CTAs
        # instead of waiting behind an HBM-saturating grid
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            pass
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
        _bind_to_gpu_numa_node(torch, dev)
    ebfi_be_b200._lib.load()
    # Data-parallel weight-gradient sum (the only exchange on the path): fused into the DCN backward's own reduction
    # kernel over NVLink peer memory (parallel.GradComm / csrc/dp_comm.cuh); `--nccl-allreduce` keeps the separate
    # flat-bucket NCCL collective of round 1 for comparison.
    comm, comm_err = None, None
    if world > 1 and not args.nccl_allreduce:
        try:
            comm = parallel.GradComm(C * C * 9 + C, dev)
        except Exception as e:      # no peer mapping on this box: say so in the line and use NCCL
            comm_err = f"{type(e).__name__}: {e}"[:200]
        ok = torch.tensor([0 if comm is None else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok) == 0:
            comm = None
    host = make_inputs(torch, dev, 1234 + rank)
    d = {k: v.to(dev) for k, v in host.items()}
    geom = (3, 3, 1, 1, 1, 1, 1, 1, DG)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    out_f = torch.empty(B_FAC, C, H, W, device=dev)
    gi_f, gk_f = torch.empty_like(d["xi"]), torch.empty_like(d["ker"])
    op_names = ["dcn_fwd", "dcn_bwd", "fac_fwd", "fac_bwd"]

    # The four operator calls of a step, each through the drop-in extension module. After the warm-up they are
    # captured into one CUDA graph per operator and replayed: a step then costs four graph launches on the host
    # instead of ~9 kernel launches + a dozen allocator calls from Python, which matters when 8 ranks share the
    # host's cores (the GPUs were starved at N = 8: 1.74 ms per step for 1.41 ms of kernels). `--no-graphs` keeps
    # the eager calls.
    ops = {
        "dcn_fwd": lambda: _ext.dcn_v2_forward(d["x"], d["w"], d["b"], d["off"], d["msk"], *geom),
        "dcn_bwd": lambda: _ext.dcn_v2_backward(d["x"], d["w"], d["b"], d["off"], d["msk"], d["go_d"], *geom, comm=comm, defer=comm is not None),
        "fac_fwd": lambda: kc.forward(d["xi"], d["ker"], K_FAC, out_f),
        "fac_bwd": lambda: kc.backward(d["xi"], d["ker"], K_FAC, d["go_f"], gi_f, gk_f),
    }
    graphs, graph_out = {}, {}

    def run(name):
        if name in graphs:
            graphs[name].replay()
            return graph_out[name]
        return ops[name]()

    def step(marks=None):
        """One pass of the hot path, device-resident. Returns the DCN output and gradients (the FAC results land in
        out_f, gi_f, gk_f)."""
        def mark():
            if marks is not None:
                e = ev(); e.record(); marks.append(e)
        mark()
        out_d = run("dcn_fwd")
        mark()
        grads = run("dcn_bwd")
        # data-parallel weight-gradient all-reduce (the only collective on the path): ONE flat bucket, issued
        # asynchronously so that its latency hides under the FAC kernels; completed before the step ends
        pending = parallel.allreduce_weight_grads(grads[3:5], async_op=True) if (world > 1 and comm is None) else None
        mark()
        run("fac_fwd")
        mark()
        run("fac_bwd")
        mark()                      # kernel intervals end here; the collective's completion is timed separately
        if comm is not None:
            # second half of the fused exchange: the backward's reduction kernel published this rank's sums ~0.9 ms ago;
            # one tiny kernel waits for the peers' flags and adds their values in rank order
            comm.complete(grads[3], grads[4])
        elif pending is not None:
            pending.wait()
        mark()
        return out_d, grads

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if not args.no_graphs:
        for name, fn in ops.items():
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                graph_out[name] = fn()
            graphs[name] = g
        for _ in range(max(3, args.warmup)):      # warm the replay path as well
            step()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    marks, t0, t1 = [], ev(), ev()
    with ClockSampler(local, _gpu_uuid(torch, dev)) as clk:
        t0.record()
        for _ in range(args.steps):
            out_d, grads_d = step(marks)
        t1.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, dict(
            zip(["dcn_out", "dcn_grad_input", "dcn_grad_offset", "dcn_grad_mask", "dcn_grad_weight", "dcn_grad_bias",
                 "fac_out", "fac_grad_input", "fac_grad_kernel"], [out_d, *grads_d, out_f, gi_f, gk_f])))
    ms_total = t0.elapsed_time(t1)
    if world > 1:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt)
    ms_step = ms_total / args.steps
    op_ms = {n: 0.0 for n in op_names}
    allreduce_wait_ms = 0.0
    for s in range(args.steps):
        for i, n in enumerate(op_names):
            op_ms[n] += marks[6 * s + i].elapsed_time(marks[6 * s + i + 1]) / args.steps
        allreduce_wait_ms += marks[6 * s + 4].elapsed_time(marks[6 * s + 5]) / args.steps

    if world > 1:
        # every rank's own kernel time per step vs its step time: tells a slow device from a late host apart
        mine = torch.tensor([sum(op_ms.values()), allreduce_wait_ms, t0.elapsed_time(t1) / args.steps], device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": i, "kernels_ms": round(float(v[0]), 4), "exchange_wait_ms": round(float(v[1]), 4),
                     "step_ms": round(float(v[2]), 4)} for i, v in enumerate(allr)]
    else:
        per_rank = None

    # ---- e2e: autograd Functions, pinned host buffers in and out, copies inside the timed region
    pin = {k: v.pin_memory() for k, v in host.items()}
    res_names = ["out_d", "g_x", "g_off", "g_msk", "g_w", "g_b", "out_f", "g_xi", "g_ker"]
    res_like = [host["go_d"], host["x"], host["off"], host["msk"], host["w"], host["b"], host["go_f"], host["xi"], host["ker"]]
    pin_out = {n: torch.empty_like(t).pin_memory() for n, t in zip(res_names, res_like)}
    h2d = sum(v.numel() * 4 for v in pin.values()); d2h = sum(v.numel() * 4 for v in pin_out.values())

    from ebfi_be_b200.host_pipeline import HostPipeline
    pipe = HostPipeline(dev)
    dcn_res = {"out": pin_out["out_d"], "grad_input": pin_out["g_x"], "grad_offset": pin_out["g_off"],
               "grad_mask": pin_out["g_msk"], "grad_weight": pin_out["g_w"], "grad_bias": pin_out["g_b"]}

    def e2e_step():
        """Host buffers in, host buffers out, through the package's host-pipeline API: per-sample
        H2D | autograd forward+backward | D2H on three streams."""
        s_out, keep = pipe.dcn_forward_backward(pin["x"], pin["off"], pin["msk"], pin["w"], pin["b"], pin["go_d"],
                                                1, 1, 1, DG, dcn_res)
        if world > 1:   # weight-gradient all-reduce; the reduced values are what a trainer would read
            gw, gb = keep[1][3].grad, keep[1][4].grad
            if comm is not None:
                comm.allreduce_(gw, gb)
            else:
                dist.all_reduce(gw); dist.all_reduce(gb)
        pipe.fac_forward_backward(pin["xi"], pin["ker"], pin["go_f"], K_FAC,
                                  pin_out["out_f"], pin_out["g_xi"], pin_out["g_ker"])
        s_out.synchronize()
        torch.cuda.current_stream().synchronize()      # the step's results are on the host

    e2e_steps = 1 if args.kernels_only else max(3, min(args.steps, 10))
    for _ in range(0 if args.kernels_only else 2):
        e2e_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - w0
    if world > 1:
        tt = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt)

    # ---- per-config breakdown with an explicit L2 flush before every timed call (DCN's 90 MB of
    # inputs fit in the 126 MB L2, so back-to-back calls would otherwise be measured warm)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    def timed(fn, n=1 if args.kernels_only else 10):
        ts = []
        for _ in range(n):
            flush.zero_()
            a, b = ev(), ev()
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)
    cold = {
        "dcn_fwd": timed(lambda: _ext.dcn_v2_forward(d["x"], d["w"], d["b"], d["off"], d["msk"], *geom)),
        "dcn_bwd": timed(lambda: _ext.dcn_v2_backward(d["x"], d["w"], d["b"], d["off"], d["msk"], d["go_d"], *geom)),
        "fac_fwd": timed(lambda: kc.forward(d["xi"], d["ker"], K_FAC, out_f)),
        "fac_bwd": timed(lambda: kc.backward(d["xi"], d["ker"], K_FAC, d["go_f"], gi_f, gk_f)),
    }

    # ---- BASELINE configs[2]: event encoders, 10 M synthetic events at 1280x720 (reported beside the
    # headline metric, not part of it). Events are device-resident; the grid memset is inside the call.
    events = None
    if rank == 0 and not args.kernels_only:
        from ebfi_be_b200 import encodings
        g = torch.Generator(device="cpu").manual_seed(7)
        NEV, EH, EW = 10_000_000, 720, 1280
        exs = torch.randint(0, EW, (NEV,), generator=g).float().to(dev)
        eys = torch.randint(0, EH, (NEV,), generator=g).float().to(dev)
        ets = torch.sort(torch.rand(NEV, generator=g, dtype=torch.float64))[0]
        ets = ((ets - ets[0]) / (ets[-1] - ets[0] + 1e-6)).float().to(dev)
        eps_ = (torch.randint(0, 2, (NEV,), generator=g) * 2 - 1).float().to(dev)
        t_vox = timed(lambda: encodings.events_to_voxel(exs, eys, ets, eps_, 5, sensor_size=(EH, EW)), n=10)
        t_stk = timed(lambda: encodings.events_to_stack(exs, eys, ets, eps_, 16, sensor_size=(EH, EW)), n=10)
        events = {"workload": "10M events, 1280x720, fp32 coordinates, uniform pixels, sorted ts",
                  "voxel_5bins": {"ms": round(t_vox, 4), "Mev_s": round(NEV / 1e6 / (t_vox * 1e-3), 1),
                                  "algorithmic_GBps": round((16 * NEV + 4 * 5 * EH * EW) / (t_vox * 1e-3) / 1e9, 1)},
                  "stack_16bins": {"ms": round(t_stk, 4), "Mev_s": round(NEV / 1e6 / (t_stk * 1e-3), 1),
                                   "algorithmic_GBps": round((16 * NEV + 4 * 32 * EH * EW) / (t_stk * 1e-3) / 1e9, 1)}}
        # SURVEY 8(d): clustered events (90 % of them on Gaussian blobs covering ~1 % of the pixels) expose the
        # atomic contention of the scatter
        nb = int(0.9 * NEV)
        cidx = torch.randint(0, 8, (nb,), generator=g)
        cx = torch.tensor([160., 480, 800, 1120, 320, 640, 960, 200])[cidx] + 16 * torch.randn(nb, generator=g)
        cy = torch.tensor([180., 540, 360, 180, 540, 120, 600, 400])[cidx] + 16 * torch.randn(nb, generator=g)
        cxs = torch.cat([cx.clamp(0, EW - 1).floor(), torch.randint(0, EW, (NEV - nb,), generator=g).float()]).to(dev)
        cys = torch.cat([cy.clamp(0, EH - 1).floor(), torch.randint(0, EH, (NEV - nb,), generator=g).float()]).to(dev)
        perm = torch.randperm(NEV, generator=g).to(dev)
        cxs, cys = cxs[perm].contiguous(), cys[perm].contiguous()
        t_cv = timed(lambda: encodings.events_to_voxel(cxs, cys, ets, eps_, 5, sensor_size=(EH, EW)), n=10)
        t_cs = timed(lambda: encodings.events_to_stack(cxs, cys, ets, eps_, 16, sensor_size=(EH, EW)), n=10)
        events["clustered_90pct_on_1pct_of_pixels"] = {
            "voxel_5bins": {"ms": round(t_cv, 4), "Mev_s": round(NEV / 1e6 / (t_cv * 1e-3), 1)},
            "stack_16bins": {"ms": round(t_cs, 4), "Mev_s": round(NEV / 1e6 / (t_cs * 1e-3), 1)}}
        del cxs, cys, perm
        # the datasets' path on the on-disk dtypes (int16, int16, float64, int8): device-resident, and end to end
        # from pageable numpy arrays (what h5py returns) through the pinned staging of EventSliceFeeder
        rxs, rys = exs.to(torch.int16), eys.to(torch.int16)
        rts = torch.sort(torch.rand(NEV, generator=g, dtype=torch.float64))[0].to(dev) * 0.5 + 100.0
        rps = eps_.to(torch.int8)
        t_raw = timed(lambda: encodings.events_raw_to_stack(rxs, rys, rts, rps, 16, (EH, EW)), n=10)
        feeder = encodings.EventSliceFeeder(dev, 16, (EH, EW), max_events=NEV)
        host_slice = tuple(t.cpu().numpy() for t in (rxs, rys, rts, rps))
        for _ in range(2):
            feeder.encode([host_slice]); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            feeder.encode([host_slice])
        torch.cuda.synchronize()
        t_feed = (time.perf_counter() - t0) / 3 * 1e3
        events["raw_stack_16bins"] = {"ms": round(t_raw, 4), "Mev_s": round(NEV / 1e6 / (t_raw * 1e-3), 1),
                                      "algorithmic_GBps": round((13 * NEV + 4 * 32 * EH * EW) / (t_raw * 1e-3) / 1e9, 1),
                                      "host_numpy_to_stack_ms": round(t_feed, 2),
                                      "host_numpy_to_stack_Mev_s": round(NEV / 1e6 / (t_feed * 1e-3), 1),
                                      "h2d_bytes": 13 * NEV}
        del exs, eys, ets, eps_, rxs, rys, rts, rps, feeder

    # ---- SURVEY 8f widenings, reported beside the headline metric (rank 0, N=1 runs only)
    widen = None
    if rank == 0 and world == 1 and not args.kernels_only:
        widen = widening_numbers(torch, dev, d, timed)

    # ---- SURVEY 8(e) row 3: every rank encodes its own event window (no collective); aggregate = N windows / max time
    enc_scaling = None
    if not args.kernels_only:
        from ebfi_be_b200 import encodings
        g = torch.Generator(device="cpu").manual_seed(70 + rank)
        NEV, EH, EW = 10_000_000, 720, 1280
        exs = torch.randint(0, EW, (NEV,), generator=g).float().to(dev)
        eys = torch.randint(0, EH, (NEV,), generator=g).float().to(dev)
        ets = torch.sort(torch.rand(NEV, generator=g))[0].to(dev)
        eps_ = (torch.randint(0, 2, (NEV,), generator=g) * 2 - 1).float().to(dev)
        if world > 1:
            dist.barrier()
        t_v = timed(lambda: encodings.events_to_voxel(exs, eys, ets, eps_, 5, sensor_size=(EH, EW)), n=10)
        t_s = timed(lambda: encodings.events_to_stack(exs, eys, ets, eps_, 16, sensor_size=(EH, EW)), n=10)
        if world > 1:
            tt = torch.tensor([t_v, t_s], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_v, t_s = float(tt[0]), float(tt[1])
        enc_scaling = {"workload": "each rank encodes its own 10M-event window at 1280x720 (no collective); max time over ranks",
                       "voxel_5bins_Gev_s": round(world * NEV / 1e9 / (t_v * 1e-3), 2),
                       "stack_16bins_Gev_s": round(world * NEV / 1e9 / (t_s * 1e-3), 2), "n_gpus": world}
        del exs, eys, ets, eps_

    # ---- BASELINE configs[3] / configs[4]: the reference's own model on these kernels (tools/bench_model.py)
    cfg4 = cfg5 = None
    if not (args.kernels_only or args.no_model):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_model
        torch.cuda.empty_cache()
        try:
            if world == 1:
                cfg4 = bench_model.cfg4_inference(torch, dev)
            cfg5 = bench_model.cfg5_train_step(torch, dev, world)
        except Exception as e:       # the legs are reported beside the headline; a failure there must not lose the line
            import traceback
            err = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-800:]}
            cfg4 = cfg4 or (err if world == 1 else None)
            cfg5 = cfg5 or err

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    op_bytes = {"dcn_fwd": DCN_FWD_BYTES, "dcn_bwd": DCN_BWD_BYTES, "fac_fwd": FAC_FWD_BYTES, "fac_bwd": FAC_BWD_BYTES}
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):      # DRAM bytes of one launch from the committed `ncu --set full` capture (ncu cannot run inside a timed bench)
        with open(tp) as f:
            tj = json.load(f)
        traffic = tj.get("fac_bwd_march")
        traffic_src = f"profiles/{tj.get('tag', '?')}_fac_bwd_march.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full)"
    dom = "fac_bwd"
    line = {
        "metric": "DCNv2+FAC fwd+bwd Mpix/s", "value": round(world * MPIX_PER_STEP / (ms_step * 1e-3), 3),
        "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[0]+[1]: DCNv2 3x3 C=64 dg=8 B=1 256x256 fwd+bwd, then FAC "
                               "KernelConv2D k=5 C=64 B=4 256x256 fwd+bwd, per GPU",
                   "pixels_per_step_per_gpu": int(MPIX_PER_STEP * 1e6), "parallelism": f"dp{world} (batch-sharded)",
                   "l2": "inputs larger than L2: each step streams 5.4 GB of FAC tensors (>> 126 MB L2) "
                         "between consecutive DCN calls; breakdown.cold_ms flushes L2 explicitly",
                   "collective": ("none" if world == 1 else
                                  "DCN grad_weight+grad_bias all-reduce fused into dcn_box_reduce_partials: the kernel publishes the rank's "
                                  "sums to NVLink peer memory, a tiny kernel after the FAC calls adds the peers' (no NCCL call)" if comm is not None else
                                  "one flat-bucket NCCL all-reduce of DCN grad_weight+grad_bias per step, overlapped with the FAC kernels"
                                  + (f" (peer-memory communicator unavailable: {comm_err})" if comm_err else ""))},
        "roofline": {"bound": "hbm", "kernel": "fac_bwd_march<5,4,ring> (FAC fused backward)",
                     "achieved": round(gbs(op_bytes[dom], op_ms[dom]), 1), "peak": peak, "unit": "GB/s",
                     "frac": round(gbs(op_bytes[dom], op_ms[dom]) / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": op_bytes[dom], "peak_source": peak_src,
                     "step_frac": round(gbs(STEP_BYTES, ms_step) / peak, 4)},
        "breakdown": {n: {"ms": round(op_ms[n], 4), "cold_ms": round(cold[n], 4),
                          "algorithmic_GBps": round(gbs(op_bytes[n], op_ms[n]), 1),
                          "hbm_frac": round(gbs(op_bytes[n], op_ms[n]) / peak, 4)} for n in op_names},
        "configs_mpix_s": {
            "cfg1_dcn_B1": round(B_DCN * H * W / 1e6 / ((cold["dcn_fwd"] + cold["dcn_bwd"]) * 1e-3), 2),
            "cfg2_fac_B4": round(B_FAC * H * W / 1e6 / ((op_ms["fac_fwd"] + op_ms["fac_bwd"]) * 1e-3), 2)},
        "e2e": {"value": round(world * MPIX_PER_STEP * e2e_steps / e2e_s, 3), "unit": "Mpix/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "api": "ebfi_be_b200.host_pipeline (dcn_v2_conv / KernelConv2DFunction autograd, pinned host in/out, "
                       "per-sample H2D | compute | D2H on three streams)"},
        "allreduce_wait_ms": round(allreduce_wait_ms, 4) if world > 1 else None,
        "per_rank": per_rank,
        "events": events,
        "events_per_rank": enc_scaling,
        "cfg4_inference_720p": cfg4,
        "cfg5_train_step": cfg5,
        "widening": widen,
        "gpu_launches": (LAUNCHES_PER_STEP + (1 if comm is not None else 0)) * args.steps,
        "launch_mode": "eager" if args.no_graphs else "one CUDA graph per operator call (4 replays per step)",
        "clocks": clk.summary(),
    }
    if world == 1 and not (args.no_cpu_baseline or args.kernels_only):
        line["cpu_baseline"] = cpu_baseline(budget_s=20.0)
        ref_gpu = reference_cuda_kernels(torch, d, timed)
        if ref_gpu:
            line["cpu_baseline"]["reference_cuda_kernels_sm100a"] = ref_gpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ELEMENTS = 1 << 21       # 8 MB of float32 per array; the nine arrays of a step stay under 64 MB


def dump_outputs(torch, out_dir, arrays):
    """--dump-outputs: write each array as out_dir/<name>.npy in float32, flattened. An array of more than
    DUMP_MAX_ELEMENTS elements is written as its values at DUMP_MAX_ELEMENTS positions drawn from a fixed seed, so
    two runs (or two builds) with the same arguments can be compared element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randint(0, flat.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.float().cpu().numpy())


def widening_numbers(torch, dev, d, timed):
    """The two operator-level widenings of SURVEY 8f at the benchmark shapes, each against the reference's own op
    sequence on the same GPU (torch/cuDNN ops + this repo's unfused operators), L2 flushed before every call."""
    from ebfi_be_b200 import dcn_v2, modification
    from ebfi_be_b200.kernelconv2d import KernelConv2D
    out = {}
    with torch.no_grad():
        # rank 1: KernelConv (3x3 conv 128 -> 1600, LeakyReLU) -> KPN, model_singleframe.py:145-146,161-162
        ev, fr = d["xi"][:, :, 2:-2, 2:-2].contiguous(), d["go_f"]
        conv = torch.nn.Conv2d(2 * C, C * K_FAC * K_FAC, 3, 1, 1).to(dev)
        act, kpn = torch.nn.LeakyReLU(), KernelConv2D(kernel_size=K_FAC)
        t_ref = timed(lambda: kpn(ev, act(conv(torch.cat([ev, fr], 1)))), n=5)
        t_fused = timed(lambda: modification.kernelconv_fac_fused(ev, fr, conv.weight, conv.bias, K_FAC, 0.01), n=5)
        # the same sequence at the fused kernel's operand precision (bf16 conv operands, fp32 accumulation and output)
        def ref_bf16():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                k = act(conv(torch.cat([ev, fr], 1)))
            return kpn(ev, k.float())
        t_ref16 = timed(ref_bf16, n=5)
        flops = 2.0 * B_FAC * H * W * (C * K_FAC * K_FAC) * (2 * C * 9)
        out["kernelconv_to_fac_forward"] = {
            "workload": f"B={B_FAC} C={C} K={K_FAC} {H}x{W}, fp32 tensors (conv operands bf16 on the tensor cores)",
            "reference_sequence_ms": round(t_ref, 4), "fused_ms": round(t_fused, 4), "speedup": round(t_ref / t_fused, 2),
            "reference_sequence_bf16_conv_ms": round(t_ref16, 4), "speedup_at_equal_precision": round(t_ref16 / t_fused, 2),
            "fused_TFLOPs": round(flops / (t_fused * 1e-3) / 1e12, 1),
            "note": "reference sequence = cuDNN conv (TF32, torch default) + LeakyReLU + this repo's FAC forward; "
                    "`_bf16_conv` = the same with the conv under bf16 autocast (the fused kernel's operand precision); the "
                    "1.68 GB kernel tensor is never materialised by the fused kernel"}
        del conv
    # rank 2: DCN_sep tail (chunk, cat, mean|offset| + host sync, sigmoid, op) forward + backward, dcn_v2.py:217-227
    x = d["x"].clone().requires_grad_()
    om = torch.cat([d["off"], torch.logit(d["msk"].clamp(1e-4, 1 - 1e-4))], 1).requires_grad_()
    w, b = d["w"].clone().requires_grad_(), d["b"].clone().requires_grad_()
    watch = dcn_v2._OffsetWatch()

    def ref_tail():
        o1, o2, mask = torch.chunk(om, 3, dim=1)
        offset = torch.cat((o1, o2), dim=1)
        if torch.mean(torch.abs(offset)) > 100:
            pass
        dcn_v2.dcn_v2_conv(x, offset, torch.sigmoid(mask), w, b, 1, 1, 1, DG).backward(d["go_d"])

    def packed_tail():
        watch.poll()
        stat = torch.empty(1, device=dev)
        o = dcn_v2.dcn_v2_conv_packed(x, om, w, b, 1, 1, 1, DG, stat)
        watch.submit(stat, om.numel() // 3 * 2)
        o.backward(d["go_d"])

    t_ref, t_pk = timed(ref_tail, n=10), timed(packed_tail, n=10)
    out["dcn_sep_tail_fwd_bwd"] = {"workload": "cfg1 (B=1, 64->64, 3x3, dg=8, 256x256)", "reference_sequence_ms": round(t_ref, 4),
                                   "packed_ms": round(t_pk, 4), "speedup": round(t_ref / t_pk, 2)}
    del x, om, w, b
    # BASELINE configs[3] (720p inference) cannot run here (the model needs the reference tree); this is the slice of
    # it that this repo owns, at that config's shapes: the two per-frame maps at 1280x720, and at the half-resolution
    # feature grid (360x640, model_singleframe.py:244-245) the packed DCN forward and the fused KernelConv -> FAC.
    from ebfi_be_b200 import frame_ops
    with torch.no_grad():
        g = torch.Generator(device="cpu").manual_seed(11)
        frame = torch.rand(1, 3, 720, 1280, generator=g).to(dev)
        fh, fw = 360, 640
        feat = torch.randn(1, C, fh, fw, generator=g).to(dev)
        fea2 = torch.randn(1, C, fh, fw, generator=g).to(dev)
        om4 = torch.randn(1, 3 * DG * 9, fh, fw, generator=g).to(dev)
        wk = (0.03 * torch.randn(C * 25, 2 * C, 3, 3, generator=g)).to(dev)
        bk = torch.zeros(C * 25, device=dev)
        t_maps = timed(lambda: (frame_ops.Frame2Lap(frame), frame_ops.Frame2DCP(frame)), n=10)
        t_dcn = timed(lambda: dcn_v2.dcn_v2_conv_packed(feat, om4, d["w"], d["b"], 1, 1, 1, DG), n=10)
        t_kpn = timed(lambda: modification.kernelconv_fac_fused(feat, fea2, wk, bk, K_FAC, 0.01), n=10)
    out["cfg4_owned_slice_720p_inference"] = {
        "frame_maps_ms": round(t_maps, 4), "dcn_packed_forward_360x640_ms": round(t_dcn, 4),
        "kernelconv_fac_fused_360x640_ms": round(t_kpn, 4), "total_ms": round(t_maps + t_dcn + t_kpn, 4),
        "note": "one call of each owned operator at the shapes of the 720p inference config; the rest of the model "
                "(stock cuDNN layers) is out of scope"}
    return out


def _load_ref_ext(subdir, name):
    import importlib.util
    d = os.path.join(ROOT, "oracle", "_ref", subdir)
    for f in (os.listdir(d) if os.path.isdir(d) else []):
        if f.startswith(name + ".") and f.endswith(".so"):
            spec = importlib.util.spec_from_file_location(name, os.path.join(d, f))
            mod = importlib.util.module_from_spec(spec)
            try:
                spec.loader.exec_module(mod)
                return mod
            except ImportError:
                return None
    return None


def reference_cuda_kernels(torch, d, timed):
    """SURVEY 8(d)(v): the reference's OWN CUDA kernels (dcn_v2_im2col_cuda.cu, KernelConv2D_kernel.cu),
    compiled unmodified for sm_100a by oracle/build_ref.py, on the same device-resident inputs as the step:
    the GPU-side baseline reported beside the CPU one. Not part of any product path."""
    ref_d, ref_f = _load_ref_ext("dcn_cuda", "_ext_cuda_ref"), _load_ref_ext("fac_cuda", "kernelconv2d_cuda")
    if ref_d is None or ref_f is None:
        return None
    geom = (3, 3, 1, 1, 1, 1, 1, 1, DG)
    allow = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False          # the reference's SGEMMs are fp32
    try:
        t = {"dcn_fwd": timed(lambda: ref_d.dcn_v2_forward(d["x"], d["w"], d["b"], d["off"], d["msk"], *geom), n=5),
             "dcn_bwd": timed(lambda: ref_d.dcn_v2_backward(d["x"], d["w"], d["b"], d["off"], d["msk"], d["go_d"], *geom), n=5)}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = allow

    def fac_fwd():                                         # KernelConv2D.py:35-37: zeroed output, then the kernel
        out = torch.zeros(B_FAC, C, H, W, device=d["xi"].device)
        ref_f.forward(d["xi"], d["ker"], K_FAC, out)

    def fac_bwd():                                         # KernelConv2D.py:50-53
        gi, gk = torch.zeros_like(d["xi"]), torch.zeros_like(d["ker"])
        ref_f.backward(d["xi"], d["ker"], K_FAC, d["go_f"], gi, gk)

    t["fac_fwd"], t["fac_bwd"] = timed(fac_fwd, n=5), timed(fac_bwd, n=5)
    total = sum(t.values())
    return {"ms": {k: round(v, 4) for k, v in t.items()}, "ms_per_step": round(total, 4),
            "value": round(MPIX_PER_STEP / (total * 1e-3), 2), "unit": "Mpix/s",
            "note": "reference .cu files compiled for sm_100a + its host sequence (cuBLAS fp32 GEMMs, column buffer, "
                    "zero-filled FAC outputs); L2 flushed before each call"}


# ---------------------------------------------------------------- CPU arms ---
def _load_ref_dcn_cpu():
    """The reference's own CPU DCNv2 (oracle/_ref/dcn_cpu/_ext*.so, built from the unmodified
    sources by oracle/build_ref.py); None when it did not travel / does not load."""
    import importlib.util
    d = os.path.join(ROOT, "oracle", "_ref", "dcn_cpu")
    if not os.path.isdir(d):
        return None
    for f in os.listdir(d):
        if f.startswith("_ext.") and f.endswith(".so"):
            try:
                spec = importlib.util.spec_from_file_location("_ext", os.path.join(d, f))
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                return mod
            except Exception:
                return None
    return None


def _cpu_step(torch, ref_dcn, oracle, rows, data):
    """DCN fwd+bwd on (1, 64, rows, 256) and FAC fwd+bwd on (4, 64, rows, 256) on the host CPU."""
    geom = (3, 3, 1, 1, 1, 1, 1, 1, DG)
    x, off, msk, go = (data[k][:, :, :rows].contiguous() for k in ("x", "off", "msk", "go_d"))
    w, b = data["w"], data["b"]
    t0 = time.perf_counter()
    if ref_dcn is not None:
        ref_dcn.dcn_v2_forward(x, w, b, off, msk, *geom)
        ref_dcn.dcn_v2_backward(x, w, b, off, msk, go, *geom)
    else:
        a = [t.numpy() for t in (x, off, msk, w, b)]
        oracle.dcn_forward(*a, 1, 1, 1, DG, "f32")
        oracle.dcn_backward(*a, go.numpy(), 1, 1, 1, DG, "f32")
    t1 = time.perf_counter()
    xi = data["xi"][:, :, :rows + 4].contiguous().numpy()
    ker = data["ker"][:, :, :rows].contiguous().numpy()
    gof = data["go_f"][:, :, :rows].contiguous().numpy()
    oracle.fac_forward(xi, ker, K_FAC, "f32")
    oracle.fac_backward(xi, ker, gof, K_FAC, "f32")
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def cpu_baseline(budget_s=20.0):
    import torch
    from oracle import oracle
    oracle.lib()
    ref_dcn = _load_ref_dcn_cpu()
    data = make_inputs(torch, None, 1234)
    td, tf = _cpu_step(torch, ref_dcn, oracle, 8, data)               # probe: 8 rows
    rows = int(max(8, min(H, 8 * budget_s / max(td + tf, 1e-6))))
    td, tf = _cpu_step(torch, ref_dcn, oracle, rows, data)
    mpix = (B_DCN + B_FAC) * rows * W / 1e6
    # encoders: the oracle's serial C port of dataloader/encodings.py on the same 10 M events distribution
    import numpy as np
    rng = np.random.default_rng(7)
    n_ev = 10_000_000          # BASELINE configs[2] in full: ~1 s of CPU work for the three encoders
    exs = rng.integers(0, 1280, n_ev).astype(np.float32); eys = rng.integers(0, 720, n_ev).astype(np.float32)
    ets = np.sort(rng.random(n_ev)).astype(np.float32); eps_ = (rng.integers(0, 2, n_ev) * 2 - 1).astype(np.float32)
    t0 = time.perf_counter(); oracle.events_to_voxel(exs, eys, ets, eps_, 5, (720, 1280)); t_v = time.perf_counter() - t0
    t0 = time.perf_counter(); oracle.events_to_stack(exs, eys, ets, eps_, 16, (720, 1280)); t_s = time.perf_counter() - t0
    rts = 100.0 + 0.5 * np.sort(rng.random(n_ev))
    t0 = time.perf_counter()
    oracle.dataset_event_stack(exs.astype(np.int16), eys.astype(np.int16), rts, eps_.astype(np.int8), 16, (720, 1280))
    t_r = time.perf_counter() - t0
    return {"events_voxel_5bins_Mev_s": round(n_ev / 1e6 / t_v, 2), "events_stack_16bins_Mev_s": round(n_ev / 1e6 / t_s, 2),
            "events_dataset_path_16bins_Mev_s": round(n_ev / 1e6 / t_r, 2),
            "value": round(mpix / (td + tf), 5), "unit": "Mpix/s", "cores": torch.get_num_threads(),
            "kind": "reference" if ref_dcn is not None else "port",
            "kind_by_leg": {"dcn": "reference" if ref_dcn is not None else "port", "fac": "port"},
            "sample": f"top {rows} of 256 rows of the same step (DCN B=1 + FAC B=4, fwd+bwd): "
                      f"DCN {td:.2f} s via " + ("the reference's CPU build oracle/_ref/dcn_cpu (serial loops + MKL GEMM)"
                                               if ref_dcn is not None else "the oracle C port")
                      + f", FAC {tf:.2f} s via the oracle C port with OpenMP (the reference has no CPU FAC path)"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    from oracle import oracle
    oracle.lib()
    ref_dcn = _load_ref_dcn_cpu()
    data = make_inputs(torch, None, 1234)
    total = args.steps + args.warmup
    td, tf = _cpu_step(torch, ref_dcn, oracle, 8, data)
    rows = int(max(4, min(H, 8 * (150.0 / total) / max(td + tf, 1e-6))))
    for _ in range(args.warmup):
        _cpu_step(torch, ref_dcn, oracle, rows, data)
    t0 = time.perf_counter()
    sd = sf = 0.0
    for _ in range(args.steps):
        a, b = _cpu_step(torch, ref_dcn, oracle, rows, data)
        sd += a; sf += b
    dt = time.perf_counter() - t0
    mpix = (B_DCN + B_FAC) * rows * W / 1e6
    val = round(mpix * args.steps / dt, 5)
    kind = "reference" if ref_dcn is not None else "port"
    sample = (f"each step = top {rows} of 256 rows of the step (DCN B=1 + FAC B=4, fwd+bwd); DCN via "
              + ("oracle/_ref/dcn_cpu (reference CPU build)" if ref_dcn is not None else "oracle C port")
              + "; FAC via oracle C port + OpenMP (reference has no CPU FAC)")
    print(json.dumps({
        "impl": "reference", "metric": "DCNv2+FAC fwd+bwd Mpix/s", "value": val, "unit": "Mpix/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[0]+[1] (DCNv2 B=1 + FAC B=4, 256x256, fwd+bwd), CPU, bounded sample",
                   "rows_per_step": rows},
        "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": torch.get_num_threads(), "kind": kind,
                         "kind_by_leg": {"dcn": kind, "fac": "port"}, "sample": sample},
        "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "breakdown": {"dcn_s_per_step": round(sd / args.steps, 3), "fac_s_per_step": round(sf / args.steps, 3)},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="eager operator calls instead of CUDA-graph replays")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="N > 1: all-reduce the weight gradients with a separate NCCL collective instead of the fused peer-memory exchange")
    ap.add_argument("--no-model", action="store_true", help="skip the full-model legs (BASELINE configs[3], configs[4])")
    ap.add_argument("--kernels-only", action="store_true",
                    help="profiling runs: skip the e2e, cold-breakdown and CPU-baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the DCN and FAC outputs and gradients of the last timed step to DIR/<name>.npy "
                         "(float32; arrays over 2M elements as a fixed seeded sample of 2M elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1; the reference arm uses all the host threads it can
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[k] = str(os.cpu_count() or 1)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
