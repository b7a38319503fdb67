"""Record tests/golden/ref_*.npz: what the GPU tests that compare with the reference's CUDA kernels check against.

    python tests/golden/make_golden_ref.py [OUT_DIR]        (on a B200; default OUT_DIR: tests/golden)

Those tests used to call the reference's dcn_v2_im2col_cuda.cu and KernelConv2D_kernel.cu, compiled unmodified for
sm_100a from a reference tree outside this repository. The stored values come from this project's kernels at commit
2078ebc. Its kernels are those of 7d91f2f, where the same tests ran against the reference's kernels on a B200 and
passed. So the FAC forward and grad_kernel values stored here are the reference's, bit for bit. The DCN values and
the FAC grad_input are within the tests' tolerances of the reference's (1e-5 forward, 1e-4 gradients, relative).

Re-recording from other kernels turns these tests into a comparison of the kernels with themselves; re-record only
where the reference's own kernels have confirmed the kernels being recorded.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))               # tests/: conftest, gpu_util
import conftest  # noqa: E402,F401  (puts the repository root on sys.path)
import gpu_util as G  # noqa: E402

GRADS = ["grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias"]


def main(out):
    import torch
    from ebfi_be_b200 import dcn_v2, kernelconv2d
    from ebfi_be_b200.shims import _ext, kernelconv2d_cuda as kc
    os.makedirs(out, exist_ok=True)

    # test_dcn_gpu.py::test_matches_reference_cuda_kernels
    d = G.ref_dcn_inputs()
    ts = [d[k].clone().requires_grad_() for k in ("x", "off", "msk", "w", "b")]
    o = dcn_v2.dcn_v2_conv(*ts, 1, 1, 1, 8)
    o.backward(d["go"])
    G.record_ref(os.path.join(out, "ref_dcn_b2_40x40.npz"), d,
                 dict(out=o, **{name: v.grad for name, v in zip(GRADS, ts)}))

    # test_fac_gpu.py::test_matches_reference_cuda_kernels
    for i, (K, f) in enumerate(G.ref_fac_inputs()):
        xg, kg = f["x"].clone().requires_grad_(), f["ker"].clone().requires_grad_()
        o = kernelconv2d.KernelConv2DFunction.apply(xg, kg, K)
        o.backward(f["go"])
        G.record_ref(os.path.join(out, f"ref_fac_case{i}.npz"), f, dict(out=o, grad_input=xg.grad, grad_kernel=kg.grad))

    # test_reference_gpu.py::test_cfg1_exact_shape_vs_reference_cuda
    d = G.cfg1_inputs()
    args = [d[k] for k in ("x", "w", "b", "off", "msk")]
    o = _ext.dcn_v2_forward(*args, *G.DCN_GEOM)
    gr = _ext.dcn_v2_backward(*args, d["go"], *G.DCN_GEOM)
    G.record_ref(os.path.join(out, "ref_cfg1_dcn.npz"), d, dict(out=o, **dict(zip(GRADS, gr))))
    del d, args, o, gr

    # test_reference_gpu.py::test_cfg2_exact_shape_vs_reference_cuda
    for tag, shape in (("cfg2_B4_256", (4, 64, 256, 256)), ("cfg4_720p_half_res", (1, 64, 360, 640))):
        f = G.cfg2_inputs(shape)
        o, gi, gk = torch.empty_like(f["go"]), torch.empty_like(f["xi"]), torch.empty_like(f["ker"])
        kc.forward(f["xi"], f["ker"], 5, o)
        kc.backward(f["xi"], f["ker"], 5, f["go"], gi, gk)
        G.record_ref(os.path.join(out, f"ref_{tag}.npz"), f, dict(out=o, grad_input=gi, grad_kernel=gk))
        del f, o, gi, gk
    torch.cuda.synchronize()
    for name in sorted(os.listdir(out)):
        if name.startswith("ref_"):
            print(name, os.path.getsize(os.path.join(out, name)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
