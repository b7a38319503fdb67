// dcn_common.cuh — geometry and bilinear-tap helpers shared by the DCNv2 kernels
// (SIMT fallback in dcn.cu, tensor-core path in dcn_tc.cu).
#pragma once
#include "common.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace ebfi_dcn {

constexpr int KC_MAX = 96;    // rows of the sampled slab in the SIMT kernels (channels-in-chunk * kh*kw)

struct DcnDims {
    int B, C, H, W, Co, Ho, Wo;
    int kh, kw, sh, sw, ph, pw, dh, dw, dg;
    int cpg;          // channels per deformable group
    int cch;          // channels per chunk (<= cpg, cch*KK <= KC_MAX)
    int nchunk;       // chunks per group
    int KK;           // kh*kw
    int ntile;        // pixel tiles per sample
    // offset / mask addressing. Separate tensors (the reference's _ext interface): off_bs = dg*2*KK*plane,
    // mask_bs = dg*KK*plane. Packed (ebfi_dcnv2_*_packed): both are views into the raw (B, 3*dg*KK, Ho, Wo)
    // output of conv_offset_mask (dcn_v2.py:217-219: offset = channels [0, 2*dg*KK), mask logits = the last
    // third), off_bs = mask_bs = 3*dg*KK*plane, and the mask is sigmoid(logit) (dcn_v2.py:225).
    long long off_bs, mask_bs;
    int off_bp, mask_bp;      // the same batch strides in planes (off_bs / (Ho*Wo), ...), for TMA plane coordinates
    int packed;
    float *abs_sum;   // packed forward only, nullable: += sum |offset| (DCN_sep's `offset_mean` warning, :221-223)
    // EBFI_DCN_DETERMINISTIC (backward): grad_input is accumulated as int64 fixed point (by the box kernel: its far
    // samples only). det_bound -> 3 device floats {max_px sum_co |gO|, max |weight|, max |mask|} whose product bounds
    // every single contribution;
    // det_head = 62 - bits(max contributions per element): sums stay below 2^62 for scale = 2^(det_head - e),
    // bound < 2^e.
    int det, det_head;
    const float *det_bound;
    int in_blocked;   // EBFI_DCN_INPUT_BLOCKED (backward): `input` already is the group-blocked copy [b][C/8][y][x][8]
};

__device__ __forceinline__ int det_scale_exp(const DcnDims &d)
{
    const float bound = d.det_bound[0] * d.det_bound[1] * d.det_bound[2];
    int e = 0;
    if (bound > 0.f && bound < 3.0e38f) frexpf(bound, &e);      // bound < 2^e
    return max(-120, min(120, d.det_head - e));
}
// A NaN / Inf in grad_output, weight or mask makes the bound non-finite: the fixed-point sums are then meaningless and
// the conversion kernels write NaN instead, so that overflow checks on grad_input (AMP GradScaler) still fire.
__device__ __forceinline__ bool det_bound_nonfinite(const DcnDims &d)
{
    const float bound = d.det_bound[0] * d.det_bound[1] * d.det_bound[2];
    return !(bound < 3.0e38f);
}
__device__ __forceinline__ void det_add(long long *p, float v, float scale)
{
    // power-of-two scaling is exact; one rounding to the fixed-point grid; integer addition is associative
    atomicAdd(reinterpret_cast<unsigned long long *>(p), (unsigned long long)__float2ll_rn(v * scale));
}

// Activation element type T (float | __nv_bfloat16 | __half) of the tensor-core kernels: input, offset, mask and
// grad_output are read as T and widened exactly, output and the activation gradients are rounded once (RN) from the fp32
// values the float instantiation stores; an fp16 store overflows to +-inf, as tensor.half() does. Everything in between
// (blocked input copy, boxes, weights, partials) is fp32.
__device__ __forceinline__ float act_f(float v) { return v; }
__device__ __forceinline__ float act_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float act_f(__half v) { return __half2float(v); }
__device__ __forceinline__ float ld_act(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ld_act(const __nv_bfloat16 *p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ld_act(const __half *p) { return __half2float(__ldg(p)); }
template <typename T> __device__ __forceinline__ T st_act(float v);
template <> __device__ __forceinline__ float st_act<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 st_act<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half st_act<__half>(float v) { return __float2half_rn(v); }

template <typename T>
__device__ __forceinline__ const T *off_ptr(const DcnDims &d, const T *offset, int b, int g, size_t plane)
{
    return offset + (size_t)b * d.off_bs + (size_t)g * 2 * d.KK * plane;
}
template <typename T>
__device__ __forceinline__ const T *mask_ptr(const DcnDims &d, const T *mask, int b, int g, size_t plane)
{
    return mask + (size_t)b * d.mask_bs + (size_t)g * d.KK * plane;
}
// modulation scalar from the stored value: identity, or the sigmoid the module applies (dcn_v2.py:225)
__device__ __forceinline__ float mask_act(const DcnDims &d, float raw)
{
    return d.packed ? 1.f / (1.f + expf(-raw)) : raw;
}
// compile-time variants for the tensor-core kernels (no branch / flag register in their inner loops)
template <bool PACKED> __device__ __forceinline__ float mask_act_t(float raw)
{
    return PACKED ? 1.f / (1.f + expf(-raw)) : raw;
}
template <bool PACKED> __device__ __forceinline__ float mask_act_grad_t(float m)
{
    return PACKED ? m * (1.f - m) : 1.f;
}
// d(mask_act)/d(raw) given the activated value
__device__ __forceinline__ float mask_act_grad(const DcnDims &d, float m)
{
    return d.packed ? m * (1.f - m) : 1.f;
}

// One bilinear tap: corner indices, validity and weights (im2col_cuda.cu:25-54, :180).
struct Tap {
    int i00, i01, i10, i11;    // plane offsets of the four corners
    bool c00, c01, c10, c11;   // corner inside the image AND sample inside the window
    float hy, hx, ly, lx;
};

__device__ __forceinline__ Tap make_tap(float y, float x, int H, int W)
{
    Tap t;
    const bool inside = (y > -1.f) && (x > -1.f) && (y < (float)H) && (x < (float)W);
    const float fy = floorf(y), fx = floorf(x);
    const int y0 = (int)fy, x0 = (int)fx;
    t.ly = y - fy; t.lx = x - fx;
    t.hy = 1.f - t.ly; t.hx = 1.f - t.lx;
    const bool ya = y0 >= 0, yb = y0 + 1 <= H - 1, xa = x0 >= 0, xb = x0 + 1 <= W - 1;
    t.c00 = inside && ya && xa; t.c01 = inside && ya && xb;
    t.c10 = inside && yb && xa; t.c11 = inside && yb && xb;
    t.i00 = y0 * W + x0; t.i01 = t.i00 + 1; t.i10 = t.i00 + W; t.i11 = t.i10 + 1;
    return t;
}

__device__ __forceinline__ void tap_coords(const DcnDims &d, const float *__restrict__ off_bg,
                                           const float *__restrict__ mask_bg, int t, int pix,
                                           float &y, float &x, float &xq, float &m, float &oy, float &ox)
{
    const size_t plane = (size_t)d.Ho * d.Wo;
    const int ho = pix / d.Wo, wo = pix - ho * d.Wo;
    const int i = t / d.kw, j = t - i * d.kw;
    oy = __ldg(off_bg + (size_t)(2 * t) * plane + pix);
    ox = __ldg(off_bg + (size_t)(2 * t + 1) * plane + pix);
    m = mask_act(d, __ldg(mask_bg + (size_t)t * plane + pix));
    y = (float)(ho * d.sh - d.ph + i * d.dh) + oy;
    x = (float)(wo * d.sw - d.pw + j * d.dw) + ox;
    xq = (float)(wo * d.sw - d.ph + j * d.dw) + ox;   // the scatter's x (pad_h quirk, :368)
}


// warp-sum of `v`, then one atomic per warp into *dst (order-dependent rounding: statistics only)
__device__ __forceinline__ void warp_atomic_sum(float *dst, float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(dst, v);
}

// Division-free read of one tap's (dy, dx, raw mask value) for kernels that already know the pixel index:
// offset channel 2t = dy, 2t+1 = dx inside the group (im2col_cuda.cu:170-171); plane = Ho * Wo.
template <typename T>
__device__ __forceinline__ void tap_read(const T *__restrict__ off_bg, const T *__restrict__ mask_bg,
                                         unsigned plane, unsigned t, unsigned pix, float &dy, float &dx, float &m)
{
    const unsigned o = 2u * t * plane + pix;
    dy = ld_act(off_bg + o);
    dx = ld_act(off_bg + o + plane);
    m = ld_act(mask_bg + t * plane + pix);
}

// 256-bit read-only global load (sm_100+: LDG.E.256): the 8 channels of one bilinear corner in the
// group-blocked layout, one instruction and one L1 wavefront per lane instead of two.
struct f8 { float v[8]; };
__device__ __forceinline__ f8 ldg_f8(const float *p32B_aligned, bool ok)
{
    f8 r;
    if (ok) {
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                     : "l"(p32B_aligned));
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) r.v[i] = 0.f;
    }
    return r;
}

// {max_px sum_co |gO|, max |weight|, max |mask|} -> bound[3] (dcn.cu)
int launch_det_bound(cudaStream_t st, const DcnDims &d, const float *gout, const float *weight, const float *mask, float *bound);

// NCHW (BG*8 planes of HW pixels, T = float | __nv_bfloat16 | __half) -> fp32 group-blocked (BG, HW, 8) copy (dcn_bwd_tc.cu)
template <typename T>
int launch_nchw_to_blocked(cudaStream_t st, const T *src, float *dst, int BG, int HW, void *zero = nullptr, int zero_f4 = 0);

}  // namespace ebfi_dcn
