// dcn.cu — DCNv2 modulated deformable convolution, forward + backward, for sm_100a.
//
// Replaces dcn_v2_cuda_forward / dcn_v2_cuda_backward (models/DCNv2/src/cuda/dcn_v2_cuda.cu:20-216)
// and the three SIMT kernels behind them (src/cuda/dcn_v2_im2col_cuda.cu:125-327).
//
// What is different from the reference, structurally:
//   * The column buffer (B, C*kh*kw, Ho*Wo) — 151 MB at the benchmark shape, written and read
//     back by the reference (dcn_v2_cuda.cu:68,78-92) — never exists in HBM. A CTA samples a
//     [k-chunk x pixel-tile] slab straight into shared memory and contracts it with the
//     weights in the same kernel.
//   * Offsets and masks are read once per (pixel, tap, group) instead of once per channel
//     (the reference re-reads them for each of the 8 channels of a group, im2col_cuda.cu:168-173).
//   * Backward is ONE pass over the pixels per deformable group: col-grad GEMM, coordinate /
//     mask gradients, grad_input scatter, the recomputed columns and the grad_weight partial
//     all come from the same slab. The reference loops over the batch on the host and runs
//     3 kernels + 3 GEMMs per sample, sampling twice (dcn_v2_cuda.cu:150-211).
//   * grad_offset / grad_mask are owned by one thread each (no atomics and none of the reference's
//     duplicated Δh/Δw bilinear work, im2col_cuda.cu:283-320);
//     grad_weight / grad_bias are per-CTA partials reduced in a fixed order.
//
// Arithmetic follows the reference exactly where it is observable: the (-1, H) x (-1, W)
// sampling window (im2col_cuda.cu:180), per-corner bounds (:38-48), the coordinate weights
// (:82-123), and the pad_h-for-both-paddings quirk of the grad_input scatter (:368).
#include "dcn_common.cuh"
#include "dp_comm.cuh"

#include <algorithm>
#include <type_traits>

namespace ebfi_dcn {
// tensor-core forward (dcn_fwd_box.cu); returns EBFI_ERR_UNSUPPORTED when the shape is not eligible.
// T = float | __nv_bfloat16 | __half: the type of input, offset, mask and output.
template <typename T>
int forward_tc(cudaStream_t st, const DcnDims &d, const T *input, const float *weight, const float *bias,
               const T *offset, const T *mask, T *output, void *workspace, size_t workspace_bytes);
size_t forward_tc_workspace(const DcnDims &d);
size_t forward_tc_blocked_offset(const DcnDims &d);
// tensor-core backward (dcn_bwd_tc.cu); splits == 0 when the shape is not eligible
int backward_box_splits(const DcnDims &d);
size_t backward_box_scratch_bytes(const DcnDims &d);
template <typename T>
int backward_box(cudaStream_t st, const DcnDims &d, const T *input, const float *weight, const T *offset,
                 const T *mask, const T *gout, T *gin, T *goff, T *gmask, float *gw, float *gb,
                 float *gw_part, float *gb_part, void *scratch, const ebfi_dp::View *dp, bool dp_defer);
int backward_tc_splits(const DcnDims &d);
size_t backward_tc_scratch_bytes(const DcnDims &d);
int backward_tc(cudaStream_t st, const DcnDims &d, const float *input, const float *weight, const float *offset,
                const float *mask, const float *gout, float *gin, float *goff, float *gmask, float *gw_part,
                float *gb_part, int S, void *scratch);
}

namespace {

using ebfi::ceil_div;
using namespace ebfi_dcn;

constexpr int TP = 64;        // output pixels per tile
constexpr int COT = 64;       // output channels per tile
constexpr int NT = 256;       // threads per CTA
constexpr int TPP = TP + 1;   // padded pitch of the backward slab (scalar, conflict-free by row)
constexpr int GP = TP + 1;    // padded pitch of the grad_output tile

// ------------------------------------------------------------------ forward ---
// grid = (pixel tiles per sample, Cout tiles, B). Each CTA walks all deformable groups /
// channel chunks, sampling a [KC x TP] slab into smem and accumulating a [COT x TP] output
// tile in registers (4 co x 4 px per thread).
__global__ void __launch_bounds__(NT)
dcn_fwd_kernel(const float *__restrict__ input, const float *__restrict__ weight,
               const float *__restrict__ bias, const float *__restrict__ offset,
               const float *__restrict__ mask, float *__restrict__ output, DcnDims d)
{
    extern __shared__ __align__(16) float smem[];
    float *col_s = smem;                         // [KC_MAX][TP]
    float *w_s = smem + KC_MAX * TP;             // [KC_MAX][COT]

    const int tid = threadIdx.x;
    const int b = blockIdx.z, co_base = blockIdx.y * COT, pix_base = blockIdx.x * TP;
    const int npix = d.Ho * d.Wo;
    const size_t plane = (size_t)npix, in_plane = (size_t)d.H * d.W;
    const int Kdim = d.C * d.KK;
    const int pq = tid % 16, cq = tid / 16;      // 4 px x 4 co per thread

    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
    float asum = 0.f;                            // sum |offset| over this thread's taps (packed entry only)

    for (int g = 0; g < d.dg; ++g) {
        const float *off_bg = off_ptr(d, offset, b, g, plane);
        const float *mask_bg = mask_ptr(d, mask, b, g, plane);
        for (int ch = 0; ch < d.nchunk; ++ch) {
            const int c0 = g * d.cpg + ch * d.cch;
            const int nc = min(d.cch, d.cpg - ch * d.cch);
            const int KC = nc * d.KK;
            __syncthreads();                      // previous slab fully consumed
            // weights of this chunk: w_s[kk][co] = weight[co_base+co][c0*KK + kk]
            for (int e = tid; e < KC * COT; e += NT) {
                const int co = e % COT, kk = e / COT;
                w_s[kk * COT + co] = (co_base + co < d.Co)
                    ? __ldg(weight + (size_t)(co_base + co) * Kdim + (size_t)c0 * d.KK + kk) : 0.f;
            }
            // sample: item = (tap, pixel), pixel fastest
            for (int it = tid; it < d.KK * TP; it += NT) {
                const int p = it % TP, t = it / TP, pix = pix_base + p;
                if (pix < npix) {
                    float y, x, xq, m, oy, ox;
                    tap_coords(d, off_bg, mask_bg, t, pix, y, x, xq, m, oy, ox);
                    if (ch == 0 && blockIdx.y == 0) asum += fabsf(oy) + fabsf(ox);
                    const Tap tp = make_tap(y, x, d.H, d.W);
                    const float w1 = tp.hy * tp.hx, w2 = tp.hy * tp.lx, w3 = tp.ly * tp.hx, w4 = tp.ly * tp.lx;
                    const float *ip = input + ((size_t)b * d.C + c0) * in_plane;
                    for (int cc = 0; cc < nc; ++cc, ip += in_plane) {
                        const float v1 = tp.c00 ? __ldg(ip + tp.i00) : 0.f;
                        const float v2 = tp.c01 ? __ldg(ip + tp.i01) : 0.f;
                        const float v3 = tp.c10 ? __ldg(ip + tp.i10) : 0.f;
                        const float v4 = tp.c11 ? __ldg(ip + tp.i11) : 0.f;
                        col_s[(cc * d.KK + t) * TP + p] = (w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4) * m;
                    }
                } else {
                    for (int cc = 0; cc < nc; ++cc) col_s[(cc * d.KK + t) * TP + p] = 0.f;
                }
            }
            __syncthreads();
            // contract: acc[co][px] += w_s[kk][co] * col_s[kk][px]
#pragma unroll 4
            for (int kk = 0; kk < KC; ++kk) {
                const float4 a = *reinterpret_cast<const float4 *>(w_s + kk * COT + cq * 4);
                const float4 c = *reinterpret_cast<const float4 *>(col_s + kk * TP + pq * 4);
                const float av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[r][q] += av[r] * cv[q];
            }
        }
    }
    if (d.abs_sum && blockIdx.y == 0) warp_atomic_sum(d.abs_sum, asum);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int co = co_base + cq * 4 + r;
        if (co >= d.Co) continue;
        const float bv = __ldg(bias + co);
        float *op = output + ((size_t)b * d.Co + co) * plane;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int pix = pix_base + pq * 4 + q;
            if (pix < npix) op[pix] = acc[r][q] + bv;
        }
    }
}

// ----------------------------------------------------------------- backward ---
// grid = (splits S, dg, Cout tiles), one launch per channel chunk `ch` of the groups (one chunk
// for every shape with channels-per-group * taps <= KC_MAX). CTA (s, g, ct) owns the k-rows of chunk `ch`
// and walks the pixel tiles s, s+S, ... of ALL samples. For ct == 0 it produces grad_offset,
// grad_mask, grad_input for its chunk; every ct accumulates its [COT x KC] grad_weight
// partial in registers across all its tiles and writes it once at the end.
// Partials: gw_part[S][Co][Kdim], gb_part[S][Co] -> dcn_reduce_partials (fixed order).
template <bool DET>
__global__ void __launch_bounds__(NT)
dcn_bwd_kernel(const float *__restrict__ input, const float *__restrict__ weight,
               const float *__restrict__ offset, const float *__restrict__ mask,
               const float *__restrict__ gout, float *__restrict__ gin,
               float *__restrict__ goff, float *__restrict__ gmask,
               float *__restrict__ gw_part, float *__restrict__ gb_part, DcnDims d, int ch)
{
    extern __shared__ __align__(16) float smem[];
    float *slab = smem;                          // [KC_MAX][TPP]  col-grad, then columns
    float *go_s = slab + KC_MAX * TPP;           // [COT][GP]      grad_output tile
    float *w_s = go_s + COT * GP;                // [COT][KC_MAX]  weights of the chunk

    const int tid = threadIdx.x;
    const int S = gridDim.x, s = blockIdx.x;
    const int g = blockIdx.y;
    const int ct = blockIdx.z, co_base = ct * COT, nco = min(COT, d.Co - co_base);
    const bool lead = (ct == 0);                 // this CTA also does the data gradients
    const int c0 = g * d.cpg + ch * d.cch;
    const int nc = min(d.cch, d.cpg - ch * d.cch);
    const int KC = nc * d.KK, Kdim = d.C * d.KK;
    const int npix = d.Ho * d.Wo;
    const size_t plane = (size_t)npix, in_plane = (size_t)d.H * d.W;
    const int n_cot = gridDim.z;

    const float det_scale = DET ? ldexpf(1.f, det_scale_exp(d)) : 0.f;   // DET: `gin` is the int64 fixed-point copy
    const int kq = tid % 16, cq = tid / 16;      // grad_weight: rows kq+16i, 4 co per thread
    float gw_acc[4][KC_MAX / 16];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int i = 0; i < KC_MAX / 16; ++i) gw_acc[r][i] = 0.f;
    float gb_acc = 0.f;                          // thread tid < nco owns bias co_base+tid

    for (int tile = s; tile < d.B * d.ntile; tile += S) {
        const int b = tile / d.ntile, pix_base = (tile % d.ntile) * TP;
        const float *off_bg = off_ptr(d, offset, b, g, plane);
        const float *mask_bg = mask_ptr(d, mask, b, g, plane);
        __syncthreads();
        // ---- (a) col-grad slab = W_chunk^T . gO_tile, accumulated over Cout tiles (lead only)
        if (lead) {
            float cg[KC_MAX / 16][4];
#pragma unroll
            for (int i = 0; i < KC_MAX / 16; ++i)
#pragma unroll
                for (int q = 0; q < 4; ++q) cg[i][q] = 0.f;
            const int pq = tid / 16;             // 4 px per thread, rows kq+16i
            for (int cb = 0; cb < n_cot; ++cb) {
                const int cbase = cb * COT, ncb = min(COT, d.Co - cbase);
                if (cb) __syncthreads();
                for (int e = tid; e < COT * TP; e += NT) {
                    const int p = e % TP, co = e / TP, pix = pix_base + p;
                    go_s[co * GP + p] = (co < ncb && pix < npix)
                        ? __ldg(gout + ((size_t)b * d.Co + cbase + co) * plane + pix) : 0.f;
                }
                for (int e = tid; e < COT * KC; e += NT) {
                    const int kk = e % KC, co = e / KC;
                    w_s[co * KC_MAX + kk] = (co < ncb)
                        ? __ldg(weight + (size_t)(cbase + co) * Kdim + (size_t)c0 * d.KK + kk) : 0.f;
                }
                __syncthreads();
                for (int co = 0; co < ncb; ++co) {
                    float gv[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) gv[q] = go_s[co * GP + pq * 4 + q];
#pragma unroll
                    for (int i = 0; i < KC_MAX / 16; ++i) {
                        const int kk = kq + 16 * i;
                        const float wv = kk < KC ? w_s[co * KC_MAX + kk] : 0.f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) cg[i][q] += wv * gv[q];
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < KC_MAX / 16; ++i) {
                const int kk = kq + 16 * i;
                if (kk < KC)
#pragma unroll
                    for (int q = 0; q < 4; ++q) slab[kk * TPP + pq * 4 + q] = cg[i][q];
            }
            __syncthreads();
        }
        // ---- (b) sampling: data gradients (lead) and the recomputed columns (all)
        for (int it = tid; it < d.KK * TP; it += NT) {
            const int p = it % TP, t = it / TP, pix = pix_base + p;
            if (pix >= npix) {
                for (int cc = 0; cc < nc; ++cc) slab[(cc * d.KK + t) * TPP + p] = 0.f;
                continue;
            }
            float y, x, xq, m, oy, ox;
            tap_coords(d, off_bg, mask_bg, t, pix, y, x, xq, m, oy, ox);
            const Tap tp = make_tap(y, x, d.H, d.W);
            const Tap tq = (d.ph == d.pw) ? tp : make_tap(y, xq, d.H, d.W);
            const float w1 = tp.hy * tp.hx, w2 = tp.hy * tp.lx, w3 = tp.ly * tp.hx, w4 = tp.ly * tp.lx;
            const float q1 = tq.hy * tq.hx, q2 = tq.hy * tq.lx, q3 = tq.ly * tq.hx, q4 = tq.ly * tq.lx;
            float s_m = 0.f, s_y = 0.f, s_x = 0.f;
            const float *ip = input + ((size_t)b * d.C + c0) * in_plane;
            float *gp = gin + ((size_t)b * d.C + c0) * in_plane;
            for (int cc = 0; cc < nc; ++cc, ip += in_plane, gp += in_plane) {
                const float v1 = tp.c00 ? __ldg(ip + tp.i00) : 0.f;
                const float v2 = tp.c01 ? __ldg(ip + tp.i01) : 0.f;
                const float v3 = tp.c10 ? __ldg(ip + tp.i10) : 0.f;
                const float v4 = tp.c11 ? __ldg(ip + tp.i11) : 0.f;
                const float val = w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4;
                float *cell = slab + (cc * d.KK + t) * TPP + p;
                if (lead) {
                    const float gc = *cell;
                    s_m += gc * val;                                     // grad_mask (:311)
                    // coordinate weights (:99-120); invalid corners already read as 0
                    const float wy = -tp.hx * v1 - tp.lx * v2 + tp.hx * v3 + tp.lx * v4;
                    const float wx = -tp.hy * v1 + tp.hy * v2 - tp.ly * v3 + tp.ly * v4;
                    const float top = gc * m;
                    s_y += wy * top;
                    s_x += wx * top;
                    // grad_input scatter (:236-251), x position with pad_h
                    if (DET) {
                        long long *gp64 = reinterpret_cast<long long *>(gin) + ((size_t)b * d.C + c0 + cc) * in_plane;
                        if (tq.c00) det_add(gp64 + tq.i00, q1 * top, det_scale);
                        if (tq.c01) det_add(gp64 + tq.i01, q2 * top, det_scale);
                        if (tq.c10) det_add(gp64 + tq.i10, q3 * top, det_scale);
                        if (tq.c11) det_add(gp64 + tq.i11, q4 * top, det_scale);
                    } else {
                        if (tq.c00) atomicAdd(gp + tq.i00, q1 * top);
                        if (tq.c01) atomicAdd(gp + tq.i01, q2 * top);
                        if (tq.c10) atomicAdd(gp + tq.i10, q3 * top);
                        if (tq.c11) atomicAdd(gp + tq.i11, q4 * top);
                    }
                }
                *cell = val * m;                                          // column for grad_weight
            }
            if (lead) {
                float *gy = goff + (size_t)b * d.off_bs + ((size_t)g * 2 * d.KK + 2 * t) * plane + pix;
                float *gm = gmask + (size_t)b * d.mask_bs + ((size_t)g * d.KK + t) * plane + pix;
                s_m *= mask_act_grad(d, m);
                if (ch == 0) { gy[0] = s_y; gy[plane] = s_x; *gm = s_m; }
                else { gy[0] += s_y; gy[plane] += s_x; *gm += s_m; }     // chunks are separate, ordered launches
            }
        }
        // ---- (c) grad_weight partial: gw[co][kk] += sum_p gO[co][p] * col[kk][p]
        if (!lead || n_cot > 1) {
            __syncthreads();
            for (int e = tid; e < COT * TP; e += NT) {
                const int p = e % TP, co = e / TP, pix = pix_base + p;
                go_s[co * GP + p] = (co < nco && pix < npix)
                    ? __ldg(gout + ((size_t)b * d.Co + co_base + co) * plane + pix) : 0.f;
            }
        }
        __syncthreads();
        for (int p = 0; p < TP; ++p) {
            float gv[4], cv[KC_MAX / 16];
#pragma unroll
            for (int r = 0; r < 4; ++r) gv[r] = go_s[(cq * 4 + r) * GP + p];
#pragma unroll
            for (int i = 0; i < KC_MAX / 16; ++i) cv[i] = (kq + 16 * i < KC) ? slab[(kq + 16 * i) * TPP + p] : 0.f;
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < KC_MAX / 16; ++i) gw_acc[r][i] += gv[r] * cv[i];
        }
        if (g == 0 && ch == 0 && tid < nco) {
            float sb = 0.f;
            for (int p = 0; p < TP; ++p) sb += go_s[tid * GP + p];
            gb_acc += sb;
        }
    }
    // ---- write the per-CTA partials
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int co = co_base + cq * 4 + r;
        if (co >= d.Co) continue;
#pragma unroll
        for (int i = 0; i < KC_MAX / 16; ++i) {
            const int kk = kq + 16 * i;
            if (kk < KC) gw_part[((size_t)s * d.Co + co) * Kdim + (size_t)c0 * d.KK + kk] = gw_acc[r][i];
        }
    }
    if (g == 0 && ch == 0 && tid < nco) gb_part[(size_t)s * d.Co + co_base + tid] = gb_acc;
}

// grad_weight[e] = sum_s gw_part[s][e], grad_bias likewise — fixed order, one thread per element.
__global__ void dcn_reduce_partials(const float *__restrict__ gw_part, const float *__restrict__ gb_part,
                                    float *__restrict__ gw, float *__restrict__ gb, int S, int n_w, int n_b)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n_w) {
        float a = 0.f;
        for (int s = 0; s < S; ++s) a += gw_part[(size_t)s * n_w + e];
        gw[e] = a;
    } else if (e < n_w + n_b) {
        const int c = e - n_w;
        float a = 0.f;
        for (int s = 0; s < S; ++s) a += gb_part[(size_t)s * n_b + c];
        gb[c] = a;
    }
}

// ---- deterministic mode (EBFI_DCN_DETERMINISTIC): bound of a single grad_input contribution ----
__device__ __forceinline__ void atomic_max_nonneg(float *dst, float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int *>(dst), __float_as_int(v));   // v >= 0: int order == float order
}

__global__ void dcn_det_bound(const float *__restrict__ gout, const float *__restrict__ weight,
                              const float *__restrict__ mask, float *__restrict__ bound, DcnDims d)
{
    const size_t plane = (size_t)d.Ho * d.Wo, tid = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    const size_t nthr = (size_t)gridDim.x * blockDim.x;
    float m0 = 0.f, m1 = 0.f, m2 = d.packed ? 1.f : 0.f;           // sigmoid(logit) <= 1
    for (size_t i = tid; i < (size_t)d.B * plane; i += nthr) {      // max over pixels of sum_co |gO|
        const size_t b = i / plane, pix = i - b * plane;
        float a = 0.f;
        for (int co = 0; co < d.Co; ++co) a += fabsf(__ldg(gout + (b * d.Co + co) * plane + pix));
        m0 = fmaxf(m0, a);
    }
    for (size_t i = tid; i < (size_t)d.Co * d.C * d.KK; i += nthr) m1 = fmaxf(m1, fabsf(__ldg(weight + i)));
    if (!d.packed)
        for (size_t i = tid; i < (size_t)d.B * d.mask_bs; i += nthr) m2 = fmaxf(m2, fabsf(__ldg(mask + i)));
    atomic_max_nonneg(bound + 0, m0);
    atomic_max_nonneg(bound + 1, m1);
    atomic_max_nonneg(bound + 2, m2);
}

// int64 fixed point -> fp32, one rounding per element (CUDA-core path: NCHW in, NCHW out)
__global__ void dcn_i64_to_f32(const long long *__restrict__ src, float *__restrict__ dst, size_t n, DcnDims d)
{
    const float inv = ldexpf(1.f, -det_scale_exp(d));
    const bool bad = det_bound_nonfinite(d);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = bad ? __uint_as_float(0x7FC00000u) : __ll2float_rn(src[i]) * inv;
}

int fill_dims(const ebfi_dcn_geom *q, DcnDims &d)
{
    EBFI_REQUIRE(q != nullptr, "dcn: null geometry");
    int Ho = 0, Wo = 0;
    if (ebfi_dcnv2_output_size(q, &Ho, &Wo) != EBFI_OK) return EBFI_ERR_INVALID;
    d.B = q->batch; d.C = q->channels; d.H = q->height; d.W = q->width; d.Co = q->channels_out;
    d.Ho = Ho; d.Wo = Wo;
    d.kh = q->kernel_h; d.kw = q->kernel_w; d.sh = q->stride_h; d.sw = q->stride_w;
    d.ph = q->pad_h; d.pw = q->pad_w; d.dh = q->dilation_h; d.dw = q->dilation_w;
    d.dg = q->deformable_group;
    d.cpg = d.C / d.dg;
    d.KK = d.kh * d.kw;
    if (d.KK > KC_MAX)
        return ebfi::fail(EBFI_ERR_UNSUPPORTED, "dcn: kernel %dx%d has more than %d taps", d.kh, d.kw, KC_MAX);
    d.cch = std::max(1, std::min(d.cpg, KC_MAX / d.KK));
    d.nchunk = ceil_div(d.cpg, d.cch);
    d.ntile = ceil_div(Ho * Wo, TP);
    EBFI_REQUIRE((long)d.H * d.W < (1L << 30) && (long)Ho * Wo < (1L << 30), "dcn: plane too large");
    EBFI_REQUIRE(d.B <= 65535 && ceil_div(d.Co, COT) <= 65535, "dcn: batch / Cout too large for the grid");
    const long long taps = (long long)d.dg * d.KK * Ho * Wo;
    d.off_bs = 2 * taps; d.mask_bs = taps; d.packed = 0; d.abs_sum = nullptr;
    d.off_bp = 2 * d.dg * d.KK; d.mask_bp = d.dg * d.KK;
    EBFI_REQUIRE((q->flags & ~(EBFI_DCN_DETERMINISTIC | EBFI_DCN_INPUT_BLOCKED)) == 0, "dcn: unknown flags 0x%x", q->flags);
    d.det = (q->flags & EBFI_DCN_DETERMINISTIC) ? 1 : 0;
    d.in_blocked = (q->flags & EBFI_DCN_INPUT_BLOCKED) ? 1 : 0;
    d.det_bound = nullptr;
    // an element of grad_input receives at most one contribution per (output pixel, tap) of its sample
    int bits = 1;
    while (((long long)1 << bits) < (long long)Ho * Wo * d.KK) ++bits;
    d.det_head = 61 - bits;
    return EBFI_OK;
}

// the raw (B, 3*dg*KK, Ho, Wo) output of conv_offset_mask as offset + mask-logit views
void set_packed(DcnDims &d)
{
    d.off_bs = d.mask_bs = 3 * d.mask_bs;
    d.off_bp = d.mask_bp = 3 * d.dg * d.KK;
    d.packed = 1;
}

int bwd_splits(const DcnDims &d)
{
    // enough CTAs for ~2 per SM over all (group, chunk, Cout-tile) rows, never more than tiles
    const int rows = d.dg * ceil_div(d.Co, COT);
    int S = std::max(1, ceil_div(2 * ebfi::sm_count(), rows));
    return std::min(S, d.B * d.ntile);
}

constexpr size_t kFwdSmem = (size_t)(KC_MAX * TP + KC_MAX * COT) * sizeof(float);
constexpr size_t kBwdSmem = (size_t)(KC_MAX * TPP + COT * GP + COT * KC_MAX) * sizeof(float);

}  // namespace

extern "C" {

int ebfi_dcnv2_output_size(const ebfi_dcn_geom *q, int *height_out, int *width_out)
{
    EBFI_REQUIRE(q && height_out && width_out, "dcn: null argument");
    EBFI_REQUIRE(q->batch > 0 && q->channels > 0 && q->height > 0 && q->width > 0 && q->channels_out > 0,
                 "dcn: non-positive tensor size");
    EBFI_REQUIRE(q->kernel_h > 0 && q->kernel_w > 0 && q->stride_h > 0 && q->stride_w > 0 &&
                 q->dilation_h > 0 && q->dilation_w > 0 && q->pad_h >= 0 && q->pad_w >= 0,
                 "dcn: bad kernel/stride/dilation/padding");
    EBFI_REQUIRE(q->deformable_group > 0 && q->channels % q->deformable_group == 0,
                 "dcn: channels (%d) not divisible by deformable_group (%d)", q->channels, q->deformable_group);
    const int Ho = (q->height + 2 * q->pad_h - (q->dilation_h * (q->kernel_h - 1) + 1)) / q->stride_h + 1;
    const int Wo = (q->width + 2 * q->pad_w - (q->dilation_w * (q->kernel_w - 1) + 1)) / q->stride_w + 1;
    EBFI_REQUIRE(Ho > 0 && Wo > 0, "dcn: empty output %dx%d", Ho, Wo);
    *height_out = Ho; *width_out = Wo;
    return EBFI_OK;
}

size_t ebfi_dcnv2_backward_workspace_bytes(const ebfi_dcn_geom *q)
{
    DcnDims d{};
    if (fill_dims(q, d) != EBFI_OK) return 0;
    const size_t S = (size_t)std::max({bwd_splits(d), backward_tc_splits(d), backward_box_splits(d)});
    const size_t det = d.det ? 256 + (size_t)d.B * d.C * d.H * d.W * sizeof(long long) : 0;   // bound + CUDA-core int64 copy
    return ebfi::round_up(S * ((size_t)d.Co * d.C * d.KK + d.Co) * sizeof(float), (size_t)256) +
           std::max({backward_tc_scratch_bytes(d), backward_box_scratch_bytes(d), det}) + 512;
}

size_t ebfi_dcnv2_blocked_input_offset(const ebfi_dcn_geom *q)
{
    DcnDims d{};
    if (fill_dims(q, d) != EBFI_OK) return 0;
    d.det = 0;
    const char *impl = getenv("EBFI_DCN_IMPL");
    if (impl && impl[0] == 's') return 0;                // the CUDA-core kernels run: no copy is made or read
    if (backward_box_splits(d) == 0) return 0;           // the backward could not use it
    return forward_tc_blocked_offset(d);
}

size_t ebfi_dcnv2_forward_workspace_bytes(const ebfi_dcn_geom *q)
{
    DcnDims d{};
    if (fill_dims(q, d) != EBFI_OK) return 0;
    return forward_tc_workspace(d) + 256;
}

}  // extern "C"

// T = float: every shape. T = __nv_bfloat16 | __half (the *_bf16 / *_fp16 entries): only where the tensor-core kernels
// run; anything else returns EBFI_ERR_UNSUPPORTED before the first launch, and the caller runs the float entry on
// widened copies.
template <typename T> static constexpr const char *act_name() { return std::is_same_v<T, __half> ? "fp16" : "bf16"; }

template <typename T>
static int run_forward(void *stream, const DcnDims &d, const T *input, const float *weight,
                       const float *bias, const T *offset, const T *mask, T *output,
                       void *workspace, size_t workspace_bytes)
{
    EBFI_REQUIRE(input && weight && bias && offset && mask && output, "dcn_forward: null pointer");
    cudaStream_t st = ebfi::as_stream(stream);
    // Tensor-core path (dcn_tc.cu) for the shapes it covers; EBFI_DCN_IMPL=simt forces the
    // CUDA-core kernel below, which handles every shape.
    const char *impl = getenv("EBFI_DCN_IMPL");
    const bool simt = impl && impl[0] == 's';
    if constexpr (!std::is_same_v<T, float>) {
        const size_t need = forward_tc_workspace(d);
        if (simt || need == 0 || !workspace || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 31u))
            return ebfi::fail(EBFI_ERR_UNSUPPORTED, "dcn_forward_%s: no tensor-core forward for this call", act_name<T>());
    }
    if (d.abs_sum) EBFI_CUDA_OK(cudaMemsetAsync(d.abs_sum, 0, sizeof(float), st));
    if (!simt) {
        const int rc = forward_tc<T>(st, d, input, weight, bias, offset, mask, output, workspace, workspace_bytes);
        if (rc != EBFI_ERR_UNSUPPORTED) return rc;
    }
    if constexpr (std::is_same_v<T, float>) {
        EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
        dim3 grid(d.ntile, ceil_div(d.Co, COT), d.B);
        dcn_fwd_kernel<<<grid, NT, kFwdSmem, st>>>(input, weight, bias, offset, mask, output, d);
        EBFI_LAUNCH_OK("dcn_fwd_kernel");
        return EBFI_OK;
    } else {
        return ebfi::fail(EBFI_ERR_UNSUPPORTED, "dcn_forward_%s: no tensor-core forward for this call", act_name<T>());
    }
}

template <typename T>
static int run_backward(void *stream, const DcnDims &d_in, const T *input, const float *weight,
                        const T *offset, const T *mask,
                        const T *grad_output, T *grad_input, T *grad_offset,
                        T *grad_mask, float *grad_weight, float *grad_bias,
                        void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm = nullptr, bool dp_defer = false)
{
    EBFI_REQUIRE(input && weight && offset && mask && grad_output && grad_input && grad_offset &&
                 grad_mask && grad_weight && grad_bias, "dcn_backward: null pointer");
    ebfi_dp::View dpv{};
    if (comm)
        if (int rc = ebfi_dp::make_view(comm, (size_t)d_in.Co * d_in.C * d_in.KK + d_in.Co, dpv)) return rc;
    const ebfi_dp::View *dp = comm ? &dpv : nullptr;
    cudaStream_t st = ebfi::as_stream(stream);
    DcnDims d = d_in;
    const char *impl = getenv("EBFI_DCN_IMPL");
    // the tensor-core backward stages grad_output with 128-bit loads (8 pixels: two for fp32, one for bf16 / fp16, when a
    // row is a whole number of 16-byte words): it needs a 16-byte aligned base for either element size
    const bool tc_ok = !(impl && impl[0] == 's') && ebfi::aligned16(grad_output);
    // box kernel (dcn_bwd_box.cu) first; the group-specialised kernel (dcn_bwd_tc.cu) serves the deterministic flag
    const int S_box = tc_ok ? backward_box_splits(d) : 0;
    if (!std::is_same_v<T, float> && S_box == 0)
        return ebfi::fail(EBFI_ERR_UNSUPPORTED, "dcn_backward_%s: no box backward for this call (shape, flags or alignment)",
                          act_name<T>());
    const int S_tc = S_box > 0 ? S_box : (tc_ok ? backward_tc_splits(d) : 0);
    const int S = S_tc > 0 ? S_tc : bwd_splits(d);
    if (d.in_blocked) {
        EBFI_REQUIRE(S_box > 0, "dcn_backward: EBFI_DCN_INPUT_BLOCKED needs the box path (ebfi_dcnv2_blocked_input_offset() != 0 "
                                "and no EBFI_DCN_DETERMINISTIC)");
        EBFI_REQUIRE((reinterpret_cast<uintptr_t>(input) & 31u) == 0, "dcn_backward: the blocked input must be 32-byte aligned");
    }
    const size_t n_w = (size_t)d.Co * d.C * d.KK, n_b = (size_t)d.Co;
    const size_t n_in = (size_t)d.B * d.C * d.H * d.W;
    // workspace: [grad_weight / grad_bias partials][scratch][deterministic mode: 3-float bound]
    const size_t part_bytes = ebfi::round_up((size_t)S * (n_w + n_b) * sizeof(float), (size_t)256);
    const size_t scratch_bytes = ebfi::round_up(
        S_box > 0 ? backward_box_scratch_bytes(d) : S_tc > 0 ? backward_tc_scratch_bytes(d) : (d.det ? n_in * sizeof(long long) : 0),
        (size_t)256);
    const size_t need = part_bytes + scratch_bytes + (d.det ? 256 : 0);
    if (!workspace || workspace_bytes < need)
        return ebfi::fail(EBFI_ERR_WORKSPACE, "dcn_backward: workspace %zu < %zu bytes", workspace_bytes, need);
    // the blocked copies inside the workspace are read with 256-bit loads and by TMA
    EBFI_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 31u) == 0, "dcn_backward: workspace must be 32-byte aligned");
    float *gw_part = static_cast<float *>(workspace);
    float *gb_part = gw_part + (size_t)S * n_w;
    char *scratch = static_cast<char *>(workspace) + part_bytes;
    if (S_box > 0) {
        // writes all five gradients, including its own fixed-order reduction of the weight-gradient partials
        return backward_box<T>(st, d, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                               grad_weight, grad_bias, gw_part, gb_part, scratch, dp, dp_defer);
    }
    if constexpr (!std::is_same_v<T, float>) {
        return EBFI_ERR_UNSUPPORTED;      // not reached: a 16-bit call without the box path returned above
    } else {
        if (d.det) {
            float *bound = reinterpret_cast<float *>(scratch + scratch_bytes);
            EBFI_CUDA_OK(cudaMemsetAsync(bound, 0, 3 * sizeof(float), st));
            dcn_det_bound<<<ebfi::sm_count() * 4, 256, 0, st>>>(grad_output, weight, mask, bound, d);
            EBFI_LAUNCH_OK("dcn_det_bound");
            d.det_bound = bound;
        }
        if (S_tc > 0) {
            // tensor-core path (dcn_bwd_tc.cu): cpg == 8, Cout == 64
            if (int rc = backward_tc(st, d, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                                     gw_part, gb_part, S, scratch))
                return rc;
        } else {
            // deterministic mode accumulates into an int64 NCHW copy in the scratch and converts at the end
            float *gin_acc = d.det ? reinterpret_cast<float *>(scratch) : grad_input;
            EBFI_CUDA_OK(cudaMemsetAsync(gin_acc, 0, n_in * (d.det ? sizeof(long long) : sizeof(float)), st));
            EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
            EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
            const int n_cot = ceil_div(d.Co, COT);
            // Chunks of one group accumulate into the same grad_offset / grad_mask elements; separate,
            // stream-ordered launches keep that read-modify-write race-free. nchunk is 1 unless
            // channels-per-group * taps exceeds the KC_MAX-row slab.
            for (int ch = 0; ch < d.nchunk; ++ch) {
                dim3 grid(S, d.dg, n_cot);
                if (d.det)
                    dcn_bwd_kernel<true><<<grid, NT, kBwdSmem, st>>>(input, weight, offset, mask, grad_output, gin_acc,
                                                                     grad_offset, grad_mask, gw_part, gb_part, d, ch);
                else
                    dcn_bwd_kernel<false><<<grid, NT, kBwdSmem, st>>>(input, weight, offset, mask, grad_output, gin_acc,
                                                                      grad_offset, grad_mask, gw_part, gb_part, d, ch);
                EBFI_LAUNCH_OK("dcn_bwd_kernel");
            }
            if (d.det) {
                dcn_i64_to_f32<<<ebfi::sm_count() * 8, 256, 0, st>>>(reinterpret_cast<const long long *>(gin_acc), grad_input, n_in, d);
                EBFI_LAUNCH_OK("dcn_i64_to_f32");
            }
        }
        const int n = (int)(n_w + n_b);
        dcn_reduce_partials<<<ceil_div(n, 256), 256, 0, st>>>(gw_part, gb_part, grad_weight, grad_bias, S, (int)n_w, (int)n_b);
        EBFI_LAUNCH_OK("dcn_reduce_partials");
        if (dp) return ebfi_dp::allreduce_sum(st, *dp, grad_weight, n_w, grad_bias, n_b, dp_defer ? 1 : 0);
        return EBFI_OK;
    }
}

extern "C" {

int ebfi_dcnv2_forward(void *stream, const ebfi_dcn_geom *q, const float *input, const float *weight,
                       const float *bias, const float *offset, const float *mask, float *output,
                       void *workspace, size_t workspace_bytes)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    return run_forward(stream, d, input, weight, bias, offset, mask, output, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward(void *stream, const ebfi_dcn_geom *q, const float *input, const float *weight,
                        const float *bias, const float *offset, const float *mask,
                        const float *grad_output, float *grad_input, float *grad_offset,
                        float *grad_mask, float *grad_weight, float *grad_bias,
                        void *workspace, size_t workspace_bytes)
{
    (void)bias;
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    return run_backward(stream, d, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                        grad_weight, grad_bias, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_dp(void *stream, const ebfi_dcn_geom *q, const float *input, const float *weight,
                           const float *bias, const float *offset, const float *mask,
                           const float *grad_output, float *grad_input, float *grad_offset,
                           float *grad_mask, float *grad_weight, float *grad_bias,
                           void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer)
{
    (void)bias;
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    EBFI_REQUIRE(comm != nullptr, "dcn_backward_dp: null communicator");
    return run_backward(stream, d, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                        grad_weight, grad_bias, workspace, workspace_bytes, comm, defer != 0);
}

int ebfi_dcnv2_forward_packed(void *stream, const ebfi_dcn_geom *q, const float *input, const float *weight,
                              const float *bias, const float *offset_mask, float *output,
                              float *abs_offset_sum, void *workspace, size_t workspace_bytes)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    EBFI_REQUIRE(offset_mask != nullptr, "dcn_forward_packed: null pointer");
    const float *mask_logits = offset_mask + 2 * d.mask_bs;      // channels [2*dg*KK, 3*dg*KK) of sample 0
    set_packed(d);
    d.abs_sum = abs_offset_sum;
    return run_forward(stream, d, input, weight, bias, offset_mask, mask_logits, output, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_packed(void *stream, const ebfi_dcn_geom *q, const float *input, const float *weight,
                               const float *bias, const float *offset_mask, const float *grad_output,
                               float *grad_input, float *grad_offset_mask, float *grad_weight, float *grad_bias,
                               void *workspace, size_t workspace_bytes)
{
    (void)bias;
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    EBFI_REQUIRE(offset_mask && grad_offset_mask, "dcn_backward_packed: null pointer");
    const long long m0 = 2 * d.mask_bs;
    set_packed(d);
    return run_backward(stream, d, input, weight, offset_mask, offset_mask + m0, grad_output, grad_input,
                        grad_offset_mask, grad_offset_mask + m0, grad_weight, grad_bias, workspace, workspace_bytes);
}

}  // extern "C"

// ---- 16-bit activations (ebfi_b200.h, T = __nv_bfloat16 | __half): same geometry handling as the float entries above ----
template <typename T>
static int forward16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight, const float *bias,
                     const void *offset, const void *mask, void *output, void *workspace, size_t workspace_bytes)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    return run_forward(stream, d, static_cast<const T *>(input), weight, bias, static_cast<const T *>(offset),
                       static_cast<const T *>(mask), static_cast<T *>(output), workspace, workspace_bytes);
}

template <typename T>
static int backward16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                      const void *offset, const void *mask, const void *grad_output, void *grad_input,
                      void *grad_offset, void *grad_mask, float *grad_weight, float *grad_bias,
                      void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm = nullptr, int defer = 0)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    return run_backward(stream, d, static_cast<const T *>(input), weight, static_cast<const T *>(offset),
                        static_cast<const T *>(mask), static_cast<const T *>(grad_output), static_cast<T *>(grad_input),
                        static_cast<T *>(grad_offset), static_cast<T *>(grad_mask), grad_weight, grad_bias,
                        workspace, workspace_bytes, comm, defer != 0);
}

template <typename T>
static int forward_packed16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                            const float *bias, const void *offset_mask, void *output, float *abs_offset_sum,
                            void *workspace, size_t workspace_bytes)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    EBFI_REQUIRE(offset_mask != nullptr, "dcn_forward_packed: null pointer");
    const T *om = static_cast<const T *>(offset_mask);
    const T *mask_logits = om + 2 * d.mask_bs;
    set_packed(d);
    d.abs_sum = abs_offset_sum;
    return run_forward(stream, d, static_cast<const T *>(input), weight, bias, om, mask_logits, static_cast<T *>(output),
                       workspace, workspace_bytes);
}

template <typename T>
static int backward_packed16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                             const void *offset_mask, const void *grad_output, void *grad_input,
                             void *grad_offset_mask, float *grad_weight, float *grad_bias,
                             void *workspace, size_t workspace_bytes)
{
    DcnDims d{};
    if (int rc = fill_dims(q, d)) return rc;
    EBFI_REQUIRE(offset_mask && grad_offset_mask, "dcn_backward_packed: null pointer");
    const long long m0 = 2 * d.mask_bs;
    set_packed(d);
    const T *om = static_cast<const T *>(offset_mask);
    T *gom = static_cast<T *>(grad_offset_mask);
    return run_backward(stream, d, static_cast<const T *>(input), weight, om, om + m0, static_cast<const T *>(grad_output),
                        static_cast<T *>(grad_input), gom, gom + m0, grad_weight, grad_bias, workspace, workspace_bytes);
}

extern "C" {

int ebfi_dcnv2_forward_bf16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                            const float *bias, const void *offset, const void *mask, void *output,
                            void *workspace, size_t workspace_bytes)
{
    return forward16<__nv_bfloat16>(stream, q, input, weight, bias, offset, mask, output, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_bf16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                             const float *bias, const void *offset, const void *mask,
                             const void *grad_output, void *grad_input, void *grad_offset,
                             void *grad_mask, float *grad_weight, float *grad_bias,
                             void *workspace, size_t workspace_bytes)
{
    (void)bias;
    return backward16<__nv_bfloat16>(stream, q, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                           grad_weight, grad_bias, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_dp_bf16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                const float *bias, const void *offset, const void *mask,
                                const void *grad_output, void *grad_input, void *grad_offset,
                                void *grad_mask, float *grad_weight, float *grad_bias,
                                void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer)
{
    (void)bias;
    EBFI_REQUIRE(comm != nullptr, "dcn_backward_dp: null communicator");
    return backward16<__nv_bfloat16>(stream, q, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                           grad_weight, grad_bias, workspace, workspace_bytes, comm, defer);
}

int ebfi_dcnv2_forward_packed_bf16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                   const float *bias, const void *offset_mask, void *output,
                                   float *abs_offset_sum, void *workspace, size_t workspace_bytes)
{
    return forward_packed16<__nv_bfloat16>(stream, q, input, weight, bias, offset_mask, output, abs_offset_sum, workspace,
                                 workspace_bytes);
}

int ebfi_dcnv2_backward_packed_bf16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                    const float *bias, const void *offset_mask, const void *grad_output,
                                    void *grad_input, void *grad_offset_mask, float *grad_weight, float *grad_bias,
                                    void *workspace, size_t workspace_bytes)
{
    (void)bias;
    return backward_packed16<__nv_bfloat16>(stream, q, input, weight, offset_mask, grad_output, grad_input, grad_offset_mask,
                                  grad_weight, grad_bias, workspace, workspace_bytes);
}

int ebfi_dcnv2_forward_fp16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                            const float *bias, const void *offset, const void *mask, void *output,
                            void *workspace, size_t workspace_bytes)
{
    return forward16<__half>(stream, q, input, weight, bias, offset, mask, output, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_fp16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                             const float *bias, const void *offset, const void *mask,
                             const void *grad_output, void *grad_input, void *grad_offset,
                             void *grad_mask, float *grad_weight, float *grad_bias,
                             void *workspace, size_t workspace_bytes)
{
    (void)bias;
    return backward16<__half>(stream, q, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                           grad_weight, grad_bias, workspace, workspace_bytes);
}

int ebfi_dcnv2_backward_dp_fp16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                const float *bias, const void *offset, const void *mask,
                                const void *grad_output, void *grad_input, void *grad_offset,
                                void *grad_mask, float *grad_weight, float *grad_bias,
                                void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer)
{
    (void)bias;
    EBFI_REQUIRE(comm != nullptr, "dcn_backward_dp: null communicator");
    return backward16<__half>(stream, q, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask,
                           grad_weight, grad_bias, workspace, workspace_bytes, comm, defer);
}

int ebfi_dcnv2_forward_packed_fp16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                   const float *bias, const void *offset_mask, void *output,
                                   float *abs_offset_sum, void *workspace, size_t workspace_bytes)
{
    return forward_packed16<__half>(stream, q, input, weight, bias, offset_mask, output, abs_offset_sum, workspace,
                                 workspace_bytes);
}

int ebfi_dcnv2_backward_packed_fp16(void *stream, const ebfi_dcn_geom *q, const void *input, const float *weight,
                                    const float *bias, const void *offset_mask, const void *grad_output,
                                    void *grad_input, void *grad_offset_mask, float *grad_weight, float *grad_bias,
                                    void *workspace, size_t workspace_bytes)
{
    (void)bias;
    return backward_packed16<__half>(stream, q, input, weight, offset_mask, grad_output, grad_input, grad_offset_mask,
                                  grad_weight, grad_bias, workspace, workspace_bytes);
}

}  // extern "C"
