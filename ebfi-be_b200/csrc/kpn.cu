// kpn.cu — KernelConv producer -> FAC consumer, fused forward (SURVEY §8f rank 1).
//
// Reference op sequence (models/Ours/model_singleframe.py:145-146,159-162, class Modification):
//     Kernel = LeakyReLU(conv3x3(cat([Event, Frame], 1)))          # ConvLayer, (B, Ce*K*K, H, W): 1.68 GB at cfg2
//     out    = KernelConv2D(K)(Event, Kernel)                      # ReplicationPad2d((K-1)/2) + FAC
// The per-pixel kernel tensor is written once and read once; fused, it never exists in HBM: the 3x3
// convolution is an implicit GEMM on the tcgen05 tensor cores whose accumulator (TMEM) is consumed in place
// by the FAC contraction.
//
// Mapping: WEIGHT-STATIONARY. The conv's output channels are cut into slices of 3 FAC channels x K*K taps
// (75 GEMM columns, N = 80); the slice's weights for all 9 x Cin reduction steps (184 KB as bf16) stay in
// shared memory while the CTA streams pixel tiles through them — the opposite arrangement (pixel tile
// stationary, weights streamed) needs ~60 B/clk/SM of weight traffic from L2 and is bandwidth-bound there.
// Work items = (slice, pixel tile) in slice-major order, split evenly over one persistent CTA per SM; a CTA
// reloads weights only when its range crosses a slice boundary.
//   tile        16 rows x 8 columns = 128 pixels = M (one TMEM lane per pixel)
//   A operand   the tile's input halo (18 x 10 pixels x Cin) in shared memory, laid out [8-ch chunk][y][x][8 ch]
//               (bf16); for tap (dy, dx) the UMMA descriptor simply starts (dy*10 + dx) pixels later, with
//               SBO = one halo row and LBO = one chunk plane: no im2col copy of any kind
//   B operand   weights [80 rows][9*Cin], K-major, K order = (32-channel part, tap, 16-channel step)
//   pipeline    the halo is held as Cin/32 channel PARTS (32 channels, 11.5 KB each). One producer lane refills a
//               part for the next tile with a single 3-D TMA tensor copy (zero fill outside the image = the
//               conv's padding) as soon as the MMAs that read it have completed, while the other parts compute;
//               two TMEM accumulators let the epilogue of item i overlap the MMAs of item i+1
//   epilogue    three warpgroups, one per FAC channel of the slice; thread = (pixel, channel): its 25 Event window
//               values are fetched BEFORE it waits for the accumulator, then 25 accumulators -> + bias -> LeakyReLU
//               -> x Event[c][clamp(y+ky-2)][clamp(x+kx-2)], summed in the reference's tap order
//               (KernelConv2D_kernel.cu:44-50) -> 1 output. (With one warpgroup doing all 75 columns after the
//               wait, the epilogue's load latency was the bottleneck: tensor pipe 42 % busy.)
//   waiting     the MMA warp spins on its barriers with all lanes (critical path); epilogue and producer warps wait
//               with ONE polling lane and a suspend hint and arrive once per warp: at N = 80 the tensor core needs
//               every shared-memory cycle for its operands (128 x 80 x 16 MMA: 52 clk = 32 for A + 20 for B), and
//               400 threads spinning on mbarrier.try_wait take some of them away
//
// Precision: tensors are fp32 at the boundary (like the reference); the conv operands are rounded to bf16
// for the tensor cores, accumulation and the whole FAC part are fp32. Stated tolerance 1e-2 of max|out|
// against the fp32/fp64 op sequence; 1e-5 against the same sequence with bf16-rounded conv operands.
// Activation I/O (event / frame / output, and grad_output / grad_pre in the backward) may instead be bf16 or fp16
// (template parameter T, the *_bf16 / *_fp16 entries): only the loads convert (exactly) and the stores round once (RN)
// from the same fp32 values, so on bf16- or fp16-valued inputs such an instantiation computes bit-identically to the
// fp32 one. The conv operands are bf16 for every T. Weights, bias, grad_event_fac and grad_bias stay fp32.
//
// Backward (ebfi_kpn_fused_backward): the same kernel with BWD = true recomputes the pre-activation P in TMEM
// through the identical main loop (same operands, same MMA chain -> bit-identical P, so forward and backward take
// the same LeakyReLU branch everywhere) and replaces the FAC epilogue by its gradient. Thread = (pixel, channel):
//   gP[c*KK+t, p]  = G[c,p] * Epad[c,p+t] * (P > 0 ? 1 : slope)      written NCHW (type T) = cuDNN's dgrad/wgrad input
//   gEpad[c, q]   += LeakyReLU(P)[c*KK+t, q-t] * G[c, q-t]            per-warp box in unclamped Epad coordinates
//   grad_bias      = per-lane running column sums of gP over the CTA's items of a slice
// gEpad: a warp holds 4 x 8 pixels, i.e. an (4+K-1) x (8+K-1) box of Epad cells, <= 3 per lane. For a fixed tap every
// cell has at most one source pixel, so its owner lane pulls the value with one shuffle: 3 shuffles per tap, summed
// in tap order. The boxes go to the workspace (every cell is covered by <= 4 boxes); kpn_gev_collect sums the boxes
// of a cell in a fixed order and folds the replication border. kpn_bias_collect sums the column partials of the
// CTAs of a slice in CTA order. No float atomics anywhere: the outputs are bit-reproducible for a given grid.
#include "common.cuh"
#include "tma.cuh"
#include "umma.cuh"

#include <algorithm>
#include <cuda_fp16.h>

namespace {

using ebfi::ceil_div;

constexpr int TH = 16, TW = 8, TM = TH * TW;     // pixel tile
constexpr int HH = TH + 2, HW = TW + 2;          // conv halo (3x3, pad 1)
constexpr int HPIX = HH * HW;                    // 180 halo pixels
constexpr int CPS = 3;                           // FAC channels per weight slice
constexpr int NEPI = CPS * 128;                  // epilogue threads: one warpgroup (128 TMEM lanes) per FAC channel of the slice
constexpr int NTHR = NEPI + 64;                  // + 1 TMA producer warp + 1 MMA warp
constexpr int PART_CH = 32;                      // channels per halo part = two K = 16 MMA steps per tap
constexpr int PART_BYTES = (PART_CH / 8) * HPIX * 16;
constexpr int TMEM_COLS = 256;                   // two accumulators at columns 0 and 128
constexpr int WR = 4;                            // pixel rows per epilogue warp (32 lanes = WR x TW pixels)
constexpr int BWD_MAX_GRID = 1024;               // backward grid cap: sizes the bias partials without a device query

struct KpnDims {
    int B, Ce, Cin, H, W, K, KK;
    int nslice, NP;              // weight slices; GEMM N (padded to 16) of a full slice
    int tiles_x, tiles_y, ntile; // pixel tiles per sample row / column, per call
    int Ktot, kchunks;           // 9 * Cin; Cin / 8
    int npart;                   // Cin / 32 halo parts
    int w_bytes;
    float slope;
};

// Activation element type T (float | __nv_bfloat16 | __half): loads widen to fp32 exactly, stores round once (RN; an
// fp16 store overflows to +-inf, as tensor.half() does).
__device__ __forceinline__ float ld_act(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ld_act(const __nv_bfloat16 *p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ld_act(const __half *p) { return __half2float(__ldg(p)); }
template <typename T> __device__ __forceinline__ T st_act(float v);
template <> __device__ __forceinline__ float st_act<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 st_act<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half st_act<__half>(float v) { return __float2half_rn(v); }

// Backward-only operands of the fused kernel (unused by the forward instantiation).
template <typename T>
struct KpnBwdArgs {
    const T *gout;          // (B, Ce, H, W) dL/dout
    T *gpre;                // (B, Ce*KK, H, W) dL/dP
    float *gbox;            // [B][Ce][tiles_y*TH/WR][tiles_x][WR+K-1][TW+K-1] per-warp dL/dEpad boxes
    float *bias_part;       // [CTA + slice][NEPI/32 warps][KK] column sums of dL/dP
};

// (ev | fr) NCHW T -> [b][chunk of 8 channels][y][x][8] bf16: one thread per (b, chunk, y, x)
template <typename T>
__global__ void kpn_prep_input(const T *__restrict__ ev, const T *__restrict__ fr, __nv_bfloat16 *__restrict__ dst,
                               KpnDims d)
{
    const size_t plane = (size_t)d.H * d.W, n = (size_t)d.B * d.kchunks * plane;
    const int Cf = d.Cin - d.Ce;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t px = i % plane, bk = i / plane;
        const int kc = (int)(bk % d.kchunks), b = (int)(bk / d.kchunks);
        unsigned short v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ch = kc * 8 + e;
            const float x = ch < d.Ce ? ld_act(ev + ((size_t)b * d.Ce + ch) * plane + px)
                                      : ld_act(fr + ((size_t)b * Cf + (ch - d.Ce)) * plane + px);
            v[e] = __bfloat16_as_ushort(__float2bfloat16_rn(x));
        }
        *reinterpret_cast<uint4 *>(dst + i * 8) = make_uint4(v[0] | ((uint32_t)v[1] << 16), v[2] | ((uint32_t)v[3] << 16),
                                                             v[4] | ((uint32_t)v[5] << 16), v[6] | ((uint32_t)v[7] << 16));
    }
}

// conv weight (Ce*KK, Cin, 3, 3) fp32 -> per slice the shared-memory image [NP/8][Ktot/8][8 rows][8 k] bf16,
// K order: chunk index = (part * 9 + tap) * 4 + j  <->  channel part * 32 + j*8 + e
__global__ void kpn_prep_weights(const float *__restrict__ w, __nv_bfloat16 *__restrict__ wimg, KpnDims d)
{
    const int per = d.NP * d.Ktot;
    const int kch = d.Ktot / 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.nslice * per; i += gridDim.x * blockDim.x) {
        const int s = i / per, e0 = i - s * per;
        const int e = e0 & 7, r = (e0 >> 3) & 7, rest = e0 >> 6;
        const int kc = rest % kch, rg = rest / kch;
        const int nrow = rg * 8 + r;
        const int j = kc % 4, pt = kc / 4, tap = pt % 9, part = pt / 9;
        const int ch = part * PART_CH + j * 8 + e;
        const int c0 = s * CPS, ncols = min(CPS, d.Ce - c0) * d.KK;
        float v = 0.f;
        if (nrow < ncols) v = __ldg(w + ((size_t)(c0 * d.KK + nrow) * d.Cin + ch) * 9 + tap);
        wimg[i] = __float2bfloat16_rn(v);
    }
}

// Epilogue of warpgroup G: FAC channel c0 + G of every item's slice.
template <int K, int G, typename T>
__device__ __forceinline__ void kpn_epilogue(uint32_t tmem, uint64_t *acc_full, uint64_t *acc_free,
                                             const float *__restrict__ bias, const T *__restrict__ ev,
                                             T *__restrict__ out, const KpnDims &d, int item0, int item1)
{
    constexpr int KK = K * K, R = (K - 1) / 2;
    constexpr int COL0 = (G * KK / 8) * 8, OFF = G * KK - COL0, NLD = (OFF + KK + 7) / 8;   // 8-column TMEM loads covering the channel
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = (warp & 3) * 32 + lane, py = p / TW, px = p % TW;
    const uint32_t lane_base = (uint32_t)(warp & 3) * 32u;
    const size_t plane = (size_t)d.H * d.W;
    const int tiles_per_sample = d.tiles_x * d.tiles_y;
    float bv[KK];
    int bias_slice = -1;
    for (int item = item0, n = 0; item < item1; ++item, ++n) {
        const int s = item / d.ntile, t = item % d.ntile;
        const int b = t / tiles_per_sample, tt = t % tiles_per_sample;
        const int y = (tt / d.tiles_x) * TH + py, x = (tt % d.tiles_x) * TW + px;
        const int c = s * CPS + G;
        const bool active = c < d.Ce;                        // warp-uniform: the last slice may hold fewer channels
        const bool valid = active && y < d.H && x < d.W;
        // Event window of this pixel: independent of the accumulator -> in flight while waiting for it
        float e[KK];
        if (valid) {
            const T *evc = ev + ((size_t)b * d.Ce + c) * plane;
            int xo[K];
#pragma unroll
            for (int kx = 0; kx < K; ++kx) xo[kx] = min(max(x + kx - R, 0), d.W - 1);   // ReplicationPad2d (KernelConv2D.py:82-86)
#pragma unroll
            for (int ky = 0; ky < K; ++ky) {
                const T *row = evc + (size_t)min(max(y + ky - R, 0), d.H - 1) * d.W;
#pragma unroll
                for (int kx = 0; kx < K; ++kx) e[ky * K + kx] = ld_act(row + xo[kx]);
            }
        }
        if (active && s != bias_slice) {
#pragma unroll
            for (int q = 0; q < KK; ++q) bv[q] = __ldg(bias + c * KK + q);
            bias_slice = s;
        }
        const int buf = n & 1;
        umma::mbar_wait_warp(&acc_full[buf], (uint32_t)((n >> 1) & 1));
        umma::fence_after_sync();
        float v[NLD * 8];
        if (active) {
#pragma unroll
            for (int q = 0; q < NLD; ++q) {
                float (&vq)[8] = *reinterpret_cast<float (*)[8]>(&v[q * 8]);
                umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, buf * 128 + COL0 + q * 8), vq);
            }
            umma::tmem_ld_wait();
        }
        umma::fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&acc_free[buf]);    // accumulator drained into registers (one arrival per warp): the next item may reuse it
        if (valid) {
            float res = 0.f;
#pragma unroll
            for (int q = 0; q < KK; ++q) {                   // tap order of KernelConv2D_kernel.cu:44-50
                float a = v[OFF + q] + bv[q];
                a = a > 0.f ? a : a * d.slope;               // nn.LeakyReLU
                res += e[q] * a;
            }
            out[((size_t)b * d.Ce + c) * plane + (size_t)y * d.W + x] = st_act<T>(res);
        }
    }
}

// Backward epilogue of warpgroup G (see the header comment): gP, the warp's dL/dEpad box, bias column sums.
template <int K, int G, typename T>
__device__ __forceinline__ void kpn_bwd_epilogue(uint32_t tmem, uint64_t *acc_full, uint64_t *acc_free,
                                                 const float *__restrict__ bias, const T *__restrict__ ev,
                                                 const KpnBwdArgs<T> &a, const KpnDims &d, int item0, int item1)
{
    constexpr int KK = K * K, R = (K - 1) / 2;
    constexpr int COL0 = (G * KK / 8) * 8, OFF = G * KK - COL0, NLD = (OFF + KK + 7) / 8;
    constexpr int BH = WR + K - 1, BW = TW + K - 1, BOX = BH * BW, NCELL = (BOX + 31) / 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wq = warp & 3;
    const int p = wq * 32 + lane, py = p / TW, px = p % TW;
    const uint32_t lane_base = (uint32_t)wq * 32u;
    const size_t plane = (size_t)d.H * d.W;
    const int tiles_per_sample = d.tiles_x * d.tiles_y;
    const int wrows = d.tiles_y * (TH / WR);
    // owned box cell j = lane + 32 j at (cy, cx): for tap (ky, kx) its source pixel is lane (cy - ky) * TW + (cx - kx)
    // = cbase[j] - (ky * TW + kx), if that pixel lies in the warp's WR x TW block: bit q of cmask[j]
    int cbase[NCELL];
    uint32_t cmask[NCELL];
#pragma unroll
    for (int j = 0; j < NCELL; ++j) {
        const int cy = (lane + 32 * j) / BW, cx = (lane + 32 * j) % BW;
        cbase[j] = cy * TW + cx;
        cmask[j] = 0;
        for (int q = 0; q < KK; ++q) {
            const int sy = cy - q / K, sx = cx - q % K;
            if (lane + 32 * j < BOX && sy >= 0 && sy < WR && sx >= 0 && sx < TW) cmask[j] |= 1u << q;
        }
    }
    // the slice's bias column of this warp in shared memory (broadcast reads): registers are the scarce resource
    // here, the epilogue already holds the Event window, the accumulators and the bias column sums
    __shared__ float bias_s[4][KK];
    float bsum[KK];
    int cur_slice = -1;
    auto flush = [&](int s) {                                // warp column sums -> bias_part[CTA + slice][warp]
#pragma unroll
        for (int q = 0; q < KK; ++q) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) bsum[q] += __shfl_xor_sync(0xffffffffu, bsum[q], o);
        }
        if (lane == 0) {
            float *dst = a.bias_part + ((size_t)(blockIdx.x + s) * (NEPI / 32) + warp) * KK;
#pragma unroll
            for (int q = 0; q < KK; ++q) dst[q] = bsum[q];
        }
    };
    for (int item = item0, n = 0; item < item1; ++item, ++n) {
        const int s = item / d.ntile, t = item % d.ntile;
        const int b = t / tiles_per_sample, tt = t % tiles_per_sample;
        const int tyi = tt / d.tiles_x, txi = tt % d.tiles_x;
        const int y = tyi * TH + py, x = txi * TW + px;
        const int c = s * CPS + G;
        const bool active = c < d.Ce;                        // warp-uniform
        const bool valid = active && y < d.H && x < d.W;
        if (s != cur_slice) {
            if (cur_slice >= 0 && cur_slice * CPS + G < d.Ce) flush(cur_slice);
            cur_slice = s;
            if (active) {
                __syncwarp();
                if (lane < KK) bias_s[wq][lane] = __ldg(bias + c * KK + lane);
                __syncwarp();
#pragma unroll
                for (int q = 0; q < KK; ++q) bsum[q] = 0.f;
            }
        }
        float e[KK], g = 0.f;
        if (valid) {
            const T *evc = ev + ((size_t)b * d.Ce + c) * plane;
            int xo[K];
#pragma unroll
            for (int kx = 0; kx < K; ++kx) xo[kx] = min(max(x + kx - R, 0), d.W - 1);
#pragma unroll
            for (int ky = 0; ky < K; ++ky) {
                const T *row = evc + (size_t)min(max(y + ky - R, 0), d.H - 1) * d.W;
#pragma unroll
                for (int kx = 0; kx < K; ++kx) e[ky * K + kx] = ld_act(row + xo[kx]);
            }
            g = ld_act(a.gout + ((size_t)b * d.Ce + c) * plane + (size_t)y * d.W + x);
        }
        const int buf = n & 1;
        umma::mbar_wait_warp(&acc_full[buf], (uint32_t)((n >> 1) & 1));
        umma::fence_after_sync();
        float v[NLD * 8];
        if (active) {
#pragma unroll
            for (int q = 0; q < NLD; ++q) {
                float (&vq)[8] = *reinterpret_cast<float (*)[8]>(&v[q * 8]);
                umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, buf * 128 + COL0 + q * 8), vq);
            }
            umma::tmem_ld_wait();
        }
        umma::fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&acc_free[buf]);
        if (active) {
            float box[NCELL];
#pragma unroll
            for (int j = 0; j < NCELL; ++j) box[j] = 0.f;
            T *gp = a.gpre + ((size_t)b * d.Ce * KK + (size_t)c * KK) * plane + (size_t)y * d.W + x;
#pragma unroll
            for (int q = 0; q < KK; ++q) {
                const float pre = v[OFF + q] + bias_s[wq][q];   // bit-identical to the forward's accumulator + bias
                const bool pos = pre > 0.f;
                float kg = 0.f;                              // LeakyReLU(P) * G: this pixel's dL/dEpad term of tap q
                if (valid) {
                    const float ge = g * e[q];               // dL/dKernel (KernelConv2D backward)
                    const float gpq = pos ? ge : ge * d.slope;   // leaky_relu_backward: P == 0 takes the slope
                    __stcs(gp + (size_t)q * plane, st_act<T>(gpq));   // bias sums use the unrounded gpq
                    bsum[q] += gpq;
                    kg = (pos ? pre : pre * d.slope) * g;
                }
#pragma unroll
                for (int j = 0; j < NCELL; ++j) {        // the lane index wraps mod 32 where the cell has no source
                    const float pulled = __shfl_sync(0xffffffffu, kg, cbase[j] - ((q / K) * TW + q % K));
                    if ((cmask[j] >> q) & 1u) box[j] += pulled;
                }
            }
            float *dst = a.gbox + ((((size_t)b * d.Ce + c) * wrows + tyi * (TH / WR) + wq) * d.tiles_x + txi) * BOX;
#pragma unroll
            for (int j = 0; j < NCELL; ++j)
                if (lane + 32 * j < BOX) dst[lane + 32 * j] = box[j];
        }
    }
    if (cur_slice >= 0 && cur_slice * CPS + G < d.Ce) flush(cur_slice);
}

// K: FAC kernel size; NPART: halo parts = Cin / 32; BWD: backward epilogue (bw) instead of the FAC one (out);
// T: activation element type of ev / out / bw.gout / bw.gpre
template <int K, int NPART, bool BWD, typename T>
__global__ void __launch_bounds__(NTHR, 1)
kpn_fused_kernel(const __grid_constant__ CUtensorMap tmap, const __nv_bfloat16 *__restrict__ wimg,
                 const float *__restrict__ bias, const T *__restrict__ ev, T *__restrict__ out,
                 KpnBwdArgs<T> bw, KpnDims d, int items_per_cta)
{
    constexpr int KK = K * K, R = (K - 1) / 2;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *w_s = smem;                               // weight slice
    unsigned char *a_s = smem + d.w_bytes;                   // NPART channel parts of the halo tile
    __shared__ __align__(8) uint64_t bar_w, bar_wfree, a_full[NPART], a_free[NPART], acc_full[2], acc_free[2];
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int total = d.nslice * d.ntile;
    const int item0 = blockIdx.x * items_per_cta, item1 = min(total, item0 + items_per_cta);

    if (warp == 0) umma::tmem_alloc<TMEM_COLS>(&tmem_slot);
    if (tid == 0) {
        umma::mbar_init(&bar_w, 1);
        umma::mbar_init(&bar_wfree, 1);
        for (int i = 0; i < NPART; ++i) { umma::mbar_init(&a_full[i], 1); umma::mbar_init(&a_free[i], 1); }
        for (int i = 0; i < 2; ++i) { umma::mbar_init(&acc_full[i], 1); umma::mbar_init(&acc_free[i], NEPI / 32); }
        umma::mbar_fence_init();
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const int tiles_per_sample = d.tiles_x * d.tiles_y;

    if (warp == NEPI / 32 + 1) {
        // ===================== MMA issue + weight loads =====================
        // All 32 lanes run this loop with warp-uniform values (descriptor arithmetic stays on the uniform
        // datapath); only the tcgen05 / bulk-copy / commit instructions themselves are issued by one elected
        // lane. With `if (lane == 0)` around the whole loop the issue cost was ~40 instructions per MMA and the
        // tensor pipe sat idle 77 % of the time (profiles/README.md).
        const bool leader = umma::elect_one();
        int cur_slice = -1, nw = 0;
        const uint32_t w_sbo = (uint32_t)(36 * NPART) * 128u;              // Ktot / 8 = 9 * Cin / 8 chunks of 128 bytes
        // descriptors differ only in their 16-byte-granular start address (low 14 bits): build once, add offsets
        const uint64_t da0 = umma::smem_desc(umma::smem_u32(a_s), HPIX * 16u, HW * 16u);
        const uint64_t db0 = umma::smem_desc(umma::smem_u32(w_s), 128u, w_sbo);
        for (int item = item0, n = 0; item < item1; ++item, ++n) {
            const int s = item / d.ntile;
            const int ncols = min(CPS, d.Ce - s * CPS) * KK;
            const uint32_t idesc = umma::instr_desc_bf16(TM, (ncols + 15) & ~15);
            if (s != cur_slice) {
                if (cur_slice >= 0) {                        // every MMA that reads the old weights has completed
                    if (leader) umma::commit(&bar_wfree);
                    umma::mbar_wait(&bar_wfree, (uint32_t)((nw - 1) & 1));
                }
                if (leader) {
                    umma::mbar_expect_tx(&bar_w, (uint32_t)d.w_bytes);
                    const unsigned char *src = reinterpret_cast<const unsigned char *>(wimg) + (size_t)s * d.w_bytes;
                    const int piece = d.w_bytes / 8;
                    for (int q = 0; q < 8; ++q) umma::bulk_g2s(w_s + q * piece, src + (size_t)q * piece, (uint32_t)piece, &bar_w);
                }
                umma::mbar_wait(&bar_w, (uint32_t)(nw & 1));
                ++nw;
                cur_slice = s;
            }
            const int buf = n & 1;
            umma::mbar_wait(&acc_free[buf], (uint32_t)(((n >> 1) & 1) ^ 1));   // epilogue of item n-2 has drained it
            umma::fence_after_sync();
            const uint32_t dcol = tmem + (uint32_t)buf * 128u;
#pragma unroll
            for (int part = 0; part < NPART; ++part) {
                umma::mbar_wait(&a_full[part], (uint32_t)(n & 1));
                umma::fence_after_sync();
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint64_t da = da0 + (uint64_t)(part * (PART_BYTES / 16) + (tap / 3) * HW + (tap % 3) + j * 2 * HPIX);
                        const uint64_t db = db0 + (uint64_t)(((part * 9 + tap) * 2 + j) * 16);
                        if (leader) umma::mma_f16(dcol, da, db, idesc, (part | tap | j) != 0);
                    }
                }
                if (leader) umma::commit(&a_free[part]);     // this part may be refilled for the next item
            }
            if (leader) umma::commit(&acc_full[buf]);
            __syncwarp();
        }
    } else if (warp == NEPI / 32) {
        // ===================== producer warp: one TMA tensor copy per (item, part) =====================
        const bool leader = umma::elect_one();
        for (int item = item0, n = 0; item < item1; ++item, ++n) {
            const int t = item % d.ntile;
            const int b = t / tiles_per_sample, tt = t % tiles_per_sample;
            const int ty0 = (tt / d.tiles_x) * TH, tx0 = (tt % d.tiles_x) * TW;
#pragma unroll
            for (int part = 0; part < NPART; ++part) {
                umma::mbar_wait_warp(&a_free[part], (uint32_t)((n & 1) ^ 1));
                if (leader) {
                    umma::mbar_expect_tx(&a_full[part], (uint32_t)PART_BYTES);
                    tma::load_3d(a_s + part * PART_BYTES, &tmap, (tx0 - 1) * 8, ty0 - 1, b * d.kchunks + part * (PART_CH / 8),
                                &a_full[part]);
                }
            }
            __syncwarp();
        }
    } else {
        // ===================== epilogue warpgroups: thread = (pixel = TMEM lane, FAC channel G of the slice) ==========
        const int g = warp >> 2;
        if constexpr (BWD) {
            if (g == 0) kpn_bwd_epilogue<K, 0, T>(tmem, acc_full, acc_free, bias, ev, bw, d, item0, item1);
            else if (g == 1) kpn_bwd_epilogue<K, 1, T>(tmem, acc_full, acc_free, bias, ev, bw, d, item0, item1);
            else kpn_bwd_epilogue<K, 2, T>(tmem, acc_full, acc_free, bias, ev, bw, d, item0, item1);
        } else {
            if (g == 0) kpn_epilogue<K, 0, T>(tmem, acc_full, acc_free, bias, ev, out, d, item0, item1);
            else if (g == 1) kpn_epilogue<K, 1, T>(tmem, acc_full, acc_free, bias, ev, out, d, item0, item1);
            else kpn_epilogue<K, 2, T>(tmem, acc_full, acc_free, bias, ev, out, d, item0, item1);
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tmem);
}

// dL/dEvent (FAC + ReplicationPad part): thread = one event cell (b, c, y, x). It sums the Epad cells that the
// replication pad maps onto it (one in the interior, up to (R+1)^2 in a corner), each from the <= 2 x 2 warp boxes
// that cover it, in a fixed order.
__global__ void kpn_gev_collect(const float *__restrict__ gbox, float *__restrict__ gev, KpnDims d)
{
    const int R = (d.K - 1) / 2, BH = WR + d.K - 1, BW = TW + d.K - 1, box = BH * BW;
    const int wrows = d.tiles_y * (TH / WR);
    const size_t plane = (size_t)d.H * d.W, n = (size_t)d.B * d.Ce * plane;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H);
        const size_t bc = i / plane;
        const int y0 = y == 0 ? 0 : y + R, y1 = y == d.H - 1 ? d.H - 1 + 2 * R : y + R;   // Epad rows folding onto y
        const int x0 = x == 0 ? 0 : x + R, x1 = x == d.W - 1 ? d.W - 1 + 2 * R : x + R;
        const float *base = gbox + bc * wrows * d.tiles_x * box;
        float acc = 0.f;
        for (int Y = y0; Y <= y1; ++Y) {
            const int r0 = Y >= BH ? (Y - BH + WR) / WR : 0, r1 = min(Y / WR, wrows - 1);
            for (int X = x0; X <= x1; ++X) {
                const int c0 = X >= BW ? (X - BW + TW) / TW : 0, c1 = min(X / TW, d.tiles_x - 1);
                for (int r = r0; r <= r1; ++r)
                    for (int cc = c0; cc <= c1; ++cc)
                        acc += __ldg(base + ((size_t)r * d.tiles_x + cc) * box + (Y - r * WR) * BW + (X - cc * TW));
            }
        }
        gev[i] = acc;
    }
}

// grad_bias[c*KK+q]: the warp partials of slice c / CPS, CTA by CTA (the CTAs whose item range meets the slice), then
// warp by warp.
__global__ void kpn_bias_collect(const float *__restrict__ part, float *__restrict__ gbias, KpnDims d, int per)
{
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= d.Ce * d.KK) return;
    const int c = col / d.KK, q = col % d.KK, s = c / CPS, g = c % CPS;
    const long k0 = (long)s * d.ntile / per, k1 = ((long)(s + 1) * d.ntile - 1) / per;
    float acc = 0.f;
    for (long k = k0; k <= k1; ++k)
        for (int w = 0; w < 4; ++w) acc += part[((size_t)(k + s) * (NEPI / 32) + g * 4 + w) * d.KK + q];
    gbias[col] = acc;
}

// featb [B*kchunks][H][W*8] bf16, box = one halo part: [4 chunks][18 rows][10 pixels * 8 channels]
int make_tmap(CUtensorMap &tm, const KpnDims &d, void *featb)
{
    const uint64_t gdim[3] = {(uint64_t)d.W * 8, (uint64_t)d.H, (uint64_t)d.B * d.kchunks};
    const uint64_t gstr[2] = {(uint64_t)d.W * 16, (uint64_t)d.H * d.W * 16};
    const uint32_t box[3] = {HW * 8, HH, PART_CH / 8};
    return tma::encode_3d(tm, featb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, gdim, gstr, box);
}

int fill(KpnDims &d, int B, int Ce, int Cf, int H, int W, int K, float slope)
{
    EBFI_REQUIRE(B > 0 && Ce > 0 && Cf >= 0 && H > 0 && W > 0, "kpn_fused: bad sizes");
    EBFI_REQUIRE(K >= 1 && (K & 1) && K * K * CPS <= 80, "kpn_fused: kernel_size must be odd and <= 5");
    d.B = B; d.Ce = Ce; d.Cin = Ce + Cf; d.H = H; d.W = W; d.K = K; d.KK = K * K; d.slope = slope;
    if (d.Cin % 32 != 0 || d.Cin > 128)
        return ebfi::fail(EBFI_ERR_UNSUPPORTED, "kpn_fused: event+frame channels (%d) must be a multiple of 32, <= 128", d.Cin);
    d.nslice = ceil_div(Ce, CPS);
    d.NP = ebfi::round_up(CPS * d.KK, 16);
    d.tiles_x = ceil_div(W, TW); d.tiles_y = ceil_div(H, TH);
    d.ntile = B * d.tiles_x * d.tiles_y;
    d.Ktot = 9 * d.Cin; d.kchunks = d.Cin / 8; d.npart = d.Cin / PART_CH;
    d.w_bytes = d.NP * d.Ktot * 2;
    EBFI_REQUIRE((long)d.nslice * d.ntile < (1L << 31), "kpn_fused: too many work items");
    return EBFI_OK;
}

size_t ws_weights(const KpnDims &d) { return ebfi::round_up((size_t)d.nslice * d.w_bytes, (size_t)256); }
size_t ws_input(const KpnDims &d) { return (size_t)d.B * d.Cin * d.H * d.W * 2; }
size_t ws_gbox(const KpnDims &d)
{
    return ebfi::round_up((size_t)d.B * d.Ce * d.tiles_y * (TH / WR) * d.tiles_x * (WR + d.K - 1) * (TW + d.K - 1) * 4, (size_t)256);
}
// bias partials are indexed by CTA + slice (injective: CTA ranges are contiguous and slice-major)
size_t ws_bias_part(const KpnDims &d) { return (size_t)(BWD_MAX_GRID + d.nslice) * (NEPI / 32) * d.KK * 4; }

// bf16 operand images for the main loop (weights per slice, channel-chunked input) and the input's tensor map
template <typename T>
int prep_operands(const KpnDims &d, cudaStream_t st, const T *ev, const T *fr, const float *w, void *workspace,
                  CUtensorMap &tmap)
{
    __nv_bfloat16 *wimg = static_cast<__nv_bfloat16 *>(workspace);
    __nv_bfloat16 *featb = reinterpret_cast<__nv_bfloat16 *>(static_cast<char *>(workspace) + ws_weights(d));
    kpn_prep_weights<<<ebfi::sm_count() * 4, 256, 0, st>>>(w, wimg, d);
    EBFI_LAUNCH_OK("kpn_prep_weights");
    kpn_prep_input<<<ebfi::sm_count() * 8, 256, 0, st>>>(ev, fr, featb, d);
    EBFI_LAUNCH_OK("kpn_prep_input");
    return make_tmap(tmap, d, featb);
}

template <bool BWD, typename T>
int launch_fused(const KpnDims &d, cudaStream_t st, const CUtensorMap &tmap, const void *workspace, const float *bias,
                 const T *ev, T *out, const KpnBwdArgs<T> &bw, int per)
{
    const __nv_bfloat16 *wimg = static_cast<const __nv_bfloat16 *>(workspace);
    const int smem = d.w_bytes + d.npart * PART_BYTES;
    const int total = d.nslice * d.ntile;
#define EBFI_KPN(KS, ST)                                                                                      \
    do {                                                                                                      \
        EBFI_CUDA_OK(cudaFuncSetAttribute(kpn_fused_kernel<KS, ST, BWD, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        kpn_fused_kernel<KS, ST, BWD, T><<<ceil_div(total, per), NTHR, smem, st>>>(tmap, wimg, bias, ev, out, bw, d, per); \
    } while (0)
#define EBFI_KPN_K(KS)                                                                                        \
    switch (d.Cin / 32) {                                                                                     \
    case 1: EBFI_KPN(KS, 1); break;                                                                           \
    case 2: EBFI_KPN(KS, 2); break;                                                                           \
    case 3: EBFI_KPN(KS, 3); break;                                                                           \
    default: EBFI_KPN(KS, 4); break;                                                                          \
    }
    switch (d.K) {
    case 1: EBFI_KPN_K(1); break;
    case 3: EBFI_KPN_K(3); break;
    default: EBFI_KPN_K(5); break;
    }
#undef EBFI_KPN_K
#undef EBFI_KPN
    EBFI_LAUNCH_OK("kpn_fused_kernel");
    return EBFI_OK;
}

template <typename T>
int kpn_forward(void *stream, const T *event_feat, const T *frame_feat, const float *conv_weight, const float *conv_bias,
                float negative_slope, T *output, int batch, int channels_event, int channels_frame, int height,
                int width, int kernel_size, void *workspace, size_t workspace_bytes)
{
    KpnDims d{};
    if (int rc = fill(d, batch, channels_event, channels_frame, height, width, kernel_size, negative_slope)) return rc;
    EBFI_REQUIRE(event_feat && (frame_feat || channels_frame == 0) && conv_weight && conv_bias && output,
                 "kpn_fused: null pointer");
    const size_t need = ws_weights(d) + ws_input(d);
    if (!workspace || workspace_bytes < need)
        return ebfi::fail(EBFI_ERR_WORKSPACE, "kpn_fused: workspace %zu < %zu bytes", workspace_bytes, need);
    EBFI_REQUIRE(ebfi::aligned16(workspace), "kpn_fused: workspace must be 16-byte aligned");
    cudaStream_t st = ebfi::as_stream(stream);
    CUtensorMap tmap;
    if (int rc = prep_operands(d, st, event_feat, frame_feat, conv_weight, workspace, tmap)) return rc;
    const int total = d.nslice * d.ntile;
    const int grid = std::min(total, ebfi::sm_count());
    return launch_fused<false>(d, st, tmap, workspace, conv_bias, event_feat, output, KpnBwdArgs<T>{}, ceil_div(total, grid));
}

template <typename T>
int kpn_backward(void *stream, const T *event_feat, const T *frame_feat, const float *conv_weight,
                 const float *conv_bias, float negative_slope, const T *grad_output, T *grad_pre,
                 float *grad_event_fac, float *grad_bias, int batch, int channels_event, int channels_frame,
                 int height, int width, int kernel_size, void *workspace, size_t workspace_bytes)
{
    KpnDims d{};
    if (int rc = fill(d, batch, channels_event, channels_frame, height, width, kernel_size, negative_slope)) return rc;
    EBFI_REQUIRE(event_feat && (frame_feat || channels_frame == 0) && conv_weight && conv_bias && grad_output &&
                 grad_pre && grad_event_fac && grad_bias, "kpn_fused_backward: null pointer");
    const size_t off_gbox = ws_weights(d) + ebfi::round_up(ws_input(d), (size_t)256);
    const size_t off_part = off_gbox + ws_gbox(d);
    const size_t need = off_part + ws_bias_part(d);
    if (!workspace || workspace_bytes < need)
        return ebfi::fail(EBFI_ERR_WORKSPACE, "kpn_fused_backward: workspace %zu < %zu bytes", workspace_bytes, need);
    EBFI_REQUIRE(ebfi::aligned16(workspace), "kpn_fused_backward: workspace must be 16-byte aligned");
    cudaStream_t st = ebfi::as_stream(stream);
    CUtensorMap tmap;
    if (int rc = prep_operands(d, st, event_feat, frame_feat, conv_weight, workspace, tmap)) return rc;
    KpnBwdArgs<T> bw;
    bw.gout = grad_output;
    bw.gpre = grad_pre;
    bw.gbox = reinterpret_cast<float *>(static_cast<char *>(workspace) + off_gbox);
    bw.bias_part = reinterpret_cast<float *>(static_cast<char *>(workspace) + off_part);
    const int total = d.nslice * d.ntile;
    const int grid = std::min(std::min(total, ebfi::sm_count()), BWD_MAX_GRID);
    const int per = ceil_div(total, grid);
    if (int rc = launch_fused<true>(d, st, tmap, workspace, conv_bias, event_feat, static_cast<T *>(nullptr), bw, per))
        return rc;
    kpn_gev_collect<<<ebfi::sm_count() * 8, 256, 0, st>>>(bw.gbox, grad_event_fac, d);
    EBFI_LAUNCH_OK("kpn_gev_collect");
    kpn_bias_collect<<<ceil_div(d.Ce * d.KK, 128), 128, 0, st>>>(bw.bias_part, grad_bias, d, per);
    EBFI_LAUNCH_OK("kpn_bias_collect");
    return EBFI_OK;
}

}  // namespace

extern "C" {

size_t ebfi_kpn_fused_workspace_bytes(int batch, int channels_event, int channels_frame, int height, int width,
                                      int kernel_size)
{
    KpnDims d{};
    if (fill(d, batch, channels_event, channels_frame, height, width, kernel_size, 0.f) != EBFI_OK) return 0;
    return ws_weights(d) + ws_input(d) + 256;
}

int ebfi_kpn_fused_forward(void *stream, const float *event_feat, const float *frame_feat, const float *conv_weight,
                           const float *conv_bias, float negative_slope, float *output, int batch,
                           int channels_event, int channels_frame, int height, int width, int kernel_size,
                           void *workspace, size_t workspace_bytes)
{
    return kpn_forward(stream, event_feat, frame_feat, conv_weight, conv_bias, negative_slope, output, batch,
                       channels_event, channels_frame, height, width, kernel_size, workspace, workspace_bytes);
}

int ebfi_kpn_fused_forward_bf16(void *stream, const void *event_feat, const void *frame_feat, const float *conv_weight,
                                const float *conv_bias, float negative_slope, void *output, int batch,
                                int channels_event, int channels_frame, int height, int width, int kernel_size,
                                void *workspace, size_t workspace_bytes)
{
    return kpn_forward(stream, static_cast<const __nv_bfloat16 *>(event_feat),
                       static_cast<const __nv_bfloat16 *>(frame_feat), conv_weight, conv_bias, negative_slope,
                       static_cast<__nv_bfloat16 *>(output), batch, channels_event, channels_frame, height, width,
                       kernel_size, workspace, workspace_bytes);
}

int ebfi_kpn_fused_forward_fp16(void *stream, const void *event_feat, const void *frame_feat, const float *conv_weight,
                                const float *conv_bias, float negative_slope, void *output, int batch,
                                int channels_event, int channels_frame, int height, int width, int kernel_size,
                                void *workspace, size_t workspace_bytes)
{
    return kpn_forward(stream, static_cast<const __half *>(event_feat), static_cast<const __half *>(frame_feat),
                       conv_weight, conv_bias, negative_slope, static_cast<__half *>(output), batch, channels_event,
                       channels_frame, height, width, kernel_size, workspace, workspace_bytes);
}

size_t ebfi_kpn_fused_backward_workspace_bytes(int batch, int channels_event, int channels_frame, int height, int width,
                                               int kernel_size)
{
    KpnDims d{};
    if (fill(d, batch, channels_event, channels_frame, height, width, kernel_size, 0.f) != EBFI_OK) return 0;
    return ws_weights(d) + ebfi::round_up(ws_input(d), (size_t)256) + ws_gbox(d) + ws_bias_part(d) + 256;
}

int ebfi_kpn_fused_backward(void *stream, const float *event_feat, const float *frame_feat, const float *conv_weight,
                            const float *conv_bias, float negative_slope, const float *grad_output, float *grad_pre,
                            float *grad_event_fac, float *grad_bias, int batch, int channels_event, int channels_frame,
                            int height, int width, int kernel_size, void *workspace, size_t workspace_bytes)
{
    return kpn_backward(stream, event_feat, frame_feat, conv_weight, conv_bias, negative_slope, grad_output, grad_pre,
                        grad_event_fac, grad_bias, batch, channels_event, channels_frame, height, width, kernel_size,
                        workspace, workspace_bytes);
}

int ebfi_kpn_fused_backward_bf16(void *stream, const void *event_feat, const void *frame_feat, const float *conv_weight,
                                 const float *conv_bias, float negative_slope, const void *grad_output, void *grad_pre,
                                 float *grad_event_fac, float *grad_bias, int batch, int channels_event,
                                 int channels_frame, int height, int width, int kernel_size, void *workspace,
                                 size_t workspace_bytes)
{
    return kpn_backward(stream, static_cast<const __nv_bfloat16 *>(event_feat),
                        static_cast<const __nv_bfloat16 *>(frame_feat), conv_weight, conv_bias, negative_slope,
                        static_cast<const __nv_bfloat16 *>(grad_output), static_cast<__nv_bfloat16 *>(grad_pre),
                        grad_event_fac, grad_bias, batch, channels_event, channels_frame, height, width, kernel_size,
                        workspace, workspace_bytes);
}

int ebfi_kpn_fused_backward_fp16(void *stream, const void *event_feat, const void *frame_feat, const float *conv_weight,
                                 const float *conv_bias, float negative_slope, const void *grad_output, void *grad_pre,
                                 float *grad_event_fac, float *grad_bias, int batch, int channels_event,
                                 int channels_frame, int height, int width, int kernel_size, void *workspace,
                                 size_t workspace_bytes)
{
    return kpn_backward(stream, static_cast<const __half *>(event_feat), static_cast<const __half *>(frame_feat),
                        conv_weight, conv_bias, negative_slope, static_cast<const __half *>(grad_output),
                        static_cast<__half *>(grad_pre), grad_event_fac, grad_bias, batch, channels_event,
                        channels_frame, height, width, kernel_size, workspace, workspace_bytes);
}

}  // extern "C"
