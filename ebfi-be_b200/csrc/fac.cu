// fac.cu — FAC KernelConv2D (per-pixel K x K kernel-prediction filter) for sm_100a.
//
// Replaces the three SIMT kernels of the reference
// (models/FAC/kernelconv2d/KernelConv2D_kernel.cu:25-53 forward, :91-125 grad-input,
// :128-150 grad-kernel). The op is pure HBM streaming: the (B, C*K*K, H, W) kernel tensor
// is 92 % of the bytes, so the design goal is "touch every byte of it exactly once, with
// 128-bit coalesced accesses, and never write or read anything that is not algorithmic".
//
// Layout facts used: for a fixed (b, c) the K*K kernel planes, the output plane and the
// grad_output plane are contiguous H*W arrays; only `input` has the (W+K-1) pitch.
//
// "march" kernels: a thread owns PX (4 or 1) adjacent output columns and walks down a
// segment of rows. The K input rows it needs live in a register window that is shifted by
// one row per step, so every input value is loaded once per thread. Forward is then
// 25 streaming 128-bit loads + 1 store per 4 outputs.
//
// Backward is ONE fused pass (the reference runs two kernels and reads `kernel` twice):
// per row it streams kernel + grad_output in, grad_kernel out, and scatters
// kernel*grad_output into a K-row register accumulator of grad_input. Column halos are
// exchanged between neighbouring threads through shared memory once per row; row halos
// between neighbouring segments (CTAs) go through a small workspace and are merged by
// whichever of the two CTAs finishes second. Every grad_input element is a sum of the same
// terms in the same order on every run (two-operand merge adds commute), so the result is
// bit-reproducible without atomics on data.
#include "common.cuh"
#include "umma.cuh"

#include <algorithm>
#include <cuda_bf16.h>      // mbarrier + 1-D bulk (TMA) copy helpers
#include <cuda_fp16.h>

namespace {

using ebfi::ceil_div;

// Element types: fp32 (the reference's), bf16 and fp16 (storage only; all arithmetic is fp32). Loads widen exactly,
// stores round once (RN); an fp16 store overflows to +-inf, as tensor.half() does.
using bf16 = __nv_bfloat16;
using fp16 = __half;
__device__ __forceinline__ float ld_elt(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ld_elt(const bf16 *p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ld_elt(const fp16 *p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ld_elt_cg(const float *p) { return __ldcg(p); }
__device__ __forceinline__ float ld_elt_cg(const bf16 *p) { return __bfloat162float(__ldcg(p)); }
__device__ __forceinline__ float ld_elt_cg(const fp16 *p) { return __half2float(__ldcg(p)); }
__device__ __forceinline__ void st_elt(float *p, float v) { *p = v; }
__device__ __forceinline__ void st_elt(bf16 *p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void st_elt(fp16 *p, float v) { *p = __float2half_rn(v); }

// PX-wide vectors (held as fp32) with streaming (evict-first) global access and shared-memory reads.
template <int PX> struct Vec;
template <> struct Vec<4> {
    float v[4];
    __device__ __forceinline__ static Vec load_stream(const float *p)
    {
        float4 t = __ldcs(reinterpret_cast<const float4 *>(p));
        return Vec{{t.x, t.y, t.z, t.w}};
    }
    __device__ __forceinline__ static Vec load_stream(const bf16 *p)
    {
        const uint2 t = __ldcs(reinterpret_cast<const uint2 *>(p));
        return Vec{{__uint_as_float(t.x << 16), __uint_as_float(t.x & 0xFFFF0000u),
                    __uint_as_float(t.y << 16), __uint_as_float(t.y & 0xFFFF0000u)}};
    }
    __device__ __forceinline__ static Vec load_stream(const fp16 *p)
    {
        const uint2 t = __ldcs(reinterpret_cast<const uint2 *>(p));
        return from_half2(t);
    }
    __device__ __forceinline__ static Vec load_smem(const float *p)
    {
        const float4 t = *reinterpret_cast<const float4 *>(p);
        return Vec{{t.x, t.y, t.z, t.w}};
    }
    __device__ __forceinline__ static Vec load_smem(const bf16 *p)
    {
        const uint2 t = *reinterpret_cast<const uint2 *>(p);
        return Vec{{__uint_as_float(t.x << 16), __uint_as_float(t.x & 0xFFFF0000u),
                    __uint_as_float(t.y << 16), __uint_as_float(t.y & 0xFFFF0000u)}};
    }
    __device__ __forceinline__ static Vec load_smem(const fp16 *p) { return from_half2(*reinterpret_cast<const uint2 *>(p)); }
    __device__ __forceinline__ static Vec from_half2(uint2 t)
    {
        const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&t.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&t.y));
        return Vec{{a.x, a.y, b.x, b.y}};
    }
    __device__ __forceinline__ void store_stream(float *p) const
    {
        __stcs(reinterpret_cast<float4 *>(p), make_float4(v[0], v[1], v[2], v[3]));
    }
    __device__ __forceinline__ void store_stream(bf16 *p) const
    {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
        __stcs(reinterpret_cast<uint2 *>(p), make_uint2(*reinterpret_cast<const uint32_t *>(&a),
                                                         *reinterpret_cast<const uint32_t *>(&b)));
    }
    __device__ __forceinline__ void store_stream(fp16 *p) const
    {
        const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
        __stcs(reinterpret_cast<uint2 *>(p), make_uint2(*reinterpret_cast<const uint32_t *>(&a),
                                                         *reinterpret_cast<const uint32_t *>(&b)));
    }
    // plain (write-back) stores
    __device__ __forceinline__ void store(float *p) const
    {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
    __device__ __forceinline__ void store(bf16 *p) const
    {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<const uint32_t *>(&a),
                                                   *reinterpret_cast<const uint32_t *>(&b));
    }
    __device__ __forceinline__ void store(fp16 *p) const
    {
        const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<const uint32_t *>(&a),
                                                   *reinterpret_cast<const uint32_t *>(&b));
    }
};
template <> struct Vec<1> {
    float v[1];
    __device__ __forceinline__ static Vec load_stream(const float *p) { return Vec{{__ldcs(p)}}; }
    __device__ __forceinline__ static Vec load_stream(const bf16 *p) { return Vec{{__bfloat162float(*p)}}; }
    __device__ __forceinline__ static Vec load_stream(const fp16 *p) { return Vec{{__half2float(*p)}}; }
    __device__ __forceinline__ void store_stream(float *p) const { __stcs(p, v[0]); }
    __device__ __forceinline__ void store_stream(bf16 *p) const { *p = __float2bfloat16_rn(v[0]); }
    __device__ __forceinline__ void store_stream(fp16 *p) const { *p = __float2half_rn(v[0]); }
    template <typename T> __device__ __forceinline__ void store(T *p) const { st_elt(p, v[0]); }
};

struct FacDims {
    int H, W;          // output size
    int seg_rows;      // rows per segment
    int nseg;          // segments per plane
    int nxb;           // thread blocks along x (forward only)
    int nstage;        // ring stages of the backward (0 = register variant)
    int xstride;       // backward: first column of block i is i * xstride (blocks overlap by `halo_thr` threads)
    int halo_thr;      // backward: leading threads of blocks > 0 that only recompute the left neighbour's columns
};

// REPL = true: `input` is the unpadded (B, C, H, W) tensor and the kernels read it through
// ReplicationPad2d((K-1)/2): padded cell (Y, X) is input[clamp(Y-p, 0, H-1)][clamp(X-p, 0, W-1)].
// `in_at` returns the address of padded cell (Y, x + j) of the thread's plane.
template <int K, bool REPL, typename T>
__device__ __forceinline__ const T *in_at(const T *inp, int Y, int x, int j, int H, int W, int Wi)
{
    if constexpr (REPL) {
        constexpr int P = (K - 1) / 2;
        return inp + (size_t)min(max(Y - P, 0), H - 1) * W + min(max(x + j - P, 0), W - 1);
    } else {
        return inp + (size_t)Y * Wi + j;      // `inp` already points at column x
    }
}

// ------------------------------------------------------------------ forward ---
template <int K, int PX, bool REPL, typename T>
__global__ void __launch_bounds__(128)
fac_fwd_march(const T *__restrict__ in, const T *__restrict__ ker, T *__restrict__ out,
              FacDims d)
{
    constexpr int WIN = PX + K - 1;
    int bid = blockIdx.x;
    const int xb = bid % d.nxb;  bid /= d.nxb;
    const int seg = bid % d.nseg;
    const int plane = bid / d.nseg;
    const int x = (xb * blockDim.x + threadIdx.x) * PX;
    if (x >= d.W) return;

    const int H = d.H, W = d.W, Wi = W + K - 1;
    const int y0 = seg * d.seg_rows, y1 = min(H, y0 + d.seg_rows);
    const T *inp = in + (REPL ? (size_t)plane * H * W : (size_t)plane * (H + K - 1) * Wi + x);
    const T *kp = ker + (size_t)plane * K * K * H * W + x;
    T *op = out + (size_t)plane * H * W + x;

    float win[K][WIN];
#pragma unroll
    for (int r = 1; r < K; ++r)
#pragma unroll
        for (int j = 0; j < WIN; ++j)
            win[r][j] = ld_elt(REPL ? in_at<K, REPL>(inp, y0 + r - 1, x, j, H, W, Wi) : inp + (size_t)(y0 + r - 1) * Wi + j);

    for (int y = y0; y < y1; ++y) {
        Vec<PX> kv[K * K];
#pragma unroll
        for (int k = 0; k < K * K; ++k) kv[k] = Vec<PX>::load_stream(kp + ((size_t)k * H + y) * W);
#pragma unroll
        for (int r = 0; r < K - 1; ++r)
#pragma unroll
            for (int j = 0; j < WIN; ++j) win[r][j] = win[r + 1][j];
#pragma unroll
        for (int j = 0; j < WIN; ++j)
            win[K - 1][j] = ld_elt(REPL ? in_at<K, REPL>(inp, y + K - 1, x, j, H, W, Wi) : inp + (size_t)(y + K - 1) * Wi + j);

        Vec<PX> acc;
#pragma unroll
        for (int i = 0; i < PX; ++i) acc.v[i] = 0.f;
        // same tap order as the reference's loop (KernelConv2D_kernel.cu:44-49)
#pragma unroll
        for (int ky = 0; ky < K; ++ky)
#pragma unroll
            for (int kx = 0; kx < K; ++kx)
#pragma unroll
                for (int i = 0; i < PX; ++i) acc.v[i] += win[ky][kx + i] * kv[ky * K + kx].v[i];
        acc.store_stream(op + (size_t)y * W);
    }
}

// ----------------------------------------------------------------- backward ---
// Workspace layout: [planes * (nseg-1)] int arrival counters (zeroed by the launcher),
// then [planes * (nseg-1)][K-1][Wi] fp32 overhang rows.
// RING = true (4 px/thread only): the K*K kernel rows and the grad_output row of each step arrive
// through a ring of `d.nstage` shared-memory stages filled by 1-D bulk (TMA) copies that one thread
// issues two rows ahead; bytes in flight then live in shared memory instead of registers (the
// register variant keeps 25 float4 loads = 100 registers per thread in flight, 8 warps per SM).
//
// REPL = true (K > 1): `in` and `gin` are the unpadded (B, C, H, W) tensors and the kernel folds
// ReplicationPad2d((K-1)/2) in. The window reads clamped cells (in_at). grad_input is still
// accumulated, exchanged and handed between segments in padded coordinates; a finished padded row
// goes into the fp32 shared row `srow`, where the padded rows that replicate the same input row
// (the first P+1 and the last P+1) are summed in ascending order. When the last of them is in, the
// row is stored once, shifted by P columns, with padded columns 0..P summed (ascending) into
// column 0 and W-1+P..W-1+2P into column W-1. Block i stores unpadded columns
// [xbase + halo_thr*PX - Q, xbase + blockDim.x*PX - Q) (Q = P rounded up to PX, so float4 stores
// stay aligned): the plan makes halo_thr*PX >= Q + P, so every padded column such a store reads is
// complete in this block. Block 0 starts at column 0 and the last block ends at W; only they fold.
// The workspace is the one of the padded op (same segments, same overhang rows).
template <int K, int PX, bool RING, bool REPL, typename T>
// (a 128-register cap for more CTAs/SM spills and loses 25 %; the REPL variant states min 1 block/SM, without which
// ptxas caps its ring variant at 128 registers and spills)
__global__ void __launch_bounds__(256, REPL ? 1 : 0)
fac_bwd_march(const T *__restrict__ in, const T *__restrict__ ker,
              const T *__restrict__ gout, T *__restrict__ gin, T *__restrict__ gker,
              int *__restrict__ counters, float *__restrict__ overhang, FacDims d)
{
    constexpr int WIN = PX + K - 1;
    constexpr int R = K - 1;                       // halo width
    constexpr int RS = R > 0 ? R : 1;
    constexpr int D = R > 0 ? (R + PX - 1) / PX : 0;   // how many left neighbours reach into my columns
    constexpr int P = R / 2;                       // replication pad (REPL)
    constexpr int Q = (P + PX - 1) / PX * PX;
    static_assert(!REPL || R > 0, "K = 1 needs no pad: run the plain op");
    extern __shared__ __align__(128) float dyn_smem[];
    float *xchg = dyn_smem;                        // [2][blockDim.x][RS]
    float *srow = dyn_smem + ((2 * blockDim.x * RS + 31) & ~31);   // REPL: [blockDim.x * PX + R] padded columns
    __shared__ int s_flag[2];
    __shared__ __align__(8) uint64_t ring_bar[4];

    // Wide rows are cut into column blocks (one CTA each). Block i > 0 starts `halo_thr` threads to
    // the left of the columns it owns: those threads re-read kernel / grad_output of the left
    // neighbour's last columns so that every grad_input column a block owns gets all its terms
    // (1.6 % extra reads at 252 owned columns); they store nothing.
    const int xb = blockIdx.x % d.nxb;
    const int seg = (blockIdx.x / d.nxb) % d.nseg;
    const int plane = blockIdx.x / (d.nxb * d.nseg);
    const int H = d.H, W = d.W, Wi = W + R;
    const int t = threadIdx.x, nthr = blockDim.x;
    const int xbase = xb * d.xstride;
    const int x = xbase + t * PX;
    const bool active = x < W;
    const bool own = active && (xb == 0 || t >= d.halo_thr);
    const bool last_xb = (xb == d.nxb - 1);
    const int nact = min(nthr, ceil_div(W - xbase, PX));   // threads of this block that hold output columns
    const int y0 = seg * d.seg_rows, y1 = min(H, y0 + d.seg_rows);
    const bool wi_vec = (PX == 4) && (Wi % 4 == 0);

    const T *inp = REPL ? in + (size_t)plane * H * W : in + (size_t)plane * (H + R) * Wi + x;
    const T *kp = ker + (size_t)plane * K * K * H * W + x;
    const T *gp = gout + (size_t)plane * H * W + x;
    T *gkp = gker + (size_t)plane * K * K * H * W + x;
    T *gip = REPL ? gin + (size_t)plane * H * W : gin + (size_t)plane * (H + R) * Wi;

    float win[K][WIN], acc[K][WIN];
#pragma unroll
    for (int r = 0; r < K; ++r)
#pragma unroll
        for (int j = 0; j < WIN; ++j) { acc[r][j] = 0.f; win[r][j] = 0.f; }
    if (active) {
#pragma unroll
        for (int r = 1; r < K; ++r)
#pragma unroll
            for (int j = 0; j < WIN; ++j) win[r][j] = ld_elt(in_at<K, REPL>(inp, y0 + r - 1, x, j, H, W, Wi));
    }

    // ---- ring of (K*K + 1) x W elements per stage: rows k of `kernel`, then the grad_output row
    T *ring = reinterpret_cast<T *>(dyn_smem + ((2 * blockDim.x * RS + 31) & ~31) +
                                    (REPL ? ((blockDim.x * PX + R + 31) & ~31) : 0));
    const int bw = nthr * PX;                      // row pitch of a stage = columns a block can hold
    const int ncols = min(bw, W - xbase);          // columns of this block that exist
    const int stage_elts = (K * K + 1) * bw;
    auto issue_row = [&](int y) {                  // thread 0: bulk copies of row y into its stage
        const int st = (y - y0) % d.nstage;
        T *dst = ring + (size_t)st * stage_elts;
        umma::mbar_expect_tx(&ring_bar[st], (uint32_t)((K * K + 1) * ncols * sizeof(T)));
        const T *src = ker + (size_t)plane * K * K * H * W + (size_t)y * W + xbase;
        for (int k = 0; k < K * K; ++k)
            umma::bulk_g2s(dst + (size_t)k * bw, src + (size_t)k * H * W, (uint32_t)(ncols * sizeof(T)), &ring_bar[st]);
        umma::bulk_g2s(dst + (size_t)K * K * bw, gout + (size_t)plane * H * W + (size_t)y * W + xbase,
                       (uint32_t)(ncols * sizeof(T)), &ring_bar[st]);
    };
    if constexpr (RING) {
        if (t == 0) {
            for (int i = 0; i < d.nstage; ++i) umma::mbar_init(&ring_bar[i], 1);
            umma::mbar_fence_init();
            for (int y = y0; y < min(y1, y0 + d.nstage - 1); ++y) issue_row(y);
        }
        __syncthreads();
    }

    // Emits one finished (or segment-partial) grad_input row held in acc[0] after the
    // neighbour exchange. `dst` is the row base (Wi floats) in gin or in the overhang buffer.
    // `dst_t` (a grad_input row) or `dst_f` (an fp32 overhang row): exactly one is non-null.
    // REPL: `dst_t` is unused; a grad_input row (dst_f null) is padded row Y and goes through srow.
    auto emit_row = [&](const float (&row)[WIN], T *dst_t, float *dst_f, int parity, int Y) {
        float *xb = xchg + (size_t)parity * nthr * RS;
        if constexpr (R > 0) {
#pragma unroll
            for (int j = 0; j < R; ++j) xb[t * RS + j] = row[PX + j];
        }
        __syncthreads();
        if constexpr (REPL) {
            if (!dst_f) {
                // padded rows Y with the same clamp(Y-P, 0, H-1) are summed in srow, first one assigns
                const bool first = Y == 0 || (Y > P && Y <= H - 1 + P);
                const bool last = Y == H - 1 + R || (Y >= P && Y <= H - 2 + P);
                if (active) {
#pragma unroll
                    for (int j = 0; j < PX; ++j) {
                        float o = row[j];
#pragma unroll
                        for (int dd = 1; dd <= D; ++dd) {
                            const int c = j + PX * dd;
                            if (t - dd >= 0 && c < WIN) o += xb[(t - dd) * RS + (c - PX)];
                        }
                        srow[t * PX + j] = first ? o : srow[t * PX + j] + o;
                    }
                }
                if (last_xb && t < R) {
                    const int X = W + t, tv = (X - xbase) / PX, j = (X - xbase) % PX;
                    float o = 0.f;
                    for (int dd = 1; dd <= D; ++dd) {
                        const int src = tv - dd, c = j + PX * dd;
                        if (src >= 0 && src < nact && c < WIN) o += xb[src * RS + (c - PX)];
                    }
                    srow[X - xbase] = first ? o : srow[X - xbase] + o;
                }
                if (!last) return;
                __syncthreads();
                T *dst = gip + (size_t)min(max(Y - P, 0), H - 1) * W;
                const int ub0 = xbase == 0 ? 0 : xbase + d.halo_thr * PX - Q;   // this block's unpadded columns
                const int ub1 = last_xb ? W : xbase + nthr * PX - Q;
                for (int u = ub0 + t * PX; u < ub1; u += nthr * PX) {
                    Vec<PX> v;
#pragma unroll
                    for (int j = 0; j < PX; ++j) v.v[j] = srow[u + j + P - xbase];
                    if (u == 0) {                // left fold: padded columns 0 .. P, ascending
                        float f = srow[0 - xbase];
                        for (int c = 1; c <= P; ++c) f += srow[c - xbase];
                        v.v[0] = f;
                    }
                    if (u + PX >= W) {           // right fold: padded columns W-1+P .. W-1+2P, ascending
                        float f = v.v[PX - 1];
                        for (int c = W + P; c <= W - 1 + R; ++c) f += srow[c - xbase];
                        v.v[PX - 1] = f;
                    }
                    v.store(dst + u);
                }
                return;
            }
        }
        if (own) {
            float o[PX];
#pragma unroll
            for (int j = 0; j < PX; ++j) o[j] = row[j];
#pragma unroll
            for (int dd = 1; dd <= D; ++dd) {
                if (t - dd >= 0) {
#pragma unroll
                    for (int j = 0; j < PX; ++j) {
                        const int c = j + PX * dd;           // column of thread t-dd's row
                        if (c < WIN) o[j] += xb[(t - dd) * RS + (c - PX)];
                    }
                }
            }
            if (dst_f) {
                if (wi_vec) {
                    *reinterpret_cast<float4 *>(dst_f + x) = make_float4(o[0], o[PX > 1 ? 1 : 0], o[PX > 2 ? 2 : 0], o[PX > 3 ? 3 : 0]);
                } else {
#pragma unroll
                    for (int j = 0; j < PX; ++j) dst_f[x + j] = o[j];
                }
            } else if (wi_vec && sizeof(T) == 4) {
                *reinterpret_cast<float4 *>(dst_t + x) = make_float4(o[0], o[PX > 1 ? 1 : 0], o[PX > 2 ? 2 : 0], o[PX > 3 ? 3 : 0]);
            } else {
#pragma unroll
                for (int j = 0; j < PX; ++j) st_elt(dst_t + x + j, o[j]);
            }
        }
        if constexpr (R > 0) {
            // right halo columns W .. W+R-1 have no owner thread: the first R threads of the last
            // column block gather them
            if (last_xb && t < R) {
                const int X = W + t, tv = (X - xbase) / PX, j = (X - xbase) % PX;
                float o = 0.f;
                for (int dd = 1; dd <= D; ++dd) {
                    const int src = tv - dd, c = j + PX * dd;
                    if (src >= 0 && src < nact && c < WIN) o += xb[src * RS + (c - PX)];
                }
                if (dst_f) dst_f[X] = o; else st_elt(dst_t + X, o);
            }
        }
    };

    int parity = 0;
    for (int y = y0; y < y1; ++y) {
        if constexpr (RING) {
            // the stage that row y + nstage - 1 reuses was consumed in iteration y - 1 (emit_row's barrier)
            if (t == 0 && y + d.nstage - 1 < y1) issue_row(y + d.nstage - 1);
            const int st = (y - y0) % d.nstage;
            umma::mbar_wait(&ring_bar[st], ((y - y0) / d.nstage) & 1);
            if (active) {
                const T *stg = ring + (size_t)st * stage_elts + t * PX;
                const Vec<4> gv = Vec<4>::load_smem(stg + (size_t)K * K * bw);
                const float *g = gv.v;
#pragma unroll
                for (int r = 0; r < K - 1; ++r)
#pragma unroll
                    for (int j = 0; j < WIN; ++j) win[r][j] = win[r + 1][j];
#pragma unroll
                for (int j = 0; j < WIN; ++j) win[K - 1][j] = ld_elt(in_at<K, REPL>(inp, y + K - 1, x, j, H, W, Wi));
#pragma unroll
                for (int ky = 0; ky < K; ++ky)
#pragma unroll
                    for (int kx = 0; kx < K; ++kx) {
                        const Vec<4> kq = Vec<4>::load_smem(stg + (size_t)(ky * K + kx) * bw);
                        const float *kvv = kq.v;
                        Vec<4> gk;
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            gk.v[i] = win[ky][kx + i] * g[i];
                            acc[ky][kx + i] += kvv[i] * g[i];
                        }
                        if (own) gk.store_stream(gkp + ((size_t)(ky * K + kx) * H + y) * W);
                    }
            }
        } else if (active) {
            Vec<PX> kv[K * K];
#pragma unroll
            for (int k = 0; k < K * K; ++k) kv[k] = Vec<PX>::load_stream(kp + ((size_t)k * H + y) * W);
            const Vec<PX> g = Vec<PX>::load_stream(gp + (size_t)y * W);
#pragma unroll
            for (int r = 0; r < K - 1; ++r)
#pragma unroll
                for (int j = 0; j < WIN; ++j) win[r][j] = win[r + 1][j];
#pragma unroll
            for (int j = 0; j < WIN; ++j) win[K - 1][j] = ld_elt(in_at<K, REPL>(inp, y + K - 1, x, j, H, W, Wi));
#pragma unroll
            for (int ky = 0; ky < K; ++ky)
#pragma unroll
                for (int kx = 0; kx < K; ++kx) {
                    Vec<PX> gk;
#pragma unroll
                    for (int i = 0; i < PX; ++i) {
                        gk.v[i] = win[ky][kx + i] * g.v[i];                 // grad_kernel (:149)
                        acc[ky][kx + i] += kv[ky * K + kx].v[i] * g.v[i];   // grad_input scatter (:117-120)
                    }
                    if (own) gk.store_stream(gkp + ((size_t)(ky * K + kx) * H + y) * W);
                }
        }
        emit_row(acc[0], gip + (size_t)y * Wi, nullptr, parity, y);
        parity ^= 1;
#pragma unroll
        for (int r = 0; r < K - 1; ++r)
#pragma unroll
            for (int j = 0; j < WIN; ++j) acc[r][j] = acc[r + 1][j];
#pragma unroll
        for (int j = 0; j < WIN; ++j) acc[K - 1][j] = 0.f;
    }

    if constexpr (R > 0) {
        // rows y1 .. y1+R-1: complete for the last segment, overhang for the others
        const bool last = (seg == d.nseg - 1);
        float *oh = last ? nullptr : overhang + ((size_t)plane * (d.nseg - 1) + seg) * R * Wi;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (last) emit_row(acc[r], gip + (size_t)(y1 + r) * Wi, nullptr, parity, y1 + r);
            else emit_row(acc[r], nullptr, oh + (size_t)r * Wi, parity, y1 + r);
            parity ^= 1;
        }
        if (d.nseg == 1) return;

        // Hand-off: each boundary between segments s|s+1 has 2 * nxb parties (the column blocks above
        // and below); the last one to arrive adds the upper segment's overhang rows onto the lower
        // segment's partial rows (always `partial + overhang`, so the result does not depend on who merges).
        __threadfence();
        __syncthreads();
        if (t == 0) {
            s_flag[0] = seg > 0 ? atomicAdd(&counters[plane * (d.nseg - 1) + seg - 1], 1) : 0;
            s_flag[1] = !last ? atomicAdd(&counters[plane * (d.nseg - 1) + seg], 1) : 0;
        }
        __syncthreads();
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            if (s_flag[side] != 2 * d.nxb - 1) continue;
            __threadfence();
            const int bseg = side == 0 ? seg - 1 : seg;             // upper segment of the boundary
            const int yb = (bseg + 1) * d.seg_rows;                 // first row of the lower segment
            const float *src = overhang + ((size_t)plane * (d.nseg - 1) + bseg) * R * Wi;
            if constexpr (REPL) {
                // the overhang rows yb .. yb+R-1 (padded) folded like emit_row: per padded column the rows
                // of one unpadded row, ascending, then the columns of one unpadded column, ascending
                const int ua = min(max(yb - P, 0), H - 1), ub = min(max(yb + R - 1 - P, 0), H - 1);
                for (int e = t; e < (ub - ua + 1) * W; e += nthr) {
                    const int u = ua + e / W, X = e % W;
                    const int ylo = max(yb, u == 0 ? 0 : u + P), yhi = min(yb + R - 1, u == H - 1 ? H - 1 + R : u + P);
                    const int clo = X == 0 ? 0 : X + P, chi = X == W - 1 ? W - 1 + R : X + P;
                    float s = 0.f;
                    for (int c = clo; c <= chi; ++c) {
                        float r = __ldcg(src + (size_t)(ylo - yb) * Wi + c);
                        for (int Y = ylo + 1; Y <= yhi; ++Y) r += __ldcg(src + (size_t)(Y - yb) * Wi + c);
                        s = c == clo ? r : s + r;
                    }
                    T *dst = gip + (size_t)u * W + X;
                    st_elt(dst, ld_elt_cg(dst) + s);
                }
            } else {
                T *dst = gip + (size_t)yb * Wi;
                for (int e = t; e < R * Wi; e += nthr) st_elt(dst + e, ld_elt_cg(dst + e) + __ldcg(src + e));
            }
        }
    }
}

// ------------------------------------------------- generic fallback kernels ---
// Any K, any size: one thread per element, no data-dependent reductions. REPL as in the march kernels:
// unpadded `in` / `gin`, the pad's clamp on every input read, and each grad_input element the sum, in a fixed
// order (per padded column its rows ascending, then the columns ascending), of the padded cells it replicates.
template <bool REPL, typename T>
__global__ void fac_fwd_generic(const T *__restrict__ in, const T *__restrict__ ker,
                                T *__restrict__ out, int planes, int H, int W, int K)
{
    const size_t n = (size_t)planes * H * W;
    const int Wi = W + K - 1, Hi = H + K - 1, P = (K - 1) / 2;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        const int x = e % W, y = (e / W) % H;
        const size_t plane = e / ((size_t)H * W);
        const T *ip = REPL ? in + plane * H * W : in + (plane * Hi + y) * Wi + x;
        const T *kp = ker + plane * K * K * H * W + (size_t)y * W + x;
        float s = 0.f;
        for (int ky = 0; ky < K; ++ky)
            for (int kx = 0; kx < K; ++kx) {
                const T *ipk = REPL ? ip + (size_t)min(max(y + ky - P, 0), H - 1) * W + min(max(x + kx - P, 0), W - 1)
                                    : ip + (size_t)ky * Wi + kx;
                s += ld_elt(ipk) * ld_elt(kp + (size_t)(ky * K + kx) * H * W);
            }
        st_elt(out + e, s);
    }
}

// grad_input of padded cell (Y, X) of one plane
template <typename T>
__device__ __forceinline__ float fac_gin_cell(const T *kp, const T *gp, int Y, int X, int H, int W, int K)
{
    float s = 0.f;
    for (int ky = 0; ky < K; ++ky)
        for (int kx = 0; kx < K; ++kx) {
            const int y = Y - ky, x = X - kx;
            if (y >= 0 && y < H && x >= 0 && x < W)
                s += ld_elt(kp + ((size_t)(ky * K + kx) * H + y) * W + x) * ld_elt(gp + (size_t)y * W + x);
        }
    return s;
}

template <bool REPL, typename T>
__global__ void fac_bwd_generic(const T *__restrict__ in, const T *__restrict__ ker,
                                const T *__restrict__ gout, T *__restrict__ gin,
                                T *__restrict__ gker, int planes, int H, int W, int K)
{
    const int Wi = W + K - 1, Hi = H + K - 1, P = (K - 1) / 2, R = K - 1;
    const int Hg = REPL ? H : Hi, Wg = REPL ? W : Wi;          // grad_input plane
    const size_t n_in = (size_t)planes * Hg * Wg, n_k = (size_t)planes * K * K * H * W;
    const size_t stride = (size_t)gridDim.x * blockDim.x, tid = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    for (size_t e = tid; e < n_in; e += stride) {
        const int X = e % Wg, Y = (e / Wg) % Hg;
        const size_t plane = e / ((size_t)Hg * Wg);
        const T *kp = ker + plane * K * K * H * W, *gp = gout + plane * H * W;
        float s = 0.f;
        if constexpr (REPL) {
            const int ylo = Y == 0 ? 0 : Y + P, yhi = Y == H - 1 ? H - 1 + R : Y + P;
            const int xlo = X == 0 ? 0 : X + P, xhi = X == W - 1 ? W - 1 + R : X + P;
            for (int c = xlo; c <= xhi; ++c) {
                float r = fac_gin_cell(kp, gp, ylo, c, H, W, K);
                for (int Yp = ylo + 1; Yp <= yhi; ++Yp) r += fac_gin_cell(kp, gp, Yp, c, H, W, K);
                s = c == xlo ? r : s + r;
            }
        } else {
            for (int ky = 0; ky < K; ++ky)
                for (int kx = 0; kx < K; ++kx) {
                    const int y = Y - ky, x = X - kx;
                    if (y >= 0 && y < H && x >= 0 && x < W)
                        s += ld_elt(kp + ((size_t)(ky * K + kx) * H + y) * W + x) * ld_elt(gp + (size_t)y * W + x);
                }
        }
        st_elt(gin + e, s);
    }
    for (size_t e = tid; e < n_k; e += stride) {
        const int x = e % W, y = (e / W) % H, k = (e / ((size_t)H * W)) % (K * K);
        const size_t plane = e / ((size_t)K * K * H * W);
        if constexpr (REPL) {
            const T *ip = in + plane * H * W + (size_t)min(max(y + k / K - P, 0), H - 1) * W + min(max(x + k % K - P, 0), W - 1);
            st_elt(gker + e, ld_elt(ip) * ld_elt(gout + (plane * H + y) * W + x));
        } else {
            st_elt(gker + e, ld_elt(in + (plane * Hi + y + k / K) * Wi + x + k % K) * ld_elt(gout + (plane * H + y) * W + x));
        }
    }
}

// ------------------------------------------------------------------ dispatch ---
struct FacPlan {
    int px;            // 4, 1, or 0 = generic
    FacDims d;
    int threads;
};

int env_int(const char *name, int dflt)
{
    const char *s = getenv(name);
    return (s && *s) ? atoi(s) : dflt;
}

// Rows per segment: enough CTAs for several waves, segments at least K-1 (and 4) rows tall.
int choose_seg(int planes, int H, int K)
{
    int seg = env_int("EBFI_FAC_SEG", 0);
    if (seg <= 0) {
        seg = 16;
        while (seg < H && (long)planes * ceil_div(H, seg) > 32768) seg *= 2;
    }
    if (seg < 4) seg = 4;
    if (seg < K - 1) seg = K - 1;
    if (seg > H) seg = H;
    return seg;
}

FacPlan make_plan(const void *const *ptrs, int nptr, int planes, int H, int W, int K, bool backward, int esize,
                  bool repl = false)
{
    FacPlan p{};
    p.d.H = H; p.d.W = W;
    const bool k_ok = (K == 1 || K == 3 || K == 5 || K == 7);
    bool al = true;
    for (int i = 0; i < nptr; ++i) al = al && ebfi::aligned16(ptrs[i]);
    // K = 7 at 4 px/thread needs more than 255 registers; it runs on the 1 px/thread variant.
    if (k_ok && K <= 5 && W % 4 == 0 && al) p.px = 4;
    else if (k_ok) p.px = 1;
    else p.px = 0;
    if (env_int("EBFI_FAC_FORCE_PX", -1) >= 0 && p.px != 0) {
        const int f = env_int("EBFI_FAC_FORCE_PX", -1);
        if (f == 0 || f == 1) p.px = f;
    }
    if (p.px == 0) return p;
    const int seg = choose_seg(planes, H, K);
    // the last segment must be the only one allowed to be shorter than K-1 rows (see merge)
    p.d.seg_rows = seg;
    p.d.nseg = ceil_div(H, seg);
    const int cols = ceil_div(W, p.px);
    p.d.nstage = 0;
    p.d.xstride = 0; p.d.halo_thr = 0;
    if (backward) {
        // One CTA per row segment up to 64 threads (256 columns at 4 px/thread: the shape the kernel was
        // tuned on); wider rows become overlapping column blocks of 64 threads. The overlap covers the
        // K-1 halo columns, rounded up so that a block's first column stays 16-byte aligned. With the pad folded
        // in (repl) it covers Q + P columns, Q = P rounded up to px (see fac_bwd_march).
        const int blk_thr = env_int("EBFI_FAC_BLOCK_THREADS", 64);
        if (cols <= blk_thr) {
            p.threads = ebfi::round_up(cols, 32);
            p.d.nxb = 1;
        } else {
            const int align_px = std::max(p.px, 16 / esize);                       // columns per 16 bytes
            const int P = (K - 1) / 2;
            const int halo_cols = ebfi::round_up(std::max(repl ? ebfi::round_up(P, p.px) + P : K - 1, 1), align_px);
            p.threads = blk_thr;
            p.d.halo_thr = ceil_div(halo_cols, p.px);
            p.d.xstride = blk_thr * p.px - p.d.halo_thr * p.px;
            p.d.nxb = ceil_div(W - p.d.halo_thr * p.px, p.d.xstride);
        }
        // ring variant: 2 stages (one row being consumed, one in flight). Measured on B200 at the
        // benchmark shape: 2 stages = 4 CTAs/SM -> 0.600 ms (91 % of HBM peak); 3 or 4 stages = 2 CTAs/SM
        // -> 0.763 ms; register variant 0.687 ms. Resident CTAs matter more than ring depth.
        if (p.px == 4 && (K == 3 || K == 5) && env_int("EBFI_FAC_RING", 1)) {
            const size_t stage = (size_t)(K * K + 1) * p.threads * p.px * esize;
            const int want = env_int("EBFI_FAC_STAGES", 0);
            // bulk copies move multiples of 16 bytes from 16-byte aligned addresses
            const bool rows16 = ((size_t)W * esize) % 16 == 0 && ((size_t)p.d.xstride * esize) % 16 == 0;
            if (!rows16) p.d.nstage = 0;
            else if (want >= 2 && want <= 4 && want * stage <= 200 * 1024) p.d.nstage = want;
            else if (2 * stage <= 72 * 1024) p.d.nstage = 2;      // >= 3 CTAs per SM, else the register variant
        }
    } else {
        p.threads = cols >= 128 ? 128 : ebfi::round_up(cols, 32);
        p.d.nxb = ceil_div(cols, p.threads);
    }
    return p;
}

// REPL launches never see K = 1 (the impls run the plain op there: a pad of 0 is no pad).
template <int PX, bool REPL, typename T>
int launch_fwd(cudaStream_t st, const FacPlan &p, const T *in, const T *ker, T *out,
               int planes, int K)
{
    const unsigned grid = (unsigned)((size_t)planes * p.d.nseg * p.d.nxb);
    switch (K) {
    case 1: if constexpr (!REPL) { fac_fwd_march<1, PX, false, T><<<grid, p.threads, 0, st>>>(in, ker, out, p.d); break; }
            return ebfi::fail(EBFI_ERR_INVALID, "fac: K=1 has no pad to fold");
    case 3: fac_fwd_march<3, PX, REPL, T><<<grid, p.threads, 0, st>>>(in, ker, out, p.d); break;
    case 5: fac_fwd_march<5, PX, REPL, T><<<grid, p.threads, 0, st>>>(in, ker, out, p.d); break;
    case 7: if constexpr (PX == 1) { fac_fwd_march<7, 1, REPL, T><<<grid, p.threads, 0, st>>>(in, ker, out, p.d); break; }
            return ebfi::fail(EBFI_ERR_INVALID, "fac: K=7 runs 1 px/thread only");
    default: return ebfi::fail(EBFI_ERR_INVALID, "fac: unsupported K=%d in march path", K);
    }
    EBFI_LAUNCH_OK("fac_fwd_march");
    return EBFI_OK;
}

template <int PX, bool REPL, typename T>
int launch_bwd(cudaStream_t st, const FacPlan &p, const T *in, const T *ker,
               const T *gout, T *gin, T *gker, int *counters, float *overhang,
               int planes, int K)
{
    const unsigned grid = (unsigned)((size_t)planes * p.d.nseg * p.d.nxb);
    const int RS = K > 1 ? K - 1 : 1;
    const size_t xch = (size_t)((2 * p.threads * RS + 31) & ~31) * sizeof(float);
    const size_t row = REPL ? (size_t)((p.threads * PX + K - 1 + 31) & ~31) * sizeof(float) : 0;   // srow
    const size_t smem = xch + row + (size_t)p.d.nstage * (K * K + 1) * p.threads * PX * sizeof(T);
#define EBFI_FAC_BWD(KK, RING)                                                                              \
    do {                                                                                                    \
        auto kern = fac_bwd_march<KK, PX, RING, REPL, T>;                                                      \
        EBFI_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
        kern<<<grid, p.threads, smem, st>>>(in, ker, gout, gin, gker, counters, overhang, p.d);            \
    } while (0)
    if (p.d.nstage > 0) {
        if constexpr (PX == 4) {
            if (K == 5) EBFI_FAC_BWD(5, true);
            else if (K == 3) EBFI_FAC_BWD(3, true);
            else return ebfi::fail(EBFI_ERR_INVALID, "fac: ring variant handles K = 3, 5");
        } else {
            return ebfi::fail(EBFI_ERR_INVALID, "fac: ring variant needs 4 px/thread");
        }
    } else {
        switch (K) {
        case 1: if constexpr (!REPL) { EBFI_FAC_BWD(1, false); break; }
                return ebfi::fail(EBFI_ERR_INVALID, "fac: K=1 has no pad to fold");
        case 3: EBFI_FAC_BWD(3, false); break;
        case 5: EBFI_FAC_BWD(5, false); break;
        case 7: if constexpr (PX == 1) { EBFI_FAC_BWD(7, false); break; }
                return ebfi::fail(EBFI_ERR_INVALID, "fac: K=7 runs 1 px/thread only");
        default: return ebfi::fail(EBFI_ERR_INVALID, "fac: unsupported K=%d in march path", K);
        }
    }
#undef EBFI_FAC_BWD
    EBFI_LAUNCH_OK("fac_bwd_march");
    return EBFI_OK;
}

int check_dims(int B, int C, int H, int W, int K)
{
    EBFI_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "fac: non-positive size B=%d C=%d H=%d W=%d", B, C, H, W);
    EBFI_REQUIRE(K > 0 && (K & 1), "fac: kernel_size must be odd and positive, got %d", K);
    EBFI_REQUIRE((long)B * C < (1L << 24), "fac: B*C too large");
    return EBFI_OK;
}

size_t ws_counter_bytes(int planes, int nseg)
{
    return ebfi::round_up((size_t)planes * (size_t)(nseg > 1 ? nseg - 1 : 1) * sizeof(int), (size_t)256);
}

// REPL: `input` is (B, C, H, W) and ReplicationPad2d((K-1)/2) is folded into the kernels.
template <typename T, bool REPL = false>
int fac_forward_impl(void *stream, const T *input, const T *kernel, T *output,
                     int batch, int channels, int height_out, int width_out, int kernel_size)
{
    if (int rc = check_dims(batch, channels, height_out, width_out, kernel_size)) return rc;
    EBFI_REQUIRE(input && kernel && output, "fac_forward: null pointer");
    if (REPL && kernel_size == 1)
        return fac_forward_impl<T>(stream, input, kernel, output, batch, channels, height_out, width_out, 1);
    const int planes = batch * channels, H = height_out, W = width_out, K = kernel_size;
    cudaStream_t st = ebfi::as_stream(stream);
    const void *ptrs[] = {kernel, output};
    const FacPlan p = make_plan(ptrs, 2, planes, H, W, K, false, (int)sizeof(T));
    if (p.px == 4) return launch_fwd<4, REPL, T>(st, p, input, kernel, output, planes, K);
    if (p.px == 1) return launch_fwd<1, REPL, T>(st, p, input, kernel, output, planes, K);
    const size_t n = (size_t)planes * H * W;
    const unsigned grid = (unsigned)std::min((size_t)ebfi::sm_count() * 16, ceil_div(n, (size_t)256));
    fac_fwd_generic<REPL, T><<<grid, 256, 0, st>>>(input, kernel, output, planes, H, W, K);
    EBFI_LAUNCH_OK("fac_fwd_generic");
    return EBFI_OK;
}

// REPL: `input` and `grad_input` are (B, C, H, W); the workspace is the padded op's
// (ebfi_fac_backward_workspace_bytes): same segments, same overhang rows.
template <typename T, bool REPL = false>
int fac_backward_impl(void *stream, const T *input, const T *kernel, const T *grad_output, T *grad_input,
                      T *grad_kernel, int batch, int channels, int height_out, int width_out, int kernel_size,
                      void *workspace, size_t workspace_bytes)
{
    if (int rc = check_dims(batch, channels, height_out, width_out, kernel_size)) return rc;
    EBFI_REQUIRE(input && kernel && grad_output && grad_input && grad_kernel, "fac_backward: null pointer");
    if (REPL && kernel_size == 1)
        return fac_backward_impl<T>(stream, input, kernel, grad_output, grad_input, grad_kernel, batch, channels,
                                           height_out, width_out, 1, workspace, workspace_bytes);
    const int planes = batch * channels, H = height_out, W = width_out, K = kernel_size;
    cudaStream_t st = ebfi::as_stream(stream);
    const void *ptrs[] = {kernel, grad_output, grad_kernel, grad_input};
    const FacPlan p = make_plan(ptrs, 4, planes, H, W, K, true, (int)sizeof(T), REPL);
    if (p.px == 0) {
        const size_t n = (size_t)planes * K * K * H * W;
        const unsigned grid = (unsigned)std::min((size_t)ebfi::sm_count() * 16, ceil_div(n, (size_t)256));
        fac_bwd_generic<REPL, T><<<grid, 256, 0, st>>>(input, kernel, grad_output, grad_input, grad_kernel, planes, H, W, K);
        EBFI_LAUNCH_OK("fac_bwd_generic");
        return EBFI_OK;
    }
    int *counters = nullptr;
    float *overhang = nullptr;
    if (p.d.nseg > 1 && K > 1) {
        const size_t cb = ws_counter_bytes(planes, p.d.nseg);
        const size_t need = cb + (size_t)planes * (p.d.nseg - 1) * (K - 1) * (size_t)(W + K - 1) * sizeof(float);
        if (!workspace || workspace_bytes < need)
            return ebfi::fail(EBFI_ERR_WORKSPACE, "fac_backward: workspace %zu < %zu bytes", workspace_bytes, need);
        EBFI_REQUIRE(ebfi::aligned16(workspace), "fac_backward: workspace must be 16-byte aligned");
        counters = static_cast<int *>(workspace);
        overhang = reinterpret_cast<float *>(static_cast<char *>(workspace) + cb);
        EBFI_CUDA_OK(cudaMemsetAsync(counters, 0, (size_t)planes * (p.d.nseg - 1) * sizeof(int), st));
    }
    if (p.px == 4)
        return launch_bwd<4, REPL, T>(st, p, input, kernel, grad_output, grad_input, grad_kernel, counters, overhang, planes, K);
    return launch_bwd<1, REPL, T>(st, p, input, kernel, grad_output, grad_input, grad_kernel, counters, overhang, planes, K);
}

}  // namespace

extern "C" {

int ebfi_fac_forward(void *stream, const float *input, const float *kernel, float *output,
                     int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<float>(stream, input, kernel, output, batch, channels, height_out, width_out, kernel_size);
}

int ebfi_fac_forward_bf16(void *stream, const void *input, const void *kernel, void *output,
                          int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<bf16>(stream, static_cast<const bf16 *>(input), static_cast<const bf16 *>(kernel),
                                  static_cast<bf16 *>(output), batch, channels, height_out, width_out, kernel_size);
}

int ebfi_fac_forward_fp16(void *stream, const void *input, const void *kernel, void *output,
                          int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<fp16>(stream, static_cast<const fp16 *>(input), static_cast<const fp16 *>(kernel),
                                  static_cast<fp16 *>(output), batch, channels, height_out, width_out, kernel_size);
}

size_t ebfi_fac_backward_workspace_bytes(int batch, int channels, int height_out, int width_out,
                                         int kernel_size)
{
    if (batch <= 0 || channels <= 0 || height_out <= 0 || width_out <= 0 || kernel_size <= 1) return 256;
    const int planes = batch * channels, R = kernel_size - 1;
    const int nseg = ceil_div(height_out, choose_seg(planes, height_out, kernel_size));
    if (nseg <= 1) return 256;
    return ws_counter_bytes(planes, nseg) +
           (size_t)planes * (nseg - 1) * R * (size_t)(width_out + R) * sizeof(float);
}

int ebfi_fac_backward(void *stream, const float *input, const float *kernel,
                      const float *grad_output, float *grad_input, float *grad_kernel,
                      int batch, int channels, int height_out, int width_out, int kernel_size,
                      void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<float>(stream, input, kernel, grad_output, grad_input, grad_kernel, batch, channels,
                                    height_out, width_out, kernel_size, workspace, workspace_bytes);
}

int ebfi_fac_backward_bf16(void *stream, const void *input, const void *kernel, const void *grad_output,
                           void *grad_input, void *grad_kernel, int batch, int channels, int height_out,
                           int width_out, int kernel_size, void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<bf16>(stream, static_cast<const bf16 *>(input), static_cast<const bf16 *>(kernel),
                                   static_cast<const bf16 *>(grad_output), static_cast<bf16 *>(grad_input),
                                   static_cast<bf16 *>(grad_kernel), batch, channels, height_out, width_out,
                                   kernel_size, workspace, workspace_bytes);
}

int ebfi_fac_backward_fp16(void *stream, const void *input, const void *kernel, const void *grad_output,
                           void *grad_input, void *grad_kernel, int batch, int channels, int height_out,
                           int width_out, int kernel_size, void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<fp16>(stream, static_cast<const fp16 *>(input), static_cast<const fp16 *>(kernel),
                                   static_cast<const fp16 *>(grad_output), static_cast<fp16 *>(grad_input),
                                   static_cast<fp16 *>(grad_kernel), batch, channels, height_out, width_out,
                                   kernel_size, workspace, workspace_bytes);
}

// ReplicationPad2d((K-1)/2) + FAC in one op: input and grad_input are (B, C, H, W)
int ebfi_fac_replpad_forward(void *stream, const float *input, const float *kernel, float *output,
                             int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<float, true>(stream, input, kernel, output, batch, channels, height_out, width_out, kernel_size);
}

int ebfi_fac_replpad_forward_bf16(void *stream, const void *input, const void *kernel, void *output,
                                  int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<bf16, true>(stream, static_cast<const bf16 *>(input), static_cast<const bf16 *>(kernel),
                                        static_cast<bf16 *>(output), batch, channels, height_out, width_out, kernel_size);
}

int ebfi_fac_replpad_forward_fp16(void *stream, const void *input, const void *kernel, void *output,
                                  int batch, int channels, int height_out, int width_out, int kernel_size)
{
    return fac_forward_impl<fp16, true>(stream, static_cast<const fp16 *>(input), static_cast<const fp16 *>(kernel),
                                        static_cast<fp16 *>(output), batch, channels, height_out, width_out, kernel_size);
}

int ebfi_fac_replpad_backward(void *stream, const float *input, const float *kernel,
                              const float *grad_output, float *grad_input, float *grad_kernel,
                              int batch, int channels, int height_out, int width_out, int kernel_size,
                              void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<float, true>(stream, input, kernel, grad_output, grad_input, grad_kernel, batch, channels,
                                          height_out, width_out, kernel_size, workspace, workspace_bytes);
}

int ebfi_fac_replpad_backward_bf16(void *stream, const void *input, const void *kernel, const void *grad_output,
                                   void *grad_input, void *grad_kernel, int batch, int channels, int height_out,
                                   int width_out, int kernel_size, void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<bf16, true>(stream, static_cast<const bf16 *>(input), static_cast<const bf16 *>(kernel),
                                         static_cast<const bf16 *>(grad_output), static_cast<bf16 *>(grad_input),
                                         static_cast<bf16 *>(grad_kernel), batch, channels, height_out, width_out,
                                         kernel_size, workspace, workspace_bytes);
}

int ebfi_fac_replpad_backward_fp16(void *stream, const void *input, const void *kernel, const void *grad_output,
                                   void *grad_input, void *grad_kernel, int batch, int channels, int height_out,
                                   int width_out, int kernel_size, void *workspace, size_t workspace_bytes)
{
    return fac_backward_impl<fp16, true>(stream, static_cast<const fp16 *>(input), static_cast<const fp16 *>(kernel),
                                         static_cast<const fp16 *>(grad_output), static_cast<fp16 *>(grad_input),
                                         static_cast<fp16 *>(grad_kernel), batch, channels, height_out, width_out,
                                         kernel_size, workspace, workspace_bytes);
}

}  // extern "C"
