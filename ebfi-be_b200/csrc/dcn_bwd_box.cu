// dcn_bwd_box.cu — DCNv2 backward from TMA-staged boxes: shared-memory gather, shared-memory (integer) scatter, both weight
// contractions on the sm_100a tensor cores, grad_input without global atomics for every sample inside the box.
//
// One persistent CTA per SM. CTA (s, h) owns the 8-channel units [h*GPC, h*GPC + GPC) (a unit = one deformable group when the
// group has 8 channels, else a part of it: its offsets / masks are the group's) and walks the 8 x 16-pixel output tiles
// s, s+S, ...; an "iteration" is one (tile, unit) — written (tile, group) below. Per tile the grad_output tile is staged
// ONCE, as bf16 hi/lo pairs in the layout Q[co][px]. The same bytes serve both contractions because kind::f16 accepts MN-major operands in the
// no-swizzle core-matrix layout (probed: tests/test_tcgen05_gpu.py):
//   GEMM1  colgrad[128 px x 72] = gO_tile . W_g        A = Q read MN-major (M = px, K = co), B = W_g^T image (bulk copy)
//   GEMM3  gW_g[co x 72]      += gO_tile^T . col       A = [Q_hi ; Q_lo] stacked to M = 128 (K = px), B = col read MN-major
// so the second grad_output copy of dcn_bwd_tc.cu is gone, a thread writes its 8 column values as ONE 16-byte chunk, and
// two MMAs per K step yield all four hi/lo products (rows 0-63 and 64-127 of the accumulator are two partial sums).
// GEMM3 accumulates in TMEM over all tiles of the CTA; an all-ones column gives grad_bias.
// Warps: 12 samplers (thread = (pixel, tap row)) + 1 issuer that runs every tcgen05 / TMA / bulk-copy instruction, signalled
// through mbarriers, so that no sampler waits for a single-thread issue loop. Per iteration:
//   * input: a 24 x 30-pixel box of the group-blocked input arrives by one 3-D TMA copy (zeros outside the image = the
//     reference's per-corner bounds tests, im2col_cuda.cu:38-48); the four corners of a sample are read with eight
//     conflict-free LDS.128 in the rotated order of dcn_box.cuh. Offsets and masks of the tile arrive by two more copies.
//     Everything is issued two iterations ahead.
//   * grad_mask / grad_offset: one owner thread per element, no atomics (im2col_cuda.cu:280-330).
//   * grad_input (im2col_cuda.cu:197-254): contributions are accumulated in a shared-memory box of the same geometry as
//     32-bit FIXED POINT (native ATOMS.ADD; a float shared atomic is a CAS loop), with a power-of-two scale chosen per
//     (tile, group) in a first pass over the samples: M = max |colgrad * mask| and n = the largest number of contributions
//     any box cell receives (one integer atomic per sample into a count box) bound every element by n * M, so
//     scale = 2^30 / (n * M) cannot overflow and resolves a contribution to ~2^-24 of M (n is ~40). Integer addition is
//     associative, so the box is bit-reproducible.
//     The box is written — converted back to fp32 — as a dense partial to global memory with plain coalesced stores;
//     dcn_gin_collect then sums, per input pixel, the <= 3 x 2 boxes that cover it in a fixed order and writes NCHW. No global
//     atomics, no order dependence: grad_input is bit-identical run to run, by default.
//   * samples whose corners leave the box (|offset| beyond ~7 pixels) fall back to 256-bit global loads and
//     red.global.add.v4.f32 into a blocked fp32 buffer that dcn_gin_collect adds last (order-dependent only then, like
//     the reference's atomicAdd, im2col_cuda.cu:249).
// Non-finite gradients: a NaN/Inf anywhere in the (tile, group) makes the scale undefined; the box is then written as NaN
// so that overflow checks on grad_input (AMP GradScaler) still fire.
// Activation type T (float | __nv_bfloat16 | __half, the *_bf16 / *_fp16 entries): offsets, masks and grad_output are
// read as T and widened (a bf16 grad_output splits into hi = the value, lo = 0, an fp16 one exactly into bf16 hi + lo:
// the bits the float path stages for the widened tensor); grad_offset / grad_mask and grad_input are rounded once from
// the fp32 values the float instantiation stores. With several units per group the running fp32 sums of the owner
// threads then stay in shared memory until the group's last unit. Boxes, partials, weights and grad_weight / grad_bias
// are fp32 in all three.
#include "dcn_box.cuh"
#include "dcn_common.cuh"
#include "dp_comm.cuh"
#include "tma.cuh"
#include "umma.cuh"

#include <algorithm>
#include <type_traits>

namespace ebfi_dcn {

namespace {

using ebfi::ceil_div;

constexpr int TM = 128, TH = 8, TW = 16, NR = 3;
constexpr int NSAMP = TM * NR, NSW = NSAMP / 32;        // sampler threads / warps
constexpr int NTHR = NSAMP + 32;                       // + the issuer warp (tensor core, TMA)
constexpr int CS = 8, CO = 64;                  // channels per group, output channels handled by this kernel
constexpr int GPC_MAX = 4;                      // deformable groups per CTA (TMEM: 2 * N1 + GPC * N3 <= 512 columns)
constexpr int TMEM_COLS = 512;
constexpr int Q_PART = CO * TM * 2;             // one bf16 image of the grad_output tile
constexpr int BOX_F = box::BYTES / 4;           // floats per box
constexpr int CNT_BYTES = box::BH * box::BW * 4; // per-cell sample counts of one iteration
constexpr int CNT_PAD = (CNT_BYTES + 127) / 128 * 128;

struct BoxBwdPlan {
    int TPR;             // taps per thread row
    int Kc;              // CS * KK
    int N1, N3;          // GEMM1 / GEMM3 N (multiples of 16)
    int GPC, NH;         // units per CTA, CTA rows
    int tiles_x, tiles_y, ntiles;
    int my, mx;          // box margins above / left of the tile's undeformed footprint
    int wt_bytes;        // one group's W^T image, hi | lo
    int col_part;        // one bf16 image of the column operand
    int om_bytes, use_om_tma;
    int off_q, off_col, off_box, off_acc, off_cnt, off_om, off_gsum, smem;
    int units, ncs, ncs_shift;      // 8-channel units (C / 8) = iterations per tile over all CTA rows; units per deformable group (2^shift)
};

__device__ __forceinline__ void st_bf16x8(unsigned char *base, int off, const unsigned short (&v)[8])
{
    const uint32_t a = v[0] | ((uint32_t)v[1] << 16), b = v[2] | ((uint32_t)v[3] << 16);
    const uint32_t c = v[4] | ((uint32_t)v[5] << 16), e = v[6] | ((uint32_t)v[7] << 16);
    *reinterpret_cast<uint4 *>(base + off) = make_uint4(a, b, c, e);
}

// (a, b) -> packed bf16 pairs hi = {bf16(a), bf16(b)}, lo = {bf16(a - hi_a), bf16(b - hi_b)}; a in the low half
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t &hi, uint32_t &lo)
{
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xFFFF0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
// eight floats -> one 16-byte chunk of bf16 hi parts and one of lo parts
__device__ __forceinline__ void st_split8(unsigned char *hi_base, unsigned char *lo_base, int off, const float (&v)[8])
{
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split_bf16x2(v[2 * i], v[2 * i + 1], h[i], l[i]);
    *reinterpret_cast<uint4 *>(hi_base + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4 *>(lo_base + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

__device__ __forceinline__ void sampler_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NSAMP) : "memory"); }

__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float e)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(e) : "memory");
}

__device__ __forceinline__ void atoms_add(uint32_t saddr, int v)
{
    asm volatile("red.shared.add.s32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}

// Where a sample lands in a box whose first cell is image pixel (by0, bx0).
struct Geo {
    bool inside;         // the sampling window of the reference (im2col_cuda.cu:180, :304); NaN coordinates fail it like they do there
    bool inbox;          // all four corners are cells of the box
    int yb, xb;          // box cell of corner (y0, x0)
    float hy, hx, ly, lx;
};
__device__ __forceinline__ Geo make_geo(float y, float x, int H, int W, int by0, int bx0)
{
    Geo q;
    q.inside = y > -1.f && x > -1.f && y < (float)H && x < (float)W;
    const float fy = floorf(y), fx = floorf(x);
    q.ly = y - fy; q.lx = x - fx; q.hy = 1.f - q.ly; q.hx = 1.f - q.lx;
    q.yb = (int)fy - by0; q.xb = (int)fx - bx0;
    q.inbox = q.inside && (unsigned)q.yb <= (unsigned)(box::BH - 2) && (unsigned)q.xb <= (unsigned)(box::BW - 2);
    return q;
}

// v'[j] = v[(j + k) & 3], k in 0..3, without dynamic register indexing
__device__ __forceinline__ void rot4(float (&v)[4], uint32_t k)
{
    if (k & 1u) { const float t = v[0]; v[0] = v[1]; v[1] = v[2]; v[2] = v[3]; v[3] = t; }
    if (k & 2u) { float t = v[0]; v[0] = v[2]; v[2] = t; t = v[1]; v[1] = v[3]; v[3] = t; }
}

// One sample (pixel, tap) of the backward: gather the four corners, grad_mask / grad_offset, the grad_input scatter and
// the recomputed column values (natural channel order). `gc` = colgrad of the tap's 8 channels.
struct SampleCtx {
    int ho, wo, by0, bx0, bxq0;
    uint32_t box_s, acc_s;
    const float *ib;     // blocked input plane of (sample, group): far-sample gathers
    float *gb;           // blocked far-sample accumulator of (sample, group)
    float scale;
};
template <bool PACKED>
__device__ __forceinline__ void sample_bwd(const DcnDims &d, const SampleCtx &sc, const float (&gc)[8], float dy, float dx, float m,
                                           int ti, int tj, int lane, uint32_t wrot, float (&colv)[8], float &g_y, float &g_x, float &g_m)
{
    const int ho = sc.ho, wo = sc.wo, by0 = sc.by0, bx0 = sc.bx0, bxq0 = sc.bxq0;
    const uint32_t box_s = sc.box_s, acc_s = sc.acc_s;
    const float *ib = sc.ib;
    float *gb = sc.gb;
    const float scale = sc.scale;
    m = mask_act_t<PACKED>(m);
    const float y = (float)(ho * d.sh - d.ph + ti * d.dh) + dy;
    const float x = (float)(wo * d.sw - d.pw + tj * d.dw) + dx;
    const Geo ge = make_geo(y, x, d.H, d.W, by0, bx0);
    const bool inside = ge.inside, inbox = ge.inbox;
    const float hy = ge.hy, hx = ge.hx, ly = ge.ly, lx = ge.lx;
    const int yb = ge.yb, xb = ge.xb;
    // A / B = the two 4-channel halves; in-box they are channels 0-3 / 4-7 unless `odd`, then swapped
    float va[4], vb[4], ya[4], yb4[4], xa[4], xb4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) va[j] = vb[j] = ya[j] = yb4[j] = xa[j] = xb4[j] = 0.f;
    bool odd = false;
    box::Rot rt{};
    if (inbox) {
        rt = box::make_rot(box_s, yb, xb, lane);
        odd = rt.odd;
        float wv[5], wyv[5], wxv[5];
        box::rot_corners(rt.c0, hy * hx, hy * lx, ly * hx, ly * lx, wv);       // bilinear weights
        box::rot_corners(rt.c0, -hx, -lx, hx, lx, wyv);                         // d/dy (im2col_cuda.cu:99-120)
        box::rot_corners(rt.c0, -hy, hy, -ly, ly, wxv);                         // d/dx
        // packed fp32x2 FMAs: accumulators [A | B half][value, d/dy, d/dx][channel pair]
        box::f32x2 acc[2][3][2] = {};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 q = box::lds128(box::step_addr(rt, i));
            const float cw = box::step_coef(wv, odd, i), cy = box::step_coef(wyv, odd, i), cx = box::step_coef(wxv, odd, i);
            const box::f32x2 q01 = box::pack2(q.x, q.y), q23 = box::pack2(q.z, q.w);
            box::f32x2 (&a)[3][2] = acc[i & 1];
            a[0][0] = box::ffma2(box::pack2(cw, cw), q01, a[0][0]); a[0][1] = box::ffma2(box::pack2(cw, cw), q23, a[0][1]);
            a[1][0] = box::ffma2(box::pack2(cy, cy), q01, a[1][0]); a[1][1] = box::ffma2(box::pack2(cy, cy), q23, a[1][1]);
            a[2][0] = box::ffma2(box::pack2(cx, cx), q01, a[2][0]); a[2][1] = box::ffma2(box::pack2(cx, cx), q23, a[2][1]);
        }
        box::unpack2(acc[0][0][0], va[0], va[1]); box::unpack2(acc[0][0][1], va[2], va[3]);
        box::unpack2(acc[1][0][0], vb[0], vb[1]); box::unpack2(acc[1][0][1], vb[2], vb[3]);
        box::unpack2(acc[0][1][0], ya[0], ya[1]); box::unpack2(acc[0][1][1], ya[2], ya[3]);
        box::unpack2(acc[1][1][0], yb4[0], yb4[1]); box::unpack2(acc[1][1][1], yb4[2], yb4[3]);
        box::unpack2(acc[0][2][0], xa[0], xa[1]); box::unpack2(acc[0][2][1], xa[2], xa[3]);
        box::unpack2(acc[1][2][0], xb4[0], xb4[1]); box::unpack2(acc[1][2][1], xb4[2], xb4[3]);
    } else if (inside) {
        const Tap tp = make_tap(y, x, d.H, d.W);
        const f8 a1 = ldg_f8(ib + (size_t)tp.i00 * CS, tp.c00), a2 = ldg_f8(ib + (size_t)tp.i01 * CS, tp.c01);
        const f8 a3 = ldg_f8(ib + (size_t)tp.i10 * CS, tp.c10), a4 = ldg_f8(ib + (size_t)tp.i11 * CS, tp.c11);
        const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            va[j] = w1 * a1.v[j] + w2 * a2.v[j] + w3 * a3.v[j] + w4 * a4.v[j];
            vb[j] = w1 * a1.v[4 + j] + w2 * a2.v[4 + j] + w3 * a3.v[4 + j] + w4 * a4.v[4 + j];
            ya[j] = -hx * a1.v[j] - lx * a2.v[j] + hx * a3.v[j] + lx * a4.v[j];
            yb4[j] = -hx * a1.v[4 + j] - lx * a2.v[4 + j] + hx * a3.v[4 + j] + lx * a4.v[4 + j];
            xa[j] = -hy * a1.v[j] + hy * a2.v[j] - ly * a3.v[j] + ly * a4.v[j];
            xb4[j] = -hy * a1.v[4 + j] + hy * a2.v[4 + j] - ly * a3.v[4 + j] + ly * a4.v[4 + j];
        }
    }
    float ta[4], tb[4];                  // colgrad * mask of the A / B halves
    {
        // channel pairs on the packed fp32x2 pipe; the two lanes of each sum are added at the end
        using box::f32x2;
        const f32x2 m2 = box::pack2(m, m);
        f32x2 sm2 = 0, sy2 = 0, sx2 = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {        // channel pairs (2h, 2h+1) of each half
            const f32x2 ga = box::pack2(odd ? gc[4 + 2 * h] : gc[2 * h], odd ? gc[5 + 2 * h] : gc[2 * h + 1]);
            const f32x2 gb2 = box::pack2(odd ? gc[2 * h] : gc[4 + 2 * h], odd ? gc[2 * h + 1] : gc[5 + 2 * h]);
            const f32x2 va2 = box::pack2(va[2 * h], va[2 * h + 1]), vb2 = box::pack2(vb[2 * h], vb[2 * h + 1]);
            sm2 = box::ffma2(ga, va2, sm2); sm2 = box::ffma2(gb2, vb2, sm2);           // grad_mask (im2col_cuda.cu:311)
            const f32x2 ta2 = box::fmul2(ga, m2), tb2 = box::fmul2(gb2, m2);
            box::unpack2(ta2, ta[2 * h], ta[2 * h + 1]); box::unpack2(tb2, tb[2 * h], tb[2 * h + 1]);
            sy2 = box::ffma2(box::pack2(ya[2 * h], ya[2 * h + 1]), ta2, sy2);           // grad_offset
            sy2 = box::ffma2(box::pack2(yb4[2 * h], yb4[2 * h + 1]), tb2, sy2);
            sx2 = box::ffma2(box::pack2(xa[2 * h], xa[2 * h + 1]), ta2, sx2);
            sx2 = box::ffma2(box::pack2(xb4[2 * h], xb4[2 * h + 1]), tb2, sx2);
            // recomputed column, natural channel order
            const f32x2 ca = box::fmul2(va2, m2), cb = box::fmul2(vb2, m2);
            box::unpack2(odd ? cb : ca, colv[2 * h], colv[2 * h + 1]);
            box::unpack2(odd ? ca : cb, colv[4 + 2 * h], colv[5 + 2 * h]);
        }
        float lo, hi;
        box::unpack2(sy2, lo, hi); g_y = lo + hi;
        box::unpack2(sx2, lo, hi); g_x = lo + hi;
        box::unpack2(sm2, lo, hi); g_m = (lo + hi) * mask_act_grad_t<PACKED>(m);
    }
    // ---- grad_input (im2col_cuda.cu:236-251); the scatter's x uses pad_h (:368)
    bool q_inside = inside, q_inbox = inbox, q_odd = odd;
    float qhx = hx, qlx = lx;
    float xs = x;
    box::Rot rq = rt;
    rq.base += acc_s - box_s;            // same cell of the accumulation box (both bases are 128-byte aligned)
    if (d.ph != d.pw) {
        xs = (float)(wo * d.sw - d.ph + tj * d.dw) + dx;
        const Geo gq = make_geo(y, xs, d.H, d.W, by0, bxq0);
        q_inside = gq.inside; q_inbox = gq.inbox;
        qlx = gq.lx; qhx = gq.hx;
        if (q_inbox) rq = box::make_rot(acc_s, gq.yb, gq.xb, lane);
        q_odd = rq.odd;
    }
    if (q_inbox) {
        if (q_odd != odd) {              // only when pad_h != pad_w moved the sample to a cell of the other parity
#pragma unroll
            for (int j = 0; j < 4; ++j) { const float tsw = ta[j]; ta[j] = tb[j]; tb[j] = tsw; }
        }
        // word rotation by the quarter-warp index on top of the chunk rotation: 32 lanes on 32 banks
        rot4(ta, wrot); rot4(tb, wrot);
        float qv[5];
        box::rot_corners(rq.c0, hy * qhx * scale, hy * qlx * scale, ly * qhx * scale, ly * qlx * scale, qv);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t a = box::step_addr(rq, i);
            const float cf = box::step_coef(qv, q_odd, i);
            const float *tt = (i & 1) ? tb : ta;
            float pr[4];
            box::unpack2(box::fmul2(box::pack2(cf, cf), box::pack2(tt[0], tt[1])), pr[0], pr[1]);
            box::unpack2(box::fmul2(box::pack2(cf, cf), box::pack2(tt[2], tt[3])), pr[2], pr[3]);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                atoms_add(a + ((((uint32_t)j + wrot) & 3u) << 2), __float2int_rn(pr[j]));
        }
    } else if (q_inside) {
        const Tap tq = make_tap(y, xs, d.H, d.W);
        const float q1 = tq.hy * tq.hx, q2 = tq.hy * tq.lx, q3 = tq.ly * tq.hx, q4 = tq.ly * tq.lx;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const float *tt = (hf == (odd ? 1 : 0)) ? ta : tb;      // natural half hf
            if (tq.c00) red_add_v4(gb + (size_t)tq.i00 * CS + 4 * hf, q1 * tt[0], q1 * tt[1], q1 * tt[2], q1 * tt[3]);
            if (tq.c01) red_add_v4(gb + (size_t)tq.i01 * CS + 4 * hf, q2 * tt[0], q2 * tt[1], q2 * tt[2], q2 * tt[3]);
            if (tq.c10) red_add_v4(gb + (size_t)tq.i10 * CS + 4 * hf, q3 * tt[0], q3 * tt[1], q3 * tt[2], q3 * tt[3]);
            if (tq.c11) red_add_v4(gb + (size_t)tq.i11 * CS + 4 * hf, q4 * tt[0], q4 * tt[1], q4 * tt[2], q4 * tt[3]);
        }
    }
}

// MULTI: more than one 8-channel unit per deformable group (the group's offset / mask gradients accumulate over its units)
template <bool PACKED, bool MULTI, typename T>
__global__ void __launch_bounds__(NTHR, 1)
dcn_bwd_box_kernel(const float *__restrict__ in_blk, const unsigned char *__restrict__ wimg,
                   const T *__restrict__ offset, const T *__restrict__ mask,
                   const T *__restrict__ gout, float *__restrict__ gin_blk, float *__restrict__ pbox,
                   T *__restrict__ goff, T *__restrict__ gmask,
                   float *__restrict__ gw_part, float *__restrict__ gb_part, DcnDims d, BoxBwdPlan pl,
                   const __grid_constant__ CUtensorMap tm_box, const __grid_constant__ CUtensorMap tm_off,
                   const __grid_constant__ CUtensorMap tm_mask)
{
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *wring = smem;                                     // [2][hi | lo][N1 rows k'][CO], K-major
    unsigned char *q_hi = smem + pl.off_q, *q_lo = q_hi + Q_PART;    // [co][px] bf16: K-major for GEMM3, MN-major for GEMM1
    unsigned char *c_hi = smem + pl.off_col, *c_lo = c_hi + pl.col_part;   // [tap][px][8 ch] bf16: MN-major B of GEMM3
    unsigned char *boxes = smem + pl.off_box;                        // [2][BH][BW][8] fp32 input boxes
    int4 *acc4 = reinterpret_cast<int4 *>(smem + pl.off_acc);        // [BH][BW][8] fixed-point grad_input box
    int *cnt = reinterpret_cast<int *>(smem + pl.off_cnt);           // [2][BH][BW] samples per cell (first corner), by iteration parity
    const T *oms = reinterpret_cast<const T *>(smem + pl.off_om);           // [2][3*KK planes][128 px]
    constexpr bool RUN_SUMS = MULTI && sizeof(T) != 4;
    float *gsum = reinterpret_cast<float *>(smem + pl.off_gsum);             // RUN_SUMS: [3*KK][128 px] fp32 running sums
    // bar_w / bar_in: bulk copies landed; bar_d1: GEMM1 complete; bar_g3: GEMM3 complete (Q, col free);
    // q_full / col_full: the sampler warps have written Q / the column operand (one arrival per warp)
    __shared__ __align__(8) uint64_t bar_w[2], bar_in[2], bar_d1[2], bar_g3, q_full, col_full;
    __shared__ uint32_t tmem_slot;
    __shared__ unsigned tile_max[2];
    __shared__ int w_max[2];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int p = tid % TM, r = tid / TM;             // samplers: thread (pixel p, tap row r)
    const int S = gridDim.x, s = blockIdx.x;
    const int g_begin = blockIdx.y * pl.GPC, ng = min(pl.GPC, pl.units - g_begin);     // this CTA's 8-channel units
    const int total_tiles = d.B * pl.ntiles;
    const int NI = ((total_tiles - s + S - 1) / S) * ng;             // iterations (tile, group) of this CTA
    const int npix = d.Ho * d.Wo, Kdim = d.C * d.KK;
    const size_t plane = (size_t)npix, in_plane = (size_t)d.H * d.W;
    const unsigned uplane = (unsigned)plane;
    const bool use_tma = pl.use_om_tma != 0;
    const int t_first = r * pl.TPR, ti_first = t_first / d.kw, tj_first = t_first - ti_first * d.kw;

    if (warp == 0) umma::tmem_alloc<TMEM_COLS>(&tmem_slot);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) { umma::mbar_init(&bar_w[i], 1); umma::mbar_init(&bar_in[i], 1); umma::mbar_init(&bar_d1[i], 1); }
        umma::mbar_init(&bar_g3, 1); umma::mbar_init(&q_full, NSW); umma::mbar_init(&col_full, NSW);
        umma::mbar_fence_init();
        tile_max[0] = tile_max[1] = 0u;
        w_max[0] = w_max[1] = 0;
    }
    for (int c = tid; c < BOX_F / 4; c += NTHR) acc4[c] = make_int4(0, 0, 0, 0);
    for (int c = tid; c < 2 * CNT_PAD / 4; c += NTHR) cnt[c] = 0;
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = (uint32_t)(warp & 3) * 32u;
    const uint32_t idesc1 = umma::instr_desc_bf16(TM, pl.N1) | (1u << 15);     // A MN-major
    const uint32_t idesc3 = umma::instr_desc_bf16(TM, pl.N3) | (1u << 16);     // B MN-major
    const uint32_t q_s = umma::smem_u32(q_hi), c_s = umma::smem_u32(c_hi), w_s = umma::smem_u32(wring);
    const uint32_t acc_s = umma::smem_u32(acc4), cnt_s = umma::smem_u32(cnt);
    const uint32_t wrot = (uint32_t)lane >> 3;

    // iteration n of this CTA = (tile s + (n / ng) * S, group g_begin + n % ng)
    // g: 8-channel unit (channels 8g .. 8g+7); its deformable group (offsets / masks) is g >> ncs_shift
    struct Iter { int n, b, ty0, tx0, g, gi, tl, ho, wo, pix; bool valid; };
    auto set_tile = [&](Iter &it, int tile) {       // divisions once per tile
        it.b = tile / pl.ntiles;
        it.tl = tile - it.b * pl.ntiles;
        const int tyi = it.tl / pl.tiles_x;
        it.ty0 = tyi * TH;
        it.tx0 = (it.tl - tyi * pl.tiles_x) * TW;
        it.ho = it.ty0 + p / TW; it.wo = it.tx0 + p % TW;
        it.valid = it.ho < d.Ho && it.wo < d.Wo;
        it.pix = it.ho * d.Wo + it.wo;
    };
    auto decode = [&](int n) {
        Iter it;
        it.n = n;
        const int k = n / ng;
        it.gi = n - k * ng;
        it.g = g_begin + it.gi;
        set_tile(it, s + k * S);
        return it;
    };
    auto next_iter = [&](const Iter &c) {           // iteration c.n + 1
        Iter it = c;
        ++it.n;
        if (++it.gi == ng) {
            it.gi = 0;
            set_tile(it, s + (it.n / ng) * S);
        }
        it.g = g_begin + it.gi;
        return it;
    };
    // ---- issue helpers: run by all lanes of the issuer warp (warp-uniform arithmetic), the elected lane issues
    const bool leader = warp == NSW && umma::elect_one();
    auto issue_in = [&](int n) {                    // input box + offsets / masks of iteration n
        const Iter it = decode(n);
        const int bb = n & 1;
        if (!leader) return;
        umma::mbar_expect_tx(&bar_in[bb], (uint32_t)(box::BYTES + (use_tma ? pl.om_bytes : 0)));
        tma::load_3d(boxes + bb * box::BYTES, &tm_box, (it.tx0 * d.sw - d.pw - pl.mx) * 8, it.ty0 * d.sh - d.ph - pl.my, it.b * pl.units + it.g, &bar_in[bb]);
        if (use_tma) {
            unsigned char *dst = smem + pl.off_om + bb * pl.om_bytes;
            tma::load_3d(dst, &tm_off, it.tx0, it.ty0, it.b * d.off_bp + (MULTI ? it.g >> pl.ncs_shift : it.g) * 2 * d.KK, &bar_in[bb]);
            tma::load_3d(dst + 2 * d.KK * TM * (int)sizeof(T), &tm_mask, it.tx0, it.ty0, it.b * d.mask_bp + (MULTI ? it.g >> pl.ncs_shift : it.g) * d.KK, &bar_in[bb]);
        }
    };
    auto issue_w = [&](int n) {                     // W^T image of iteration n's group
        const int g = g_begin + n % ng;
        if (!leader) return;
        umma::mbar_expect_tx(&bar_w[n & 1], (uint32_t)pl.wt_bytes);
        umma::bulk_g2s(wring + (n & 1) * pl.wt_bytes, wimg + (size_t)g * pl.wt_bytes, (uint32_t)pl.wt_bytes, &bar_w[n & 1]);
    };
    auto issue_gemm1 = [&](int n) {                 // D1[n & 1][px][k'] = Q^T . W^T   (K = co)
        umma::mbar_wait(&bar_w[n & 1], (uint32_t)((n >> 1) & 1));
        const uint32_t d1 = tmem + (uint32_t)((n & 1) * pl.N1);
        const uint32_t wb = w_s + (uint32_t)((n & 1) * pl.wt_bytes), wlo = (uint32_t)(pl.N1 * CO * 2);
        for (int ks = 0; ks < CO / 16; ++ks) {
            // A: 16-byte chunks run along px (SBO 128 between chunks), 8-co groups 2048 B apart (LBO)
            const uint64_t ah = umma::smem_desc(q_s + ks * 4096u, 2048, 128), al = umma::smem_desc(q_s + Q_PART + ks * 4096u, 2048, 128);
            const uint64_t bh = umma::smem_desc(wb + ks * 256u, 128, (CO / 8) * 128), bl = umma::smem_desc(wb + wlo + ks * 256u, 128, (CO / 8) * 128);
            if (leader) {
                umma::mma_f16(d1, al, bh, idesc1, ks > 0);
                umma::mma_f16(d1, ah, bl, idesc1, true);
                umma::mma_f16(d1, ah, bh, idesc1, true);
            }
        }
        if (leader) umma::commit(&bar_d1[n & 1]);
        __syncwarp();
    };
    auto issue_gemm3 = [&](int gi, bool accumulate) {   // D3[gi][hi rows | lo rows][k'] += [Q_hi ; Q_lo] . col^T   (K = px)
        const uint32_t d3 = tmem + (uint32_t)(2 * pl.N1 + gi * pl.N3);
        for (int ks = 0; ks < TM / 16; ++ks) {
            const uint64_t a = umma::smem_desc(q_s + ks * 256u, 128, (TM / 8) * 128);
            // B: 16-byte chunks run along k' (one tap = one chunk, SBO 2048 between taps), 8-px groups 128 B apart (LBO)
            const uint64_t bh = umma::smem_desc(c_s + ks * 256u, 128, TM * 16), bl = umma::smem_desc(c_s + pl.col_part + ks * 256u, 128, TM * 16);
            if (leader) {
                umma::mma_f16(d3, a, bh, idesc3, accumulate || ks > 0);
                umma::mma_f16(d3, a, bl, idesc3, true);
            }
        }
        if (leader) umma::commit(&bar_g3);
        __syncwarp();
    };

    uint32_t ph_g3 = 0;
    // ================= new tile: grad_output -> Q (bf16 hi / lo), once for all groups of the CTA =================
    // item = (co, chunk of 8 consecutive tile pixels); lanes run over co % 8 first -> conflict-free 16-byte stores.
    // All loads of a thread are issued before the wait for the previous tile's last GEMM3 (which still reads Q and col).
    constexpr int QI = (CO * (TM / 8) + NSAMP - 1) / NSAMP;
    auto tile_start = [&](const Iter &it, bool wait_g3) {
        const T *go_b = gout + (size_t)it.b * d.Co * plane;
        float4 va[QI], vb[QI];
        const bool vec = d.Wo % (16 / (int)sizeof(T)) == 0;    // 8 pixels = whole 16-byte words
#pragma unroll
        for (int q = 0; q < QI; ++q) {
            const int item = tid + q * NSAMP;
            va[q] = vb[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (item < CO * (TM / 8)) {
                const int j = item & 7, pc = (item >> 3) & (TM / 8 - 1), co = (item >> 7) * 8 + j;
                const int hh = it.ty0 + (pc * 8) / TW, ww = it.tx0 + (pc * 8) % TW;
                const T *src = go_b + (size_t)co * plane + (size_t)hh * d.Wo + ww;
                if (vec && hh < d.Ho && ww + 7 < d.Wo) {
                    if constexpr (sizeof(T) == 4) {
                        va[q] = __ldg(reinterpret_cast<const float4 *>(src));
                        vb[q] = __ldg(reinterpret_cast<const float4 *>(src) + 1);
                    } else if constexpr (std::is_same_v<T, __half>) {
                        const uint4 u = __ldg(reinterpret_cast<const uint4 *>(src));     // fp16 -> fp32: exact conversion
                        const __half2 *h = reinterpret_cast<const __half2 *>(&u);
                        const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
                        const float2 c = __half22float2(h[2]), e = __half22float2(h[3]);
                        va[q] = make_float4(a.x, a.y, b.x, b.y);
                        vb[q] = make_float4(c.x, c.y, e.x, e.y);
                    } else {
                        const uint4 u = __ldg(reinterpret_cast<const uint4 *>(src));     // bf16 -> fp32: the bits move up
                        va[q] = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u),
                                            __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xFFFF0000u));
                        vb[q] = make_float4(__uint_as_float(u.z << 16), __uint_as_float(u.z & 0xFFFF0000u),
                                            __uint_as_float(u.w << 16), __uint_as_float(u.w & 0xFFFF0000u));
                    }
                } else if (hh < d.Ho) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = (ww + i < d.Wo) ? ld_act(src + i) : 0.f;
                    va[q] = make_float4(v[0], v[1], v[2], v[3]); vb[q] = make_float4(v[4], v[5], v[6], v[7]);
                }
            }
        }
        if (wait_g3) {
            umma::mbar_wait(&bar_g3, ph_g3);
            ph_g3 ^= 1u;
        }
#pragma unroll
        for (int q = 0; q < QI; ++q) {
            const int item = tid + q * NSAMP;
            if (item < CO * (TM / 8)) {
                const int j = item & 7, pc = (item >> 3) & (TM / 8 - 1), co = (item >> 7) * 8 + j;
                const float v[8] = {va[q].x, va[q].y, va[q].z, va[q].w, vb[q].x, vb[q].y, vb[q].z, vb[q].w};
                st_split8(q_hi, q_lo, (co >> 3) * ((TM / 8) * 128) + pc * 128 + j * 16, v);
            }
        }
        // column chunks past the taps: the ones column (grad_bias) and zero padding up to N3
        for (int c = tid; c < (pl.N3 / 8 - d.KK) * TM; c += NSAMP) {
            const int pp = c % TM, ch = d.KK + c / TM;
            const bool one = ch == d.KK && (it.ty0 + pp / TW) < d.Ho && (it.tx0 + pp % TW) < d.Wo;
            *reinterpret_cast<uint4 *>(c_hi + ch * (TM * 16) + pp * 16) = make_uint4(one ? 0x3F80u : 0u, 0u, 0u, 0u);   // bf16(1.0)
            *reinterpret_cast<uint4 *>(c_lo + ch * (TM * 16) + pp * 16) = make_uint4(0u, 0u, 0u, 0u);
        }
        umma::fence_smem_to_async();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&q_full);
    };
    // ================= pass 1 of an iteration: M = max |colgrad * mask| (unsigned order of the float bits: NaN > Inf > finite,
    // so a non-finite value anywhere is seen) and the per-cell sums of the scatter's bilinear weights (rounded up, 16.16) ======
    struct P1 { const T *om, *off_g, *mask_g; uint32_t d1, cnt_s; int by0, bxq0; };
    auto pass1_begin = [&](const Iter &it) {
        const int bb = it.n & 1;
        const uint32_t par = (uint32_t)((it.n >> 1) & 1);
        umma::mbar_wait(&bar_d1[bb], par);           // colgrad of this group is in TMEM
        umma::fence_after_sync();
        umma::mbar_wait(&bar_in[bb], par);           // box + offsets / masks have landed
        P1 q;
        q.om = oms + bb * (pl.om_bytes / (int)sizeof(T));
        q.off_g = offset + (size_t)it.b * d.off_bs + (size_t)(MULTI ? it.g >> pl.ncs_shift : it.g) * 2 * d.KK * plane;
        q.mask_g = mask + (size_t)it.b * d.mask_bs + (size_t)(MULTI ? it.g >> pl.ncs_shift : it.g) * d.KK * plane;
        q.d1 = tmem + (uint32_t)(bb * pl.N1);
        q.cnt_s = cnt_s + (uint32_t)(bb * CNT_PAD);
        q.by0 = it.ty0 * d.sh - d.ph - pl.my; q.bxq0 = it.tx0 * d.sw - d.ph - pl.mx;
        return q;
    };
    auto pass1_tap = [&](const Iter &it, const P1 &q, int t, int ti, int tj, unsigned &um) {
        float gc[8];
        umma::tmem_ld8(umma::tmem_addr(q.d1, lane_base, t * 8), gc);
        umma::tmem_ld_wait();
        if (it.valid) {
            float dy, dx, m;
            if (use_tma) {
                dy = act_f(q.om[(2 * t) * TM + p]);
                dx = act_f(q.om[(2 * t + 1) * TM + p]);
                m = act_f(q.om[(2 * d.KK + t) * TM + p]);
            } else {
                tap_read(q.off_g, q.mask_g, uplane, (unsigned)t, (unsigned)it.pix, dy, dx, m);
            }
            m = mask_act_t<PACKED>(m);
#pragma unroll
            for (int cc = 0; cc < CS; ++cc) um = max(um, __float_as_uint(fabsf(gc[cc] * m)));
            // the scatter's x uses pad_h (im2col_cuda.cu:368)
            const Geo ge = make_geo((float)(it.ho * d.sh - d.ph + ti * d.dh) + dy, (float)(it.wo * d.sw - d.ph + tj * d.dw) + dx,
                                    d.H, d.W, q.by0, q.bxq0);
            if (ge.inbox) atoms_add(q.cnt_s + (uint32_t)(ge.yb * box::BW + ge.xb) * 4u, 1);
        }
    };
    auto pass1_end = [&](int bb, unsigned um) {
        um = __reduce_max_sync(0xffffffffu, um);
        if (lane == 0 && um) atomicMax(&tile_max[bb], um);
    };
    auto pass1 = [&](const Iter &it) {
        const P1 q = pass1_begin(it);
        unsigned um = 0u;
        int t = t_first, ti = ti_first, tj = tj_first;
        for (int sidx = 0; sidx < pl.TPR && t < d.KK; ++sidx, ++t) {
            pass1_tap(it, q, t, ti, tj, um);
            if (++tj == d.kw) { tj = 0; ++ti; }
        }
        pass1_end(it.n & 1, um);
    };
    // n_max = the largest number of contributions any box cell receives = max over cells (Y, X) of the samples whose first
    // corner is (Y, X), (Y, X-1), (Y-1, X) or (Y-1, X-1), from the counts pass 1 left in cnt[bb]
    auto cell_max = [&](int bb) {
        const int *cb = cnt + bb * (CNT_PAD / 4);
        int wm = 0;
        for (int c = tid; c < box::BH * box::BW; c += NSAMP) {
            const int yy = c / box::BW, xx = c - yy * box::BW;
            int v = cb[c];
            if (xx > 0) v += cb[c - 1];
            if (yy > 0) { v += cb[c - box::BW]; if (xx > 0) v += cb[c - box::BW - 1]; }
            wm = max(wm, v);
        }
        wm = __reduce_max_sync(0xffffffffu, wm);
        if (lane == 0 && wm) atomicMax(&w_max[bb], wm);
    };

    if (warp == NSW) {
        // ================= issuer warp: tensor-core and copy-engine work, off the samplers' critical path =================
        issue_w(0); issue_in(0);
        if (NI > 1) { issue_w(1); issue_in(1); }
        int gi = 0, k = 0;
        for (int n = 0; n < NI; ++n) {
            if (gi == 0) {
                umma::mbar_wait(&q_full, (uint32_t)(k & 1));         // Q of this tile is staged
                umma::fence_after_sync();
                issue_gemm1(n);
                if (ng > 1) issue_gemm1(n + 1);
                // the next tile's grad_output -> L2, so that its staging pays an L2 hit instead of a DRAM miss
                const int ntile = s + (k + 1) * S;
                if (ntile < total_tiles) {
                    const int nb = ntile / pl.ntiles, ntl = ntile - nb * pl.ntiles;
                    const int nty0 = (ntl / pl.tiles_x) * TH, ntx0 = (ntl % pl.tiles_x) * TW;
                    for (int c = lane; c < CO * TH; c += 32) {
                        const int co = c / TH, hh = nty0 + c % TH;
                        if (hh < d.Ho)
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(gout + ((size_t)nb * d.Co + co) * plane + (size_t)hh * d.Wo + ntx0));
                    }
                }
            }
            umma::mbar_wait(&bar_d1[n & 1], (uint32_t)((n >> 1) & 1));
            if (n + 2 < NI) issue_w(n + 2);                          // GEMM1(n) is complete: its weight slot is free
            umma::mbar_wait(&col_full, (uint32_t)(n & 1));           // pass 2 of iteration n is done in every sampler warp
            umma::fence_after_sync();
            issue_gemm3(gi, n >= ng);                                // the first tile of the CTA starts the accumulation
            if (n + 2 < NI) {
                issue_in(n + 2);                                     // box / offset buffers of this iteration are free
                if (gi + 2 < ng) issue_gemm1(n + 2);                 // same tile: Q is staged (else: at the tile start), D1 slot is free
            }
            if (++gi == ng) { gi = 0; ++k; }
        }
    } else {
    // ================= sampler warps =================
    Iter cur = decode(0);
    if (NI > 0) {
        tile_start(cur, false);
        pass1(cur);
        sampler_sync();
        cell_max(0);
        sampler_sync();
    }
    for (int n = 0; n < NI; ++n) {
        const int bb = n & 1;
        const Iter nxt = n + 1 < NI ? next_iter(cur) : cur;
        const bool has_next = n + 1 < NI, next_same_tile = has_next && nxt.gi != 0;
        // ---- fixed-point scale of this (tile, group): every element |sum| <= n_max * (M * scale + 1/2) <= 2^30 + 2^10
        const unsigned tmax = tile_max[bb];
        const bool nonfinite = tmax >= 0x7F800000u;
        int e2 = 0;
        if (tmax && !nonfinite) frexpf(__uint_as_float(tmax), &e2);      // M < 2^e2
        const int wbits = 32 - __clz(max(w_max[bb], 1));                 // contributions per element < 2^wbits
        const int k2 = max(-126, min(126, 30 - wbits - e2));            // 2^k2 and 2^-k2 are normal fp32 numbers
        const float inv_scale = ldexpf(1.f, -k2);
        // ================= pass 2: the samples =================
        {
            SampleCtx sc;
            sc.ho = cur.ho; sc.wo = cur.wo;
            sc.by0 = cur.ty0 * d.sh - d.ph - pl.my; sc.bx0 = cur.tx0 * d.sw - d.pw - pl.mx; sc.bxq0 = cur.tx0 * d.sw - d.ph - pl.mx;
            sc.box_s = umma::smem_u32(boxes + bb * box::BYTES); sc.acc_s = acc_s;
            sc.ib = in_blk + ((size_t)cur.b * pl.units + cur.g) * in_plane * CS;
            sc.gb = gin_blk + ((size_t)cur.b * pl.units + cur.g) * in_plane * CS;
            sc.scale = ldexpf(1.f, k2);
            const T *om = oms + bb * (pl.om_bytes / (int)sizeof(T));
            const T *off_g = offset + (size_t)cur.b * d.off_bs + (size_t)(MULTI ? cur.g >> pl.ncs_shift : cur.g) * 2 * d.KK * plane;
            const T *mask_g = mask + (size_t)cur.b * d.mask_bs + (size_t)(MULTI ? cur.g >> pl.ncs_shift : cur.g) * d.KK * plane;
            T *goff_g = goff + (size_t)cur.b * d.off_bs + (size_t)(MULTI ? cur.g >> pl.ncs_shift : cur.g) * 2 * d.KK * plane;
            T *gmask_g = gmask + (size_t)cur.b * d.mask_bs + (size_t)(MULTI ? cur.g >> pl.ncs_shift : cur.g) * d.KK * plane;
            const uint32_t d1 = tmem + (uint32_t)(bb * pl.N1);
            // pass 1 of the next group of the same tile is interleaved tap by tap (its colgrad was issued two iterations
            // ago): two independent instruction streams per warp; a new tile needs its Q first
            P1 q1{};
            unsigned um = 0u;
            if (next_same_tile) q1 = pass1_begin(nxt);
            int t = t_first, ti = ti_first, tj = tj_first;
            // rolled on purpose: unrolling it (three samples in flight per thread) measured slower on B200 (238 vs 230 us)
#pragma unroll 1
            for (int sidx = 0; sidx < pl.TPR && t < d.KK; ++sidx, ++t) {
                if (next_same_tile) pass1_tap(nxt, q1, t, ti, tj, um);
                float gc[8];
                umma::tmem_ld8(umma::tmem_addr(d1, lane_base, t * 8), gc);     // colgrad[p][t*8 .. t*8+7]
                umma::tmem_ld_wait();
                float colv[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) colv[j] = 0.f;
                if (cur.valid) {
                    float dy, dx, m;
                    if (use_tma) {
                        dy = act_f(om[(2 * t) * TM + p]);
                        dx = act_f(om[(2 * t + 1) * TM + p]);
                        m = act_f(om[(2 * d.KK + t) * TM + p]);
                    } else {
                        tap_read(off_g, mask_g, uplane, (unsigned)t, (unsigned)cur.pix, dy, dx, m);
                    }
                    float g_y, g_x, g_m;
                    sample_bwd<PACKED>(d, sc, gc, dy, dx, m, ti, tj, lane, wrot, colv, g_y, g_x, g_m);
                    // more than 8 channels per deformable group: the group's units follow each other in this CTA and the
                    // same thread owns the element in each of them -> plain read-modify-write, fixed order
                    T *gy = goff_g + (2u * (unsigned)t * uplane + (unsigned)cur.pix);
                    if constexpr (RUN_SUMS) {
                        // 16-bit outputs: the running sums stay fp32 (same additions as below), one rounding at the last unit
                        float *gs = gsum + 3 * t * TM + p;
                        if (cur.g & (pl.ncs - 1)) { g_y += gs[0]; g_x += gs[TM]; g_m += gs[2 * TM]; }
                        if ((cur.g & (pl.ncs - 1)) != pl.ncs - 1) {
                            gs[0] = g_y; gs[TM] = g_x; gs[2 * TM] = g_m;
                        } else {
                            gy[0] = st_act<T>(g_y); gy[uplane] = st_act<T>(g_x);
                            gmask_g[(unsigned)t * uplane + (unsigned)cur.pix] = st_act<T>(g_m);
                        }
                    } else {
                        if (MULTI && (cur.g & (pl.ncs - 1))) {
                            g_y += act_f(gy[0]); g_x += act_f(gy[uplane]); g_m += act_f(gmask_g[(unsigned)t * uplane + (unsigned)cur.pix]);
                        }
                        gy[0] = st_act<T>(g_y); gy[uplane] = st_act<T>(g_x);
                        gmask_g[(unsigned)t * uplane + (unsigned)cur.pix] = st_act<T>(g_m);
                    }
                }
                // column operand: the 8 channels of (tap t, pixel p) are one 16-byte chunk. col is read by GEMM3 of the
                // previous iteration until bar_g3 completes: waited for here, behind the first sample's gather and scatter
                if (sidx == 0 && cur.gi != 0) {
                    umma::mbar_wait(&bar_g3, ph_g3);
                    ph_g3 ^= 1u;
                }
                st_split8(c_hi, c_lo, t * (TM * 16) + p * 16, colv);
                if (++tj == d.kw) { tj = 0; ++ti; }
            }
            if (cur.gi != 0 && t_first >= d.KK) {        // a tap row without taps keeps its barrier phase in step
                umma::mbar_wait(&bar_g3, ph_g3);
                ph_g3 ^= 1u;
            }
            if (next_same_tile) pass1_end(bb ^ 1, um);
        }
        umma::fence_smem_to_async();
        umma::fence_before_sync();                       // orders this thread's tcgen05.ld of D1 before the arrival
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&col_full);
        sampler_sync();                                  // the accumulation box is complete
        if (tid == 0) { tile_max[bb] = 0u; w_max[bb] = 0; }
        // ---- the accumulation box -> dense fp32 partial (plain coalesced stores), cleared for the next iteration
        {
            float4 *dst = reinterpret_cast<float4 *>(pbox + (((size_t)cur.b * pl.ntiles + cur.tl) * pl.units + cur.g) * BOX_F);
            const float qnan = __uint_as_float(0x7FC00000u);
            for (int c = tid; c < box::BH * box::BW; c += NSAMP) cnt[bb * (CNT_PAD / 4) + c] = 0;    // read by cell_max an interval ago
            for (int c = tid; c < BOX_F / 4; c += NSAMP) {
                const int4 v = acc4[c];
                acc4[c] = make_int4(0, 0, 0, 0);
                dst[c] = nonfinite ? make_float4(qnan, qnan, qnan, qnan)
                                   : make_float4((float)v.x * inv_scale, (float)v.y * inv_scale, (float)v.z * inv_scale, (float)v.w * inv_scale);
            }
        }
        if (next_same_tile) {
            cell_max(bb ^ 1);
        } else if (has_next) {
            tile_start(nxt, true);
            pass1(nxt);
            sampler_sync();
            cell_max(bb ^ 1);
        }
        sampler_sync();
        cur = nxt;
    }
    // ---- partials of this CTA, [slot][k = (c0 + cc) * KK + tap][co] so that a warp writes 128 contiguous bytes:
    //      rows 0-63 of D3 (Q_hi products) -> slot 2s, rows 64-127 (Q_lo products) -> slot 2s+1
    if (NI > 0) {
        umma::mbar_wait(&bar_g3, ph_g3);
        umma::fence_after_sync();
    }
    {
        const int row = (int)lane_base + lane, half = row >> 6, co = row & 63;
        const size_t slot = (size_t)2 * s + half;
        for (int gi = 0; gi < ng; ++gi) {
            const int c0 = (g_begin + gi) * CS;
            for (int cb = r * 8; cb < pl.N3; cb += NR * 8) {
                float v[8];
                if (NI > 0) {
                    umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, 2 * pl.N1 + gi * pl.N3 + cb), v);
                    umma::tmem_ld_wait();
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = 0.f;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int kp = cb + i;
                    if (kp < pl.Kc)
                        gw_part[(slot * Kdim + (size_t)(c0 + (kp & 7)) * d.KK + (kp >> 3)) * CO + co] = v[i];
                    else if (kp == pl.Kc && g_begin + gi == 0)
                        gb_part[slot * CO + co] = v[i];
                }
            }
        }
    }
    }   // sampler warps
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tmem);
}

// grad_weight[co][k] = sum over the slots of part[slot][k][co], grad_bias likewise: fixed order (four interleaved slot
// quarters per element, combined in a fixed order), coalesced reads along co.
// DP: the first half of the data-parallel all-reduce of the two gradients is part of this kernel — the local sums also
// are stored into every peer's symmetric buffer over NVLink and the last block raises the peers' flags (dp_comm.cuh: no NCCL
// call, no bucket copies). The outputs hold the local sums until ebfi_dp_complete adds the peers' in rank order.
template <int DP>
__global__ void __launch_bounds__(256)
dcn_box_reduce_partials(const float *__restrict__ gw_part, const float *__restrict__ gb_part,
                        float *__restrict__ gw, float *__restrict__ gb, int nslot, int Kdim, ebfi_dp::View v)
{
    const int e = blockIdx.x * (blockDim.x / 4) + (threadIdx.x >> 2), q = threadIdx.x & 3;
    const int n_w = Kdim * CO;
    float a = 0.f;
    if (e < n_w) {
        for (int sl = q; sl < nslot; sl += 4) a += gw_part[(size_t)sl * n_w + e];
    } else if (e < n_w + CO) {
        for (int sl = q; sl < nslot; sl += 4) a += gb_part[(size_t)sl * CO + (e - n_w)];
    }
    const float b1 = __shfl_xor_sync(0xffffffffu, a, 1);
    a = (q & 1) ? b1 + a : a + b1;           // (q0 + q1), (q2 + q3): the same operand order in both lanes
    const float b2 = __shfl_xor_sync(0xffffffffu, a, 2);
    a = (q & 2) ? b2 + a : a + b2;
    unsigned epoch = 0;
    if (DP) {
        epoch = ebfi_dp::epoch_of_launch(v);
        // in the order of the outputs (grad_weight | grad_bias): ebfi_dp_complete works on those two tensors
        if (q == 0 && e < n_w + CO) ebfi_dp::push(v, epoch, e < n_w ? (size_t)(e % CO) * Kdim + e / CO : (size_t)e, a);
    }
    if (q == 0) {
        if (e < n_w) gw[(size_t)(e % CO) * Kdim + e / CO] = a;
        else if (e < n_w + CO) gb[e - n_w] = a;
    }
    if (DP) ebfi_dp::publish(v, epoch);
}

// W^T images for the bulk copies: [group][hi | lo][N1 rows k'][CO] bf16 in the K-major core-matrix order,
// k' = tap * 8 + cc  <-  weight[co][(g * 8 + cc) * KK + tap]; zero rows past Kc.
__global__ void dcn_bwd_prep_weights(const float *__restrict__ weight, unsigned short *__restrict__ wimg, DcnDims d, BoxBwdPlan pl)
{
    const int per = pl.N1 * CO, Kdim = d.C * d.KK;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < pl.units * per; i += gridDim.x * blockDim.x) {
        const int g = i / per, e = i - g * per;
        const int j = e & 7, rr = (e >> 3) & 7, rest = e >> 6;
        const int kc = rest % (CO / 8), rg = rest / (CO / 8);
        const int kp = rg * 8 + rr, co = kc * 8 + j;
        unsigned short hi = 0, lo = 0;
        if (kp < pl.Kc)
            umma::split_bf16(__ldg(weight + (size_t)co * Kdim + (size_t)(g * CS + (kp & 7)) * d.KK + (kp >> 3)), hi, lo);
        wimg[(size_t)g * 2 * per + e] = hi;
        wimg[(size_t)g * 2 * per + per + e] = lo;
    }
}

// grad_input[b][g*8 + c][y][x] = sum, in a fixed order, over the boxes that cover (y, x) + the far-sample buffer.
// One thread per (b, g, y, x): 32 contiguous bytes per box, coalesced along x; NCHW plane stores.
template <typename T>
__global__ void dcn_gin_collect(const float *__restrict__ pbox, const float *__restrict__ gin_blk, T *__restrict__ gin,
                                DcnDims d, BoxBwdPlan pl)
{
    const int HW = d.H * d.W;
    const size_t n = (size_t)d.B * pl.units * HW;
    const int sy = TH * d.sh, sx = TW * d.sw;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t bg = i / HW;
        const int px = (int)(i - bg * HW), b = (int)(bg / pl.units), g = (int)(bg - (size_t)b * pl.units);
        const int y = px / d.W, x = px - y * d.W;
        const float4 *fp = reinterpret_cast<const float4 *>(gin_blk + i * CS);
        float4 a0 = __ldg(fp), a1 = __ldg(fp + 1);
        // box of tile (ty, tx): rows [ty*sy - ph - my, +BH), pixels [tx*sx - ph - mx, +BW)   (pad_h for x too, :368)
        const int ny = y + d.ph + pl.my, nx = x + d.ph + pl.mx;
        const int ty_hi = min(pl.tiles_y - 1, ny / sy), tx_hi = min(pl.tiles_x - 1, nx / sx);
        const int ty_lo = ny - (box::BH - 1) <= 0 ? 0 : (ny - (box::BH - 1) + sy - 1) / sy;
        const int tx_lo = nx - (box::BW - 1) <= 0 ? 0 : (nx - (box::BW - 1) + sx - 1) / sx;
        // at most ceil(BH / 8) x ceil(BW / 16) = 3 x 2 boxes cover a pixel: all loads are issued before the first add,
        // the additions keep the fixed (ty, tx) order
        constexpr int NY = (box::BH + TH - 1) / TH, NX = (box::BW + TW - 1) / TW;
        float4 u0[NY * NX], u1[NY * NX];
#pragma unroll
        for (int a = 0; a < NY; ++a)
#pragma unroll
            for (int c = 0; c < NX; ++c) {
                const int ty = ty_lo + a, tx = tx_lo + c;
                u0[a * NX + c] = u1[a * NX + c] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ty <= ty_hi && tx <= tx_hi) {
                    const size_t bx = ((size_t)b * pl.ntiles + (size_t)ty * pl.tiles_x + tx) * pl.units + g;
                    const int cell = (ny - ty * sy) * box::BW + (nx - tx * sx);
                    const float4 *bp = reinterpret_cast<const float4 *>(pbox + bx * BOX_F + (size_t)cell * CS);
                    u0[a * NX + c] = __ldg(bp); u1[a * NX + c] = __ldg(bp + 1);
                }
            }
#pragma unroll
        for (int q = 0; q < NY * NX; ++q) {
            a0.x += u0[q].x; a0.y += u0[q].y; a0.z += u0[q].z; a0.w += u0[q].w;
            a1.x += u1[q].x; a1.y += u1[q].y; a1.z += u1[q].z; a1.w += u1[q].w;
        }
        T *dp = gin + bg * CS * HW + px;
        dp[0] = st_act<T>(a0.x); dp[(size_t)HW] = st_act<T>(a0.y); dp[(size_t)2 * HW] = st_act<T>(a0.z); dp[(size_t)3 * HW] = st_act<T>(a0.w);
        dp[(size_t)4 * HW] = st_act<T>(a1.x); dp[(size_t)5 * HW] = st_act<T>(a1.y); dp[(size_t)6 * HW] = st_act<T>(a1.z); dp[(size_t)7 * HW] = st_act<T>(a1.w);
    }
}

// act_bytes: size of one activation element (4 or 2). It sets the offset / mask planes in shared memory and the TMA
// row alignment; with 2 (bf16 outputs) and several units per group the owners' fp32 running sums take the bytes saved.
bool make_plan(const DcnDims &d, BoxBwdPlan &pl, int act_bytes = 4)
{
    if (d.cpg % CS != 0 || d.Co != CO || d.det) return false;
    pl.units = d.C / CS;
    pl.ncs = d.cpg / CS;
    if (pl.ncs & (pl.ncs - 1)) return false;             // units per group: a power of two (1, 2, 4)
    pl.ncs_shift = 0;
    while ((1 << pl.ncs_shift) < pl.ncs) ++pl.ncs_shift;
    if (getenv("EBFI_DCN_BWD_NO_BOX")) return false;
    if ((long)2 * d.KK * d.Ho * d.Wo >= (1L << 31) || d.KK > 15) return false;       // 32-bit offsets; <= 2^11 contributions per element
    if ((long)d.B * pl.units >= (1L << 31) || (long)d.W * 8 >= (1L << 31)) return false;
    pl.TPR = ceil_div(d.KK, NR);
    pl.Kc = CS * d.KK;
    pl.N1 = ebfi::round_up(pl.Kc, 16);
    pl.N3 = ebfi::round_up(pl.Kc + 1, 16);
    pl.GPC = std::min({GPC_MAX, pl.units, (TMEM_COLS - 2 * pl.N1) / pl.N3});
    if (pl.GPC < 1 || pl.N1 > 256 || pl.N3 > 256) return false;
    // all units of a deformable group run in ONE CTA (their grad_offset / grad_mask sums are accumulated by the owner thread)
    if (pl.GPC % pl.ncs != 0) return false;
    pl.NH = ceil_div(pl.units, pl.GPC);
    pl.tiles_x = ceil_div(d.Wo, TW);
    pl.tiles_y = ceil_div(d.Ho, TH);
    pl.ntiles = pl.tiles_x * pl.tiles_y;
    // the undeformed footprint of a tile (+1 for the second bilinear row / pixel) must fit the box; margins centre it
    const int fh = (TH - 1) * d.sh + (d.kh - 1) * d.dh + 1, fw = (TW - 1) * d.sw + (d.kw - 1) * d.dw + 1;
    if (fh > box::BH - 1 || fw > box::BW - 1) return false;
    pl.my = (box::BH - 1 - fh + 1) / 2;
    pl.mx = (box::BW - 1 - fw + 1) / 2;
    pl.wt_bytes = 2 * pl.N1 * CO * 2;
    pl.col_part = (pl.N3 / 8) * TM * 16;
    pl.om_bytes = 3 * d.KK * TM * act_bytes;
    pl.use_om_tma = d.Wo % (16 / act_bytes) == 0 && getenv("EBFI_DCN_NO_TMA") == nullptr;
    pl.off_q = 2 * pl.wt_bytes;
    pl.off_col = pl.off_q + 2 * Q_PART;
    pl.off_box = pl.off_col + 2 * pl.col_part;
    pl.off_acc = pl.off_box + 2 * box::BYTES;
    pl.off_cnt = pl.off_acc + box::BYTES;
    pl.off_om = pl.off_cnt + 2 * CNT_PAD;
    pl.off_gsum = pl.off_om + 2 * pl.om_bytes;
    pl.smem = pl.off_gsum + (act_bytes != 4 && pl.ncs > 1 ? 3 * d.KK * TM * 4 : 0);
    return pl.smem <= 226 * 1024;
}

int box_splits(const DcnDims &d, const BoxBwdPlan &pl)
{
    return std::max(1, std::min(d.B * pl.ntiles, ebfi::sm_count() / pl.NH));
}

}  // namespace

// Number of [Co][C*KK] partial slots the box backward writes (two per CTA column), 0 when the shape is not covered.
int backward_box_splits(const DcnDims &d)
{
    BoxBwdPlan pl{};
    if (!make_plan(d, pl)) return 0;
    return 2 * box_splits(d, pl);
}

// scratch: blocked input | blocked far-sample accumulator | W^T images | dense partial boxes
size_t backward_box_scratch_bytes(const DcnDims &d)
{
    BoxBwdPlan pl{};
    if (!make_plan(d, pl)) return 0;
    const size_t n = (size_t)d.B * d.C * d.H * d.W;
    return 2 * n * sizeof(float) + ebfi::round_up((size_t)pl.units * pl.wt_bytes, (size_t)256) +
           (size_t)d.B * pl.ntiles * pl.units * box::BYTES;
}

template <typename T>
int backward_box(cudaStream_t st, const DcnDims &d, const T *input, const float *weight, const T *offset,
                 const T *mask, const T *gout, T *gin, T *goff, T *gmask, float *gw, float *gb,
                 float *gw_part, float *gb_part, void *scratch, const ebfi_dp::View *dp, bool dp_defer)
{
    BoxBwdPlan pl{};
    if (!make_plan(d, pl, (int)sizeof(T))) return EBFI_ERR_UNSUPPORTED;
    const size_t n = (size_t)d.B * d.C * d.H * d.W;
    float *in_blk = static_cast<float *>(scratch), *gin_blk = in_blk + n;
    unsigned char *wimg = reinterpret_cast<unsigned char *>(gin_blk + n);
    float *pbox = reinterpret_cast<float *>(wimg + ebfi::round_up((size_t)pl.units * pl.wt_bytes, (size_t)256));
    const int BG = d.B * pl.units, HW = d.H * d.W;
    if (d.in_blocked) {
        // the caller kept the forward's blocked copy (EBFI_DCN_INPUT_BLOCKED): only the far-sample accumulator is cleared
        in_blk = const_cast<float *>(reinterpret_cast<const float *>(input));
        EBFI_CUDA_OK(cudaMemsetAsync(gin_blk, 0, n * sizeof(float), st));
    } else if (int rc = launch_nchw_to_blocked(st, input, in_blk, BG, HW, gin_blk, 2)) {
        return rc;       // blocked copy of the input + zero fill of the far-sample accumulator in one pass
    }
    dcn_bwd_prep_weights<<<ceil_div(pl.units * pl.N1 * CO, 256), 256, 0, st>>>(weight, reinterpret_cast<unsigned short *>(wimg), d, pl);
    EBFI_LAUNCH_OK("dcn_bwd_prep_weights");

    CUtensorMap tm_box{}, tm_off{}, tm_mask{};
    {
        const uint64_t dims[3] = {(uint64_t)d.W * 8, (uint64_t)d.H, (uint64_t)BG};
        const uint64_t str[2] = {(uint64_t)d.W * 32, (uint64_t)HW * 32};
        const uint32_t bx[3] = {box::BW * 8, box::BH, 1};
        if (int rc = tma::encode_3d(tm_box, in_blk, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dims, str, bx)) return rc;
    }
    if (pl.use_om_tma && !(ebfi::aligned16(offset) && ebfi::aligned16(mask))) pl.use_om_tma = 0;
    if (pl.use_om_tma) {
        constexpr CUtensorMapDataType om_type = tma::elem_type<T>();
        const uint64_t str[2] = {(uint64_t)d.Wo * sizeof(T), (uint64_t)d.Ho * d.Wo * sizeof(T)};
        const uint64_t dims_o[3] = {(uint64_t)d.Wo, (uint64_t)d.Ho, (uint64_t)(d.B - 1) * d.off_bp + 2 * d.dg * d.KK};
        const uint64_t dims_m[3] = {(uint64_t)d.Wo, (uint64_t)d.Ho, (uint64_t)(d.B - 1) * d.mask_bp + d.dg * d.KK};
        const uint32_t box_o[3] = {TW, TH, (uint32_t)(2 * d.KK)}, box_m[3] = {TW, TH, (uint32_t)d.KK};
        if (int rc = tma::encode_3d(tm_off, offset, om_type, dims_o, str, box_o)) return rc;
        if (int rc = tma::encode_3d(tm_mask, mask, om_type, dims_m, str, box_m)) return rc;
    }
    dim3 grid(box_splits(d, pl), pl.NH);
#define EBFI_BWD_BOX(P, M)                                                                                             \
    do {                                                                                                               \
        EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_bwd_box_kernel<P, M, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem)); \
        dcn_bwd_box_kernel<P, M, T><<<grid, NTHR, pl.smem, st>>>(in_blk, wimg, offset, mask, gout, gin_blk, pbox, goff, gmask, \
                                                                 gw_part, gb_part, d, pl, tm_box, tm_off, tm_mask);    \
    } while (0)
    if (pl.ncs > 1) { if (d.packed) EBFI_BWD_BOX(true, true); else EBFI_BWD_BOX(false, true); }
    else            { if (d.packed) EBFI_BWD_BOX(true, false); else EBFI_BWD_BOX(false, false); }
#undef EBFI_BWD_BOX
    EBFI_LAUNCH_OK("dcn_bwd_box_kernel");
    const unsigned cgrid = (unsigned)std::min<size_t>(ceil_div((size_t)BG * HW, (size_t)256), (size_t)ebfi::sm_count() * 16);
    dcn_gin_collect<T><<<cgrid, 256, 0, st>>>(pbox, gin_blk, gin, d, pl);
    EBFI_LAUNCH_OK("dcn_gin_collect");
    const int Kdim = d.C * d.KK;
    const int rblocks = ceil_div(Kdim * CO + CO, 64);
    if (dp)
        dcn_box_reduce_partials<1><<<rblocks, 256, 0, st>>>(gw_part, gb_part, gw, gb, 2 * (int)grid.x, Kdim, *dp);
    else
        dcn_box_reduce_partials<0><<<rblocks, 256, 0, st>>>(gw_part, gb_part, gw, gb, 2 * (int)grid.x, Kdim, ebfi_dp::View{});
    EBFI_LAUNCH_OK("dcn_box_reduce_partials");
    if (dp && !dp_defer) return ebfi_dp::allreduce_sum(st, *dp, gw, (size_t)Kdim * CO, gb, (size_t)CO, 2);
    return EBFI_OK;
}
template int backward_box<float>(cudaStream_t, const DcnDims &, const float *, const float *, const float *, const float *,
                                 const float *, float *, float *, float *, float *, float *, float *, float *, void *,
                                 const ebfi_dp::View *, bool);
template int backward_box<__nv_bfloat16>(cudaStream_t, const DcnDims &, const __nv_bfloat16 *, const float *,
                                         const __nv_bfloat16 *, const __nv_bfloat16 *, const __nv_bfloat16 *, __nv_bfloat16 *,
                                         __nv_bfloat16 *, __nv_bfloat16 *, float *, float *, float *, float *, void *,
                                         const ebfi_dp::View *, bool);
template int backward_box<__half>(cudaStream_t, const DcnDims &, const __half *, const float *, const __half *,
                                  const __half *, const __half *, __half *, __half *, __half *, float *, float *,
                                  float *, float *, void *, const ebfi_dp::View *, bool);

}  // namespace ebfi_dcn
