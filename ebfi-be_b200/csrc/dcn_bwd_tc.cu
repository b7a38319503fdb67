// dcn_bwd_tc.cu — DCNv2 backward with both weight contractions on the sm_100a tensor cores.
//
// Group-specialised persistent CTAs, like the CUDA-core kernel in dcn.cu: CTA (s, g) owns
// deformable group g (8 channels x KK taps = the K' columns) and walks the 128-pixel tiles
// s, s+S, ... of all samples. Per tile, everything comes from ONE pass over the pixels:
//   GEMM1  colgrad[128 px x K'] = gO_tile[128 x Co] . W_g[Co x K']       (tcgen05, bf16x3, D1 in TMEM)
//   each thread (pixel p, tap) reads its 8 colgrad values straight from TMEM (lane = pixel),
//   gathers the 8 channels at the 4 bilinear corners and produces
//       grad_mask, grad_offset (one owner thread per element: no atomics, fixed order),
//       the grad_input scatter (fp32 red.global.add, like the reference's atomicAdd, :249),
//       and the recomputed column value * mask, written as the B operand of
//   GEMM3  gW_g[Co x K'] += gO_tile^T[Co x 128 px] . col[128 px x K']     (tcgen05, accumulates in TMEM
//          across ALL tiles of the CTA; an extra all-ones column yields grad_bias for free).
// At the end the CTA writes its [Co x K'] partial; dcn_reduce_partials (dcn.cu) sums the S partials
// in a fixed order. The reference runs 3 kernels + 3 cuBLAS GEMMs per sample and materialises the
// 151 MB column buffer twice (dcn_v2_cuda.cu:150-211).
//
// Operand precision: bf16 hi/lo pairs, 3 MMAs per product (umma.cuh) -> ~2^-16 relative, inside the
// 1e-4 gradient gate with a wide margin, at half the shared memory of TF32 pairs (two CTAs per SM).
// grad_output is needed in two K-major layouts ([px][co] for GEMM1, [co][px] for GEMM3) because
// kind::tf32/f16 MN-major no-swizzle operands are not usable (see DESIGN.md); the [px][co] copy
// shares its storage with the column operand, which is written only after GEMM1 has completed.
#include "dcn_common.cuh"
#include "tma.cuh"
#include "umma.cuh"

#include <algorithm>

namespace ebfi_dcn {

namespace {

using ebfi::ceil_div;

constexpr int TM = 128, TH = 8, TW = 16, NR = 3, NTHR = TM * NR;
constexpr int CS = 8;                 // channels per group handled by this kernel
constexpr int TMEM_COLS = 256;
constexpr int COL_LBO = 144;          // padded K-chunk pitch of the column operand (bank-conflict-free 2-byte stores)

struct BwdPlan {
    int TPR;             // taps per thread row
    int Kc;              // CS * KK  (real K' columns)
    int N1;              // GEMM1 N: Kc rounded up to 16
    int N3;              // GEMM3 N: Kc + 1 (ones column -> grad_bias) rounded up to 8
    int kch1;            // Co / 8: K chunks of the Co-contraction operands
    int tiles_x, tiles_y;
    int wt_part, p_part, q_part, col_part, col_sbo;    // bytes of one (hi or lo) image
    int om_off, om_bytes;                              // offset/mask tile staged by TMA (0 bytes: read from global)
    int smem;
};

__device__ __forceinline__ void st_bf16(unsigned char *base, int off, unsigned short v)
{
    *reinterpret_cast<unsigned short *>(base + off) = v;
}

// 16-byte vector reduction into global memory (sm_90+): 4 fp32 adds, one L2 transaction
__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float e)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(e) : "memory");
}

// eight bf16 values -> one 16-byte K chunk
__device__ __forceinline__ void st_bf16x8(unsigned char *base, int off, const unsigned short (&v)[8])
{
    const uint32_t a = v[0] | ((uint32_t)v[1] << 16), b = v[2] | ((uint32_t)v[3] << 16);
    const uint32_t c = v[4] | ((uint32_t)v[5] << 16), e = v[6] | ((uint32_t)v[7] << 16);
    *reinterpret_cast<uint4 *>(base + off) = make_uint4(a, b, c, e);
}

template <bool PACKED, bool DET>
__global__ void __launch_bounds__(NTHR, 2)
dcn_bwd_tc_kernel(const float *__restrict__ in_blk, const float *__restrict__ weight,
                  const float *__restrict__ offset, const float *__restrict__ mask,
                  const float *__restrict__ gout, float *__restrict__ gin_blk,
                  float *__restrict__ goff, float *__restrict__ gmask,
                  float *__restrict__ gw_part, float *__restrict__ gb_part, DcnDims d, BwdPlan pl,
                  const __grid_constant__ CUtensorMap tm_off, const __grid_constant__ CUtensorMap tm_mask)
{
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *wt_hi = smem, *wt_lo = smem + pl.wt_part;                       // B of GEMM1: [N1 rows k'][Co]
    unsigned char *q_hi = smem + 2 * pl.wt_part, *q_lo = q_hi + pl.q_part;         // A of GEMM3: [Co rows][128 px]
    unsigned char *u_base = q_lo + pl.q_part;                                      // union: P (A of GEMM1) | col (B of GEMM3)
    unsigned char *p_hi = u_base, *p_lo = u_base + pl.p_part;                      //   P: [128 px rows][Co]
    unsigned char *c_hi = u_base, *c_lo = u_base + pl.col_part;                    //   col: [N3 rows k'][128 px], LBO 144
    // offsets (2*KK planes) and mask (KK planes) of the tile, [plane][8 x 16 pixels] fp32: one TMA tensor copy each,
    // issued at the top of the tile loop -> their DRAM latency (every element is read exactly once) hides behind the
    // grad_output staging and GEMM1, without holding registers
    const float *s_om = reinterpret_cast<const float *>(smem + pl.om_off);
    const bool use_tma = pl.om_bytes > 0;
    __shared__ __align__(8) uint64_t bar1, bar3, bar_om;
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int p = tid % TM, r = tid / TM;
    const int S = gridDim.x, s = blockIdx.x, g = blockIdx.y;
    const int c0 = g * d.cpg;
    const int npix = d.Ho * d.Wo, Kdim = d.C * d.KK;
    const size_t plane = (size_t)npix, in_plane = (size_t)d.H * d.W;
    const int ntile = pl.tiles_x * pl.tiles_y;

    if (warp == 0) umma::tmem_alloc<TMEM_COLS>(&tmem_slot);
    if (tid == 0) { umma::mbar_init(&bar1, 1); umma::mbar_init(&bar3, 1); umma::mbar_init(&bar_om, 1); umma::mbar_fence_init(); }
    // ---- W_g^T, resident for the whole CTA: wt[k'][co] = weight[co][(c0 + cc) * KK + tap], k' = tap * 8 + cc
    for (int e = tid; e < pl.N1 * d.Co; e += NTHR) {
        const int j = e & 7, rr = (e >> 3) & 7, rest = e >> 6;
        const int kc = rest % pl.kch1, rg = rest / pl.kch1;
        const int kp = rg * 8 + rr, co = kc * 8 + j;
        unsigned short hi = 0, lo = 0;
        if (kp < pl.Kc) {
            const int t = kp >> 3, cc = kp & 7;
            umma::split_bf16(__ldg(weight + (size_t)co * Kdim + (size_t)(c0 + cc) * d.KK + t), hi, lo);
        }
        st_bf16(wt_hi, e * 2, hi); st_bf16(wt_lo, e * 2, lo);
    }
    umma::fence_smem_to_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t d1 = tmem, d3h = tmem + pl.N1, d3x = tmem + pl.N1 + pl.N3;
    const uint32_t idesc1 = umma::instr_desc_bf16(TM, pl.N1), idesc3 = umma::instr_desc_bf16(d.Co, pl.N3);
    const uint32_t lane_base = (uint32_t)(warp & 3) * 32u;

    const unsigned uplane = (unsigned)plane;
    const float det_scale = DET ? ldexpf(1.f, det_scale_exp(d)) : 0.f;

    uint32_t ph1 = 0, ph3 = 0, ph_om = 0;
    int ntiles_done = 0;
    for (int tile = s; tile < d.B * ntile; tile += S, ++ntiles_done) {
        const int b = tile / ntile, tl = tile % ntile;
        const int ty0 = (tl / pl.tiles_x) * TH, tx0 = (tl % pl.tiles_x) * TW;
        const int ho = ty0 + p / TW, wo = tx0 + p % TW;
        const bool valid = ho < d.Ho && wo < d.Wo;
        const int pix = ho * d.Wo + wo;
        const float *go_b = gout + (size_t)b * d.Co * plane;
        if (use_tma && tid == 0) {                   // every reader of the previous tile's copy has passed the barrier before GEMM3
            umma::mbar_expect_tx(&bar_om, (uint32_t)pl.om_bytes);
            tma::load_3d(smem + pl.om_off, &tm_off, tx0, ty0, b * d.off_bp + g * 2 * d.KK, &bar_om);
            tma::load_3d(smem + pl.om_off + 2 * d.KK * TM * 4, &tm_mask, tx0, ty0, b * d.mask_bp + g * d.KK, &bar_om);
        }
        if (ntiles_done > 0) {                       // GEMM3 of the previous tile has read Q and col
            umma::mbar_wait(&bar3, ph3);
            ph3 ^= 1;
        }
        // ---- grad_output tile in both K-major layouts (bf16 hi/lo)
        // P[px][co]: item = (pixel, chunk of 8 co); lanes run over pixels -> coalesced plane reads
        for (int it = tid; it < TM * pl.kch1; it += NTHR) {
            const int pp = it % TM, kc = it / TM;
            const int hh = ty0 + pp / TW, ww = tx0 + pp % TW;
            unsigned short hi[8], lo[8];
            const bool ok = hh < d.Ho && ww < d.Wo;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float v = ok ? __ldg(go_b + (size_t)(kc * 8 + j) * plane + (size_t)hh * d.Wo + ww) : 0.f;
                umma::split_bf16(v, hi[j], lo[j]);
            }
            const int off = (pp >> 3) * (pl.kch1 * 128) + kc * 128 + (pp & 7) * 16;
            st_bf16x8(p_hi, off, hi); st_bf16x8(p_lo, off, lo);
        }
        // Q[co][px]: item = (co, chunk of 8 consecutive tile pixels = half a tile row)
        for (int it = tid; it < d.Co * (TM / 8); it += NTHR) {
            const int pc = it % (TM / 8), co = it / (TM / 8);
            const int hh = ty0 + (pc * 8) / TW, ww = tx0 + (pc * 8) % TW;
            unsigned short hi[8], lo[8];
            float v[8];
            const float *src = go_b + (size_t)co * plane + (size_t)hh * d.Wo + ww;
            if ((d.Wo & 3) == 0 && hh < d.Ho && ww + 7 < d.Wo) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(src)), c = __ldg(reinterpret_cast<const float4 *>(src) + 1);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = (hh < d.Ho && ww + j < d.Wo) ? __ldg(src + j) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) umma::split_bf16(v[j], hi[j], lo[j]);
            const int off = (co >> 3) * ((TM / 8) * 128) + pc * 128 + (co & 7) * 16;
            st_bf16x8(q_hi, off, hi); st_bf16x8(q_lo, off, lo);
        }
        umma::fence_smem_to_async();
        __syncthreads();
        // ---- GEMM1: D1[px][k'] = P . Wt^T   (K = Co)
        if (tid == 0) {
            umma::fence_after_sync();
            for (int ks = 0; ks < d.Co / 16; ++ks) {
                const uint32_t ko = ks * 256u, sb = pl.kch1 * 128u;
                const uint64_t ah = umma::smem_desc(umma::smem_u32(p_hi) + ko, 128, sb), al = umma::smem_desc(umma::smem_u32(p_lo) + ko, 128, sb);
                const uint64_t bh = umma::smem_desc(umma::smem_u32(wt_hi) + ko, 128, sb), bl = umma::smem_desc(umma::smem_u32(wt_lo) + ko, 128, sb);
                umma::mma_f16(d1, al, bh, idesc1, ks > 0);
                umma::mma_f16(d1, ah, bl, idesc1, true);
                umma::mma_f16(d1, ah, bh, idesc1, true);
            }
            umma::commit(&bar1);
        }
        // ---- sampling positions of this thread's taps (overlaps GEMM1)
        // element offsets of this (sample, group) inside offset / mask AND inside their gradients (same layout)
        const size_t off_e = (size_t)b * d.off_bs + (size_t)g * 2 * d.KK * plane;
        const size_t mask_e = (size_t)b * d.mask_bs + (size_t)g * d.KK * plane;
        umma::mbar_wait(&bar1, ph1);                 // D1 complete; P is dead, its storage becomes `col`
        ph1 ^= 1;
        umma::fence_after_sync();
        if (use_tma) {
            umma::mbar_wait(&bar_om, ph_om);
            ph_om ^= 1;
        }
        for (int sidx = 0; sidx < pl.TPR; ++sidx) {
            const int t = r * pl.TPR + sidx;
            if (t >= d.KK) break;
            const int ti = t / d.kw, tj = t - ti * d.kw;
            float gc[8];
            umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, t * 8), gc);     // colgrad[p][t*8 .. t*8+7]
            umma::tmem_ld_wait();
            float colv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) colv[j] = 0.f;
            if (valid) {
                float dy, dx, m;
                if (use_tma) {
                    dy = s_om[(2 * t) * TM + p];
                    dx = s_om[(2 * t + 1) * TM + p];
                    m = s_om[(2 * d.KK + t) * TM + p];
                } else {
                    tap_read(offset + off_e, mask + mask_e, uplane, (unsigned)t, (unsigned)pix, dy, dx, m);
                }
                m = mask_act_t<PACKED>(m);
                const float y = (float)(ho * d.sh - d.ph + ti * d.dh) + dy;
                const float x = (float)(wo * d.sw - d.pw + tj * d.dw) + dx;
                const float xq = (float)(wo * d.sw - d.ph + tj * d.dw) + dx;   // the scatter's x uses pad_h (im2col_cuda.cu:368)
                const Tap tp = make_tap(y, x, d.H, d.W);
                const Tap tq = (d.ph == d.pw) ? tp : make_tap(y, xq, d.H, d.W);
                const float w1 = tp.hy * tp.hx, w2 = tp.hy * tp.lx, w3 = tp.ly * tp.hx, w4 = tp.ly * tp.lx;
                const float q1 = tq.hy * tq.hx, q2 = tq.hy * tq.lx, q3 = tq.ly * tq.hx, q4 = tq.ly * tq.lx;
                float s_m = 0.f, s_y = 0.f, s_x = 0.f;
                // group-blocked layout [b][g][y][x][8 ch]: the 8 channels of a corner are 32 contiguous bytes
                const float *ib = in_blk + ((size_t)b * d.dg + g) * in_plane * CS;
                float *gb = gin_blk + ((size_t)b * d.dg + g) * in_plane * CS;
                const f8 a1 = ldg_f8(ib + (size_t)tp.i00 * CS, tp.c00), a2 = ldg_f8(ib + (size_t)tp.i01 * CS, tp.c01);
                const f8 a3 = ldg_f8(ib + (size_t)tp.i10 * CS, tp.c10), a4 = ldg_f8(ib + (size_t)tp.i11 * CS, tp.c11);
                float top[CS];
#pragma unroll
                for (int cc = 0; cc < CS; ++cc) {
                    const float v1 = a1.v[cc], v2 = a2.v[cc], v3 = a3.v[cc], v4 = a4.v[cc];
                    const float val = w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4;
                    s_m += gc[cc] * val;                                            // grad_mask (im2col_cuda.cu:311)
                    const float wy = -tp.hx * v1 - tp.lx * v2 + tp.hx * v3 + tp.lx * v4;   // coordinate weights (:99-120)
                    const float wx = -tp.hy * v1 + tp.hy * v2 - tp.ly * v3 + tp.ly * v4;
                    top[cc] = gc[cc] * m;
                    s_y += wy * top[cc];
                    s_x += wx * top[cc];
                    colv[cc] = val * m;
                }
                // grad_input scatter (:236-251): 16-byte vector reductions, two per corner; deterministic mode:
                // scalar 64-bit integer reductions into the fixed-point copy
                if (DET) {
                    long long *g64 = reinterpret_cast<long long *>(gin_blk) + ((size_t)b * d.dg + g) * in_plane * CS;
#pragma unroll
                    for (int cc = 0; cc < CS; ++cc) {
                        if (tq.c00) det_add(g64 + (size_t)tq.i00 * CS + cc, q1 * top[cc], det_scale);
                        if (tq.c01) det_add(g64 + (size_t)tq.i01 * CS + cc, q2 * top[cc], det_scale);
                        if (tq.c10) det_add(g64 + (size_t)tq.i10 * CS + cc, q3 * top[cc], det_scale);
                        if (tq.c11) det_add(g64 + (size_t)tq.i11 * CS + cc, q4 * top[cc], det_scale);
                    }
                }
#pragma unroll
                for (int h = 0; h < (DET ? 0 : 2); ++h) {
                    const float *tt = top + 4 * h;
                    if (tq.c00) red_add_v4(gb + (size_t)tq.i00 * CS + 4 * h, q1 * tt[0], q1 * tt[1], q1 * tt[2], q1 * tt[3]);
                    if (tq.c01) red_add_v4(gb + (size_t)tq.i01 * CS + 4 * h, q2 * tt[0], q2 * tt[1], q2 * tt[2], q2 * tt[3]);
                    if (tq.c10) red_add_v4(gb + (size_t)tq.i10 * CS + 4 * h, q3 * tt[0], q3 * tt[1], q3 * tt[2], q3 * tt[3]);
                    if (tq.c11) red_add_v4(gb + (size_t)tq.i11 * CS + 4 * h, q4 * tt[0], q4 * tt[1], q4 * tt[2], q4 * tt[3]);
                }
                float *gy = goff + off_e + (2u * t * uplane + (unsigned)pix);
                gy[0] = s_y; gy[uplane] = s_x;
                gmask[mask_e + ((unsigned)t * uplane + (unsigned)pix)] = s_m * mask_act_grad_t<PACKED>(m);
            }
            // column operand: col[k' = t*8+cc][px = p]; rows t*8..t*8+7 are one 8-row group
            const int off = t * pl.col_sbo + (p >> 3) * COL_LBO + (p & 7) * 2;
#pragma unroll
            for (int cc = 0; cc < CS; ++cc) {
                unsigned short hi, lo;
                umma::split_bf16(colv[cc], hi, lo);
                st_bf16(c_hi, off + cc * 16, hi); st_bf16(c_lo, off + cc * 16, lo);
            }
        }
        // last 8-row group: the ones column (grad_bias) and zero padding; rewritten every tile because
        // the grad_output copy P overlays it
        for (int it = tid; it < 8 * TM; it += NTHR) {
            const int pp = it % TM, rr = it / TM;
            const int hh = ty0 + pp / TW, ww = tx0 + pp % TW;
            const int row = pl.Kc + rr;
            if (row < pl.N3) {
                const unsigned short one = (rr == 0 && hh < d.Ho && ww < d.Wo) ? 0x3F80 : 0;   // bf16(1.0)
                const int off = (row >> 3) * pl.col_sbo + (pp >> 3) * COL_LBO + (row & 7) * 16 + (pp & 7) * 2;
                st_bf16(c_hi, off, one); st_bf16(c_lo, off, 0);
            }
        }
        umma::fence_smem_to_async();
        umma::fence_before_sync();                   // orders this thread's tcgen05.ld of D1 before the sync
        __syncthreads();
        // ---- GEMM3: D3[co][k'] += Q . col^T   (K = 128 tile pixels), accumulated across tiles
        if (tid == 0) {
            umma::fence_after_sync();
            for (int ks = 0; ks < TM / 16; ++ks) {
                const uint32_t qo = ks * 256u, co_ = ks * 2u * COL_LBO, qsb = (TM / 8) * 128u;
                const uint64_t ah = umma::smem_desc(umma::smem_u32(q_hi) + qo, 128, qsb), al = umma::smem_desc(umma::smem_u32(q_lo) + qo, 128, qsb);
                const uint64_t bh = umma::smem_desc(umma::smem_u32(c_hi) + co_, COL_LBO, pl.col_sbo);
                const uint64_t bl = umma::smem_desc(umma::smem_u32(c_lo) + co_, COL_LBO, pl.col_sbo);
                const bool acc = ntiles_done > 0 || ks > 0;
                umma::mma_f16(d3x, al, bh, idesc3, acc);
                umma::mma_f16(d3x, ah, bl, idesc3, true);
                umma::mma_f16(d3h, ah, bh, idesc3, acc);
            }
            umma::commit(&bar3);
        }
    }
    // ---- partials of this CTA: gw_part[s][co][(c0+cc)*KK + t], gb_part[s][co]
    if (ntiles_done > 0) {
        umma::mbar_wait(&bar3, ph3);
        umma::fence_after_sync();
    }
    // D3 is an M = Co accumulator: Co = 64 -> row co = 16*q + l lives in lane 32*q + l (l < 16);
    // Co = 128 -> row = lane. Thread rows r split the 8-column blocks.
    const int q4 = warp & 3;
    const int co = (d.Co == 128) ? (q4 * 32 + lane) : (lane < 16 ? q4 * 16 + lane : -1);
    for (int cb = r * 8; cb < pl.N3; cb += NR * 8) {
        float v[8], u[8];
        if (ntiles_done > 0) {
            umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, pl.N1 + cb), v);
            umma::tmem_ld8(umma::tmem_addr(tmem, lane_base, pl.N1 + pl.N3 + cb), u);
            umma::tmem_ld_wait();
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = u[i] = 0.f;
        }
        if (co >= 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int kp = cb + i;
                const float val = v[i] + u[i];
                if (kp < pl.Kc)
                    gw_part[((size_t)s * d.Co + co) * Kdim + (size_t)(c0 + (kp & 7)) * d.KK + (kp >> 3)] = val;
                else if (kp == pl.Kc && g == 0)
                    gb_part[(size_t)s * d.Co + co] = val;
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tmem);
}

// NCHW (B, dg*8, H, W)  <->  group-blocked (B, dg, H, W, 8): one thread per (b, g, y, x); reads and
// writes are both coalesced (8 plane reads of consecutive x, 32 contiguous bytes per thread).
// `zero` (nullable): a second (BG, HW, 8)-shaped buffer of `zero_f4` float4 per item that is cleared in the same pass
// (the backward's grad_input accumulator: 2 float4 per item, 4 for the int64 copy of the deterministic mode) — saves the
// separate memset launch.
template <typename T>
__global__ void nchw_to_blocked(const T *__restrict__ src, float *__restrict__ dst, int BG, int HW,
                                float4 *__restrict__ zero, int zero_f4)
{
    const size_t n = (size_t)BG * HW;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t bg = i / HW, px = i - bg * HW;
        const T *sp = src + bg * CS * HW + px;
        float v[CS];
#pragma unroll
        for (int c = 0; c < CS; ++c) v[c] = ld_act(sp + (size_t)c * HW);
        float4 *dp = reinterpret_cast<float4 *>(dst + i * CS);
        dp[0] = make_float4(v[0], v[1], v[2], v[3]);
        dp[1] = make_float4(v[4], v[5], v[6], v[7]);
        if (zero)
            for (int q = 0; q < zero_f4; ++q) zero[i * zero_f4 + q] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

__global__ void blocked_to_nchw(const float *__restrict__ src, float *__restrict__ dst, int BG, int HW)
{
    const size_t n = (size_t)BG * HW;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t bg = i / HW, px = i - bg * HW;
        const float4 *sp = reinterpret_cast<const float4 *>(src + i * CS);
        const float4 a = sp[0], c = sp[1];
        float *dp = dst + bg * CS * HW + px;
        dp[0] = a.x; dp[(size_t)HW] = a.y; dp[(size_t)2 * HW] = a.z; dp[(size_t)3 * HW] = a.w;
        dp[(size_t)4 * HW] = c.x; dp[(size_t)5 * HW] = c.y; dp[(size_t)6 * HW] = c.z; dp[(size_t)7 * HW] = c.w;
    }
}

// fixed-point (BG, HW, 8) int64 -> fp32 NCHW: one rounding per element
__global__ void blocked_i64_to_nchw(const long long *__restrict__ src, float *__restrict__ dst, int BG, int HW, DcnDims d)
{
    const float inv = det_bound_nonfinite(d) ? __uint_as_float(0x7FC00000u) : ldexpf(1.f, -det_scale_exp(d));   // NaN propagates
    const size_t n = (size_t)BG * HW;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t bg = i / HW, px = i - bg * HW;
        const longlong2 *sp = reinterpret_cast<const longlong2 *>(src + i * CS);
        float *dp = dst + bg * CS * HW + px;
#pragma unroll
        for (int c = 0; c < CS / 2; ++c) {
            const longlong2 v = sp[c];
            dp[(size_t)(2 * c) * HW] = __ll2float_rn(v.x) * inv;
            dp[(size_t)(2 * c + 1) * HW] = __ll2float_rn(v.y) * inv;
        }
    }
}

bool make_plan(const DcnDims &d, BwdPlan &pl)
{
    if (d.cpg != CS || d.Co != 64) return false;          // other shapes: CUDA-core kernel in dcn.cu
    if ((long)2 * d.KK * d.Ho * d.Wo >= (1L << 31)) return false;   // 32-bit offsets inside one group
    pl.TPR = ceil_div(d.KK, NR);
    pl.Kc = CS * d.KK;
    pl.N1 = ebfi::round_up(pl.Kc, 16);
    pl.N3 = ebfi::round_up(pl.Kc + 1, 8);
    if (pl.N1 + 2 * pl.N3 > TMEM_COLS) return false;      // 3x3: 80 + 2*80
    pl.kch1 = d.Co / 8;
    pl.tiles_x = ceil_div(d.Wo, TW);
    pl.tiles_y = ceil_div(d.Ho, TH);
    pl.wt_part = pl.N1 * d.Co * 2;
    pl.p_part = TM * d.Co * 2;
    pl.q_part = d.Co * TM * 2;
    pl.col_sbo = (TM / 8) * COL_LBO;
    pl.col_part = (pl.N3 / 8) * pl.col_sbo;
    pl.om_off = 2 * pl.wt_part + 2 * pl.q_part + 2 * std::max(pl.p_part, pl.col_part);
    // TMA staging of the offset/mask tile needs 16-byte row strides; two CTAs (+1 KB each) must fit one SM's 228 KB
    const bool tma_ok = d.Wo % 4 == 0 && getenv("EBFI_DCN_NO_TMA") == nullptr;
    pl.om_bytes = tma_ok ? 3 * d.KK * TM * 4 : 0;
    if (pl.om_off + pl.om_bytes > 113 * 1024) pl.om_bytes = 0;
    pl.smem = pl.om_off + pl.om_bytes;
    return pl.smem <= 113 * 1024;
}

}  // namespace

int backward_tc_splits(const DcnDims &d)
{
    BwdPlan pl{};
    if (!make_plan(d, pl)) return 0;
    const int tiles = d.B * pl.tiles_x * pl.tiles_y;
    return std::max(1, std::min(tiles, ceil_div(2 * ebfi::sm_count(), d.dg)));
}

template <typename T>
int launch_nchw_to_blocked(cudaStream_t st, const T *src, float *dst, int BG, int HW, void *zero, int zero_f4)
{
    const unsigned tgrid = (unsigned)std::min<size_t>(ceil_div((size_t)BG * HW, (size_t)256), (size_t)ebfi::sm_count() * 16);
    nchw_to_blocked<T><<<tgrid, 256, 0, st>>>(src, dst, BG, HW, static_cast<float4 *>(zero), zero_f4);
    EBFI_LAUNCH_OK("nchw_to_blocked");
    return EBFI_OK;
}
template int launch_nchw_to_blocked<float>(cudaStream_t, const float *, float *, int, int, void *, int);
template int launch_nchw_to_blocked<__nv_bfloat16>(cudaStream_t, const __nv_bfloat16 *, float *, int, int, void *, int);
template int launch_nchw_to_blocked<__half>(cudaStream_t, const __half *, float *, int, int, void *, int);

// Extra scratch of the tensor-core backward: group-blocked copies of input and grad_input.
size_t backward_tc_scratch_bytes(const DcnDims &d)
{
    BwdPlan pl{};
    if (!make_plan(d, pl)) return 0;
    return (d.det ? 3 : 2) * (size_t)d.B * d.C * d.H * d.W * sizeof(float);     // int64 grad_input copy when deterministic
}

// Tensor-core backward: writes grad_input / grad_offset / grad_mask in full and the partials
// gw_part[S][Co][C*KK], gb_part[S][Co] with S = backward_tc_splits(d). `scratch` holds
// backward_tc_scratch_bytes(d) bytes, 16-byte aligned.
int backward_tc(cudaStream_t st, const DcnDims &d, const float *input, const float *weight, const float *offset,
                const float *mask, const float *gout, float *gin, float *goff, float *gmask, float *gw_part,
                float *gb_part, int S, void *scratch)
{
    BwdPlan pl{};
    if (!make_plan(d, pl)) return EBFI_ERR_UNSUPPORTED;
    const size_t n = (size_t)d.B * d.C * d.H * d.W;
    float *in_blk = static_cast<float *>(scratch), *gin_blk = in_blk + n;
    const int BG = d.B * d.dg, HW = d.H * d.W;
    const unsigned tgrid = (unsigned)std::min<size_t>(ceil_div((size_t)BG * HW, (size_t)256), (size_t)ebfi::sm_count() * 16);
    // blocked copy of the input + zero fill of the grad_input accumulator (fp32, or int64 in deterministic mode) in one pass
    if (int rc = launch_nchw_to_blocked(st, input, in_blk, BG, HW, gin_blk, d.det ? 4 : 2)) return rc;
    dim3 grid(S, d.dg);
    CUtensorMap tm_off{}, tm_mask{};
    if (pl.om_bytes > 0 && !(ebfi::aligned16(offset) && ebfi::aligned16(mask))) {   // TMA needs 16-byte aligned bases
        pl.om_bytes = 0;
        pl.smem = pl.om_off;
    }
    if (pl.om_bytes > 0) {
        const uint64_t str[2] = {(uint64_t)d.Wo * 4, (uint64_t)d.Ho * d.Wo * 4};
        const uint64_t dims_o[3] = {(uint64_t)d.Wo, (uint64_t)d.Ho, (uint64_t)(d.B - 1) * d.off_bp + 2 * d.dg * d.KK};
        const uint64_t dims_m[3] = {(uint64_t)d.Wo, (uint64_t)d.Ho, (uint64_t)(d.B - 1) * d.mask_bp + d.dg * d.KK};
        const uint32_t box_o[3] = {TW, TH, (uint32_t)(2 * d.KK)}, box_m[3] = {TW, TH, (uint32_t)d.KK};
        if (int rc = tma::encode_3d(tm_off, offset, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dims_o, str, box_o)) return rc;
        if (int rc = tma::encode_3d(tm_mask, mask, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dims_m, str, box_m)) return rc;
    }
#define EBFI_BWD_TC(P, D)                                                                                     \
    do {                                                                                                      \
        EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_bwd_tc_kernel<P, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem)); \
        dcn_bwd_tc_kernel<P, D><<<grid, NTHR, pl.smem, st>>>(in_blk, weight, offset, mask, gout, gin_blk, goff, gmask, \
                                                             gw_part, gb_part, d, pl, tm_off, tm_mask);       \
    } while (0)
    if (d.det) { if (d.packed) EBFI_BWD_TC(true, true); else EBFI_BWD_TC(false, true); }
    else       { if (d.packed) EBFI_BWD_TC(true, false); else EBFI_BWD_TC(false, false); }
#undef EBFI_BWD_TC
    EBFI_LAUNCH_OK("dcn_bwd_tc_kernel");
    if (d.det) {
        blocked_i64_to_nchw<<<tgrid, 256, 0, st>>>(reinterpret_cast<const long long *>(gin_blk), gin, BG, HW, d);
        EBFI_LAUNCH_OK("blocked_i64_to_nchw");
        return EBFI_OK;
    }
    blocked_to_nchw<<<tgrid, 256, 0, st>>>(gin_blk, gin, BG, HW);
    EBFI_LAUNCH_OK("blocked_to_nchw");
    return EBFI_OK;
}

}  // namespace ebfi_dcn
