// dcn_fwd_box.cu — DCNv2 forward: bilinear sampling from a TMA-staged input box fused into a tcgen05 GEMM.
//
// Persistent kernel, one CTA per SM, 19 warps with fixed roles; a CTA walks 8 x 16-pixel output tiles
// (128 pixels = the M of a 128 x Cout UMMA, one TMEM lane per pixel):
//   box loader (1 warp)  : per (tile, 8-channel chunk) ONE 3-D TMA copy of a 24 x 30-pixel box of the group-blocked
//                          input [b][chunk][y][x][8 ch] (out-of-image rows/pixels arrive as zeros = the reference's
//                          per-corner bounds tests, im2col_cuda.cu:38-48), and per (tile, group) two TMA copies of the
//                          tile's offset / mask planes. Double buffered.
//   weight loader (1 warp): the pre-split weight image of each stage by one bulk copy into a 3-slot ring.
//   samplers (12 warps)  : thread (pixel p, row r) handles tap r*TPR + s in stage s. The four corners of a sample are
//                          2 x 2 x 32 B = 128 B of the box. The box pitch is 30 px * 32 B = 64 (mod 128), so those
//                          eight 16-byte chunks tile all 32 banks exactly once; lane L reads its chunks in the ROTATED
//                          order c = (L - b + i) mod 8 (b = bank group of the sample's first chunk), which puts the
//                          eight lanes of every quarter-warp on eight different bank groups whatever the offsets are:
//                          conflict-free LDS.128, 1.18 clk per sample measured (tools/microbench/scatter_probe.cu)
//                          against 3.5 clk in natural order and ~4 L1 wavefronts per sample for the global gathers
//                          this replaces. Samples whose corners leave the box (|offset| > ~6 px) take predicated
//                          256-bit global loads. Values are mask-modulated, split into TF32 hi + lo and stored as the
//                          K-major A operand of the stage.
//   MMA issuer (1 warp)  : 3xTF32 tcgen05.mma chain per stage into the tile's TMEM accumulators (double buffered
//                          across tiles), commit -> slot free / accumulator full.
//   epilogue (4 warps)   : tcgen05.ld (lane = pixel), sum of the split accumulators, + bias, NCHW stores — while the
//                          samplers are already on the next tile.
// The reference's 151 MB column buffer (dcn_v2_cuda.cu:68) never exists; input traffic from L2 is one box per
// (tile, chunk) instead of four scattered sectors per sample.
//
// fp32 parity: products are 3xTF32 (umma.cuh); the hi*hi chain is spread over several TMEM accumulators because
// the tensor core's fp32 accumulate rounds toward zero.
// Activation type T (float | __nv_bfloat16 | __half, the *_bf16 / *_fp16 entries): the input is widened into the same
// fp32 blocked copy, offsets / masks arrive by TMA as T planes and are widened where the samplers read them, the
// epilogue rounds once.
#include "dcn_box.cuh"
#include "dcn_common.cuh"
#include "tma.cuh"
#include "umma.cuh"

#include <algorithm>

namespace ebfi_dcn {

namespace {

using ebfi::ceil_div;

constexpr int TM = 128, TH = 8, TW = 16, NR = 3;
constexpr int KSTEPS = NR;                      // a stage's K = NR taps x 8 channels = NR tf32 MMA steps
constexpr int BH = 24, BW = 30;                 // staged box: rows x pixels (8 channels each)
constexpr int BOX_PITCH = BW * 32;              // bytes; 960 = 64 (mod 128)
constexpr int BOX_BYTES = BH * BOX_PITCH;       // 23,040 (a multiple of 128)
constexpr int NS = 3;                           // operand ring slots (A image + weight image)
constexpr int N_EPI = 4, N_SAMP = 12;           // warps
constexpr int W_MMA = N_EPI + N_SAMP, W_BOX = W_MMA + 1, W_WGT = W_MMA + 2, NWARP = W_MMA + 3;
constexpr int NTHR = NWARP * 32;
constexpr int TMEM_COLS = 512, ACC_COLS = 256;  // two tile accumulator sets

struct BoxPlan {
    int ncs;             // 8-channel chunks per deformable group
    int TPR;             // taps per thread row = stages per chunk: tap = r * TPR + s
    int Ks, Ksp, kch;    // K of a stage (NR * 8), padded to 8, 16-byte chunks per operand row
    int nacc;            // hi*hi accumulators (+1 for the cross terms)
    int tiles_x, tiles_y, ntiles;
    int a_bytes, b_bytes;
    int om_bytes, use_om_tma;
    int my, mx;          // rows / pixels of the box above / left of the tile's undeformed footprint
    int unit_bytes;      // weight images of one (group, chunk) unit: TPR stages x (hi | lo)
    int off_w, off_box, off_om, smem;
};

__device__ __forceinline__ float4 lds128(uint32_t saddr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}

// One modulated bilinear sample of 8 channels. In-box: rotated conflict-free LDS.128 gather (see the file header);
// the two 16-byte halves (channels 0-3 / 4-7) come back in `ha` / `hb`, SWAPPED when the function returns true (the
// caller swaps the store addresses instead of eight values). `ibf` = the chunk's blocked global plane for the fallback.
__device__ __forceinline__ bool sample8(float y, float x, float m, int H, int W, uint32_t box_s, int by0, int bx0,
                                        const float *__restrict__ ibf, int lane, float (&ha)[4], float (&hb)[4])
{
#pragma unroll
    for (int j = 0; j < 4; ++j) ha[j] = hb[j] = 0.f;
    // the sampling window of the reference (im2col_cuda.cu:180); NaN coordinates fail it like they do there
    if (!(y > -1.f && x > -1.f && y < (float)H && x < (float)W)) return false;
    const float fy = floorf(y), fx = floorf(x);
    const int y0 = (int)fy, x0 = (int)fx;
    const float ly = y - fy, lx = x - fx, hy = 1.f - ly, hx = 1.f - lx;
    const float my = m * hy, mly = m * ly;
    const int yb = y0 - by0, xb = x0 - bx0;
    if ((unsigned)yb <= (unsigned)(BH - 2) && (unsigned)xb <= (unsigned)(BW - 2)) {
        const uint32_t base = box_s + (uint32_t)(yb * BW + xb) * 32u;
        const uint32_t c0 = ((uint32_t)lane - (base >> 4)) & 7u;   // first chunk: bank group of (base + 16*c0) = lane (mod 8)
        const bool odd = c0 & 1u;
        // corner weights (mask folded in) rotated so that w[j] belongs to corner (c0/2 + j) mod 4;
        // corners: 0 (y0,x0)  1 (y0,x0+1)  2 (y0+1,x0)  3 (y0+1,x0+1)
        float w0 = my * hx, w1 = my * lx, w2 = mly * hx, w3 = mly * lx;
        if (c0 & 2u) { const float t = w0; w0 = w1; w1 = w2; w2 = w3; w3 = t; }
        if (c0 & 4u) { float t = w0; w0 = w2; w2 = t; t = w1; w1 = w3; w3 = t; }
        const float wr[5] = {w0, w1, w2, w3, w0};
        // byte table of chunk offsets / 16 = {0,1,2,3, 60,61,62,63} (second row = +BOX_PITCH), rotated by c0 bytes
        constexpr uint32_t T_LO = 0x03020100u, T_HI = 0x03020100u + 0x01010101u * (BOX_PITCH / 16);
        const uint32_t ta = (c0 & 4u) ? T_HI : T_LO, tb = (c0 & 4u) ? T_LO : T_HI, sh = (c0 & 3u) * 8u;
        const uint32_t r_lo = __funnelshift_r(ta, tb, sh), r_hi = __funnelshift_r(tb, ta, sh);
        // packed fp32x2 FMAs (FFMA2): half the FMA issue slots; the scalar weight is the instruction's broadcast operand
        box::f32x2 acc[2][2] = {};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t o16 = __byte_perm(i < 4 ? r_lo : r_hi, 0u, 0x4440u | (uint32_t)(i & 3));
            const float4 q = lds128(base + (o16 << 4));
            const float wi = odd ? wr[(i + 1) >> 1] : wr[i >> 1];
            box::f32x2 (&a)[2] = acc[i & 1];                   // even / odd steps = the two 16-byte halves
            a[0] = box::ffma2(box::pack2(wi, wi), box::pack2(q.x, q.y), a[0]);
            a[1] = box::ffma2(box::pack2(wi, wi), box::pack2(q.z, q.w), a[1]);
        }
        box::unpack2(acc[0][0], ha[0], ha[1]); box::unpack2(acc[0][1], ha[2], ha[3]);
        box::unpack2(acc[1][0], hb[0], hb[1]); box::unpack2(acc[1][1], hb[2], hb[3]);
        return odd;
    }
    const Tap tp = make_tap(y, x, H, W);
    const float w1 = tp.hy * tp.hx * m, w2 = tp.hy * tp.lx * m, w3 = tp.ly * tp.hx * m, w4 = tp.ly * tp.lx * m;
    const f8 a = ldg_f8(ibf + (size_t)tp.i00 * 8, tp.c00), bq = ldg_f8(ibf + (size_t)tp.i01 * 8, tp.c01);
    const f8 c = ldg_f8(ibf + (size_t)tp.i10 * 8, tp.c10), e8 = ldg_f8(ibf + (size_t)tp.i11 * 8, tp.c11);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        ha[j] = w1 * a.v[j] + w2 * bq.v[j] + w3 * c.v[j] + w4 * e8.v[j];
        hb[j] = w1 * a.v[4 + j] + w2 * bq.v[4 + j] + w3 * c.v[4 + j] + w4 * e8.v[4 + j];
    }
    return false;
}

template <int TPR, bool PACKED, typename T>
__global__ void __launch_bounds__(NTHR, 1)
dcn_fwd_box_kernel(const float *__restrict__ in_blk, const float *__restrict__ bias,
                   const T *__restrict__ offset, const T *__restrict__ mask,
                   T *__restrict__ output, const float *__restrict__ wimg, DcnDims d, BoxPlan pl,
                   const __grid_constant__ CUtensorMap tm_box, const __grid_constant__ CUtensorMap tm_off,
                   const __grid_constant__ CUtensorMap tm_mask)
{
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *aring = smem;                       // [NS][a_hi | a_lo]
    unsigned char *wring = smem + pl.off_w;            // [2 units][TPR stages][b_hi | b_lo], one unit ahead of the samplers
    unsigned char *boxes = smem + pl.off_box;          // [2][BH][BW][8] fp32
    const T *oms = reinterpret_cast<const T *>(smem + pl.off_om);           // [2][3*KK planes][128 px]
    __shared__ __align__(8) uint64_t slot_free[NS], a_full[NS], wu_full[2], wu_free[2];
    __shared__ __align__(8) uint64_t box_full[2], box_free[2], om_full[2], om_free[2], acc_full[2], acc_free[2];
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int units = d.dg * pl.ncs;                   // (group, chunk) pairs per tile
    const int stages = units * TPR;                    // operand stages per tile
    const int total_tiles = d.B * pl.ntiles;
    const uint32_t sbo = (uint32_t)pl.kch * 128u;
    const uint32_t wb = 2u * (uint32_t)pl.b_bytes;       // one stage's weight image (hi | lo)

    if (warp == 0) umma::tmem_alloc<TMEM_COLS>(&tmem_slot);
    if (tid == 32) {
        for (int i = 0; i < NS; ++i) { umma::mbar_init(&slot_free[i], 1); umma::mbar_init(&a_full[i], N_SAMP); }
        for (int i = 0; i < 2; ++i) {
            umma::mbar_init(&wu_full[i], 1); umma::mbar_init(&wu_free[i], 1);
            umma::mbar_init(&box_full[i], 1); umma::mbar_init(&box_free[i], N_SAMP);
            umma::mbar_init(&om_full[i], 1); umma::mbar_init(&om_free[i], N_SAMP);
            umma::mbar_init(&acc_full[i], 1); umma::mbar_init(&acc_free[i], N_EPI);
        }
        umma::mbar_fence_init();
    }
#ifdef EBFI_DEBUG_HANG_ADDR
    if (tid == 0 && blockIdx.x == 0)
        printf("fwd barriers: slot_free 0x%x a_full 0x%x wu_full 0x%x wu_free 0x%x box_full 0x%x box_free 0x%x om_full 0x%x om_free 0x%x acc_full 0x%x acc_free 0x%x\n",
               umma::smem_u32(slot_free), umma::smem_u32(a_full), umma::smem_u32(wu_full), umma::smem_u32(wu_free), umma::smem_u32(box_full),
               umma::smem_u32(box_free), umma::smem_u32(om_full), umma::smem_u32(om_free), umma::smem_u32(acc_full), umma::smem_u32(acc_free));
#endif
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;

    auto tile_origin = [&](int tile, int &b, int &ty0, int &tx0) {
        tx0 = (tile % pl.tiles_x) * TW; tile /= pl.tiles_x;
        ty0 = (tile % pl.tiles_y) * TH;
        b = tile / pl.tiles_y;
    };

    if (warp < N_EPI) {
        // ================= epilogue: TMEM -> + bias -> NCHW =================
        const size_t plane = (size_t)d.Ho * d.Wo;
        const int p = warp * 32 + lane;
        const uint32_t lane_base = (uint32_t)warp * 32u;
        const int total_steps = stages * KSTEPS, nused = min(pl.nacc, total_steps);
        int k = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++k) {
            const int ab = k & 1;
            int b, ty0, tx0;
            tile_origin(tile, b, ty0, tx0);
            const int ho = ty0 + p / TW, wo = tx0 + p % TW;
            const bool valid = ho < d.Ho && wo < d.Wo;
            T *out_p = output + (size_t)b * d.Co * plane + (size_t)ho * d.Wo + wo;
            umma::mbar_wait(&acc_full[ab], (uint32_t)((k >> 1) & 1));
            umma::fence_after_sync();
            const uint32_t tb = tmem + (uint32_t)(ab * ACC_COLS);
            for (int cb = 0; cb < d.Co; cb += 8) {
                float v[8], u[8];
                umma::tmem_ld8(umma::tmem_addr(tb, lane_base, pl.nacc * d.Co + cb), v);
                umma::tmem_ld_wait();
                for (int j = 0; j < nused; ++j) {
                    umma::tmem_ld8(umma::tmem_addr(tb, lane_base, j * d.Co + cb), u);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] += u[i];
                }
                if (valid) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) out_p[(size_t)(cb + i) * plane] = st_act<T>(v[i] + __ldg(bias + cb + i));
                }
            }
            umma::fence_before_sync();
            __syncwarp();
            if (lane == 0) umma::mbar_arrive(&acc_free[ab]);
        }
    } else if (warp < W_MMA) {
        // ================= samplers: thread (pixel p, row r) =================
        const int st = tid - N_EPI * 32;
        const int p = st % TM, r = st / TM;
        const size_t plane = (size_t)d.Ho * d.Wo, in_plane = (size_t)d.H * d.W;
        const unsigned uplane = (unsigned)plane;
        const int a_row = (p >> 3) * (pl.kch * 32) + (p & 7) * 4;         // floats, row of pixel p in an A image
        float asum = 0.f;                          // sum |offset| of this thread's taps (packed entry)
        int slot = 0; uint32_t sph = 0;            // ring slot / parity of the current stage
        int n = 0, U = 0, G = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int b, ty0, tx0;
            tile_origin(tile, b, ty0, tx0);
            const int ho = ty0 + p / TW, wo = tx0 + p % TW;
            const bool valid = ho < d.Ho && wo < d.Wo;
            const unsigned upix = (unsigned)(ho * d.Wo + wo);
            const int by0 = ty0 * d.sh - d.ph - pl.my, bx0 = tx0 * d.sw - d.pw - pl.mx;
            float by[TPR], bx[TPR];
            bool tv[TPR];
#pragma unroll
            for (int s = 0; s < TPR; ++s) {
                const int t = r * TPR + s, i = t / d.kw, j = t - i * d.kw;
                tv[s] = valid && t < d.KK;
                by[s] = (float)(ho * d.sh - d.ph + i * d.dh);
                bx[s] = (float)(wo * d.sw - d.pw + j * d.dw);
            }
            for (int g = 0; g < d.dg; ++g, ++G) {
                float sy[TPR], sx[TPR], sm[TPR];
                if (pl.use_om_tma) {
                    const int ob = G & 1;
                    umma::mbar_wait(&om_full[ob], (uint32_t)((G >> 1) & 1));
                    const T *om = oms + ob * (pl.om_bytes / (int)sizeof(T));
#pragma unroll
                    for (int s = 0; s < TPR; ++s) {
                        const int t = r * TPR + s;
                        float dy = 0.f, dx = 0.f, m = 0.f;
                        if (tv[s]) { dy = act_f(om[(2 * t) * TM + p]); dx = act_f(om[(2 * t + 1) * TM + p]); m = act_f(om[(2 * d.KK + t) * TM + p]); }
                        sy[s] = tv[s] ? by[s] + dy : -2.f;
                        sx[s] = tv[s] ? bx[s] + dx : -2.f;
                        sm[s] = mask_act_t<PACKED>(m);
                        if (PACKED) asum += fabsf(dy) + fabsf(dx);
                    }
                    __syncwarp();
                    if (lane == 0) umma::mbar_arrive(&om_free[ob]);
                } else {
                    const T *off_bg = off_ptr(d, offset, b, g, plane);
                    const T *mask_bg = mask_ptr(d, mask, b, g, plane);
#pragma unroll
                    for (int s = 0; s < TPR; ++s) {
                        float dy = 0.f, dx = 0.f, m = 0.f;
                        if (tv[s]) tap_read(off_bg, mask_bg, uplane, (unsigned)(r * TPR + s), upix, dy, dx, m);
                        sy[s] = tv[s] ? by[s] + dy : -2.f;
                        sx[s] = tv[s] ? bx[s] + dx : -2.f;
                        sm[s] = mask_act_t<PACKED>(m);
                        if (PACKED) asum += fabsf(dy) + fabsf(dx);
                    }
                }
                for (int ci = 0; ci < pl.ncs; ++ci, ++U) {
                    const int bb = U & 1;
                    umma::mbar_wait(&box_full[bb], (uint32_t)((U >> 1) & 1));
                    const uint32_t box_s = umma::smem_u32(boxes + bb * BOX_BYTES);
                    const float *ibf = in_blk + (((size_t)b * d.dg + g) * pl.ncs + ci) * in_plane * 8;
#pragma unroll 1
                    for (int s = 0; s < TPR; ++s, ++n) {
                        float y = sy[0], x = sx[0], m = sm[0];               // register select, no local-memory indexing
#pragma unroll
                        for (int q = 1; q < TPR; ++q)
                            if (s == q) { y = sy[q]; x = sx[q]; m = sm[q]; }
                        float ha[4], hb[4], hi[8], lo[8];
                        const bool swapped = sample8(y, x, m, d.H, d.W, box_s, by0, bx0, ibf, lane, ha, hb);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            umma::split_tf32(ha[j], hi[j], lo[j]);
                            umma::split_tf32(hb[j], hi[4 + j], lo[4 + j]);
                        }
                        if (n >= NS) umma::mbar_wait(&slot_free[slot], sph ^ 1u);      // MMAs of stage n - NS are done
                        float *a_hi = reinterpret_cast<float *>(aring + slot * 2 * pl.a_bytes);
                        float *a_lo = reinterpret_cast<float *>(aring + slot * 2 * pl.a_bytes + pl.a_bytes);
                        // K order: row r major, channel minor; the two 16-byte K chunks of this tap trade places when swapped
                        const int off_a = a_row + (r * 2 + (swapped ? 1 : 0)) * 32, off_b = a_row + (r * 2 + (swapped ? 0 : 1)) * 32;
                        *reinterpret_cast<float4 *>(a_hi + off_a) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<float4 *>(a_lo + off_a) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                        *reinterpret_cast<float4 *>(a_hi + off_b) = make_float4(hi[4], hi[5], hi[6], hi[7]);
                        *reinterpret_cast<float4 *>(a_lo + off_b) = make_float4(lo[4], lo[5], lo[6], lo[7]);
                        umma::fence_smem_to_async();
                        __syncwarp();
                        if (lane == 0) umma::mbar_arrive(&a_full[slot]);
                        if (++slot == NS) { slot = 0; sph ^= 1u; }
                    }
                    __syncwarp();
                    if (lane == 0) umma::mbar_arrive(&box_free[bb]);
                }
            }
        }
        if (PACKED && d.abs_sum) warp_atomic_sum(d.abs_sum, asum);
    } else if (warp == W_MMA) {
        // ================= MMA issuer: all lanes run the loop with warp-uniform values, one elected lane issues =================
        const bool leader = umma::elect_one();
        const uint32_t idesc = umma::instr_desc_tf32(TM, d.Co, 0, 0);
        int slot = 0; uint32_t sph = 0;
        int k = 0, U = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++k) {
            const int ab = k & 1;
            if (k >= 2) umma::mbar_wait(&acc_free[ab], (uint32_t)(((k >> 1) - 1) & 1));
            umma::fence_after_sync();
            const uint32_t tb = tmem + (uint32_t)(ab * ACC_COLS);
            int step = 0;
            uint32_t hsel = 0;
            const uint32_t d_x = tb + (uint32_t)(pl.nacc * d.Co);
            for (int u = 0; u < units; ++u, ++U) {
                const int ub = U & 1;
                umma::mbar_wait(&wu_full[ub], (uint32_t)((U >> 1) & 1));
                for (int s = 0; s < TPR; ++s) {
                    umma::mbar_wait(&a_full[slot], sph);
                    umma::fence_after_sync();
                    const uint32_t ah = umma::smem_u32(aring + slot * 2 * pl.a_bytes);
                    const uint32_t bh = umma::smem_u32(wring + ub * pl.unit_bytes) + (uint32_t)s * wb;
                    uint64_t dah = umma::smem_desc(ah, 128, sbo), dal = umma::smem_desc(ah + (uint32_t)pl.a_bytes, 128, sbo);
                    uint64_t dbh = umma::smem_desc(bh, 128, sbo), dbl = umma::smem_desc(bh + (uint32_t)pl.b_bytes, 128, sbo);
                    // K steps of 8 (two 16-byte chunks = +256 B = +16 in the descriptor's address field); the hi*hi products
                    // rotate over `nacc` accumulators (no division: hsel is carried), the cross terms share one
#pragma unroll
                    for (int ks = 0; ks < KSTEPS; ++ks) {
                        const uint32_t d_h = tb + hsel * (uint32_t)d.Co;
                        if (leader) {
                            umma::mma_tf32(d_x, dal + 16 * ks, dbh + 16 * ks, idesc, step > 0);
                            umma::mma_tf32(d_x, dah + 16 * ks, dbl + 16 * ks, idesc, true);
                            umma::mma_tf32(d_h, dah + 16 * ks, dbh + 16 * ks, idesc, step >= pl.nacc);
                        }
                        ++step;
                        if (++hsel == (uint32_t)pl.nacc) hsel = 0;
                    }
                    if (leader) {
                        umma::commit(&slot_free[slot]);
                        if (s == TPR - 1) umma::commit(&wu_free[ub]);
                        if (s == TPR - 1 && u == units - 1) umma::commit(&acc_full[ab]);
                    }
                    __syncwarp();
                    if (++slot == NS) { slot = 0; sph ^= 1u; }
                }
            }
        }
    } else if (warp == W_BOX) {
        // ================= box / offset-mask loader =================
        if (lane == 0) {
            int U = 0, G = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int b, ty0, tx0;
                tile_origin(tile, b, ty0, tx0);
                const int by0 = ty0 * d.sh - d.ph - pl.my, bx0 = tx0 * d.sw - d.pw - pl.mx;
                for (int g = 0; g < d.dg; ++g, ++G) {
                    if (pl.use_om_tma) {
                        const int ob = G & 1;
                        if (G >= 2) umma::mbar_wait(&om_free[ob], (uint32_t)(((G >> 1) - 1) & 1));
                        unsigned char *dst = smem + pl.off_om + ob * pl.om_bytes;
                        umma::mbar_expect_tx(&om_full[ob], (uint32_t)pl.om_bytes);
                        tma::load_3d(dst, &tm_off, tx0, ty0, b * d.off_bp + g * 2 * d.KK, &om_full[ob]);
                        tma::load_3d(dst + 2 * d.KK * TM * (int)sizeof(T), &tm_mask, tx0, ty0, b * d.mask_bp + g * d.KK, &om_full[ob]);
                    }
                    for (int ci = 0; ci < pl.ncs; ++ci, ++U) {
                        const int bb = U & 1;
                        if (U >= 2) umma::mbar_wait(&box_free[bb], (uint32_t)(((U >> 1) - 1) & 1));
                        umma::mbar_expect_tx(&box_full[bb], (uint32_t)BOX_BYTES);
                        tma::load_3d(boxes + bb * BOX_BYTES, &tm_box, bx0 * 8, by0, (b * d.dg + g) * pl.ncs + ci, &box_full[bb]);
                    }
                }
            }
        }
    } else if (warp == W_WGT) {
        // ================= weight-image loader =================
        if (lane == 0) {
            int U = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                for (int u = 0; u < units; ++u, ++U) {
                    const int ub = U & 1;
                    if (U >= 2) umma::mbar_wait(&wu_free[ub], (uint32_t)(((U >> 1) - 1) & 1));
                    umma::mbar_expect_tx(&wu_full[ub], (uint32_t)pl.unit_bytes);
                    umma::bulk_g2s(wring + ub * pl.unit_bytes, wimg + (size_t)u * (pl.unit_bytes / 4), (uint32_t)pl.unit_bytes, &wu_full[ub]);
                }
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tmem);
}

// Weight images for the bulk copies: [chunk][stage][hi | lo][Co * Ksp] in operand (shared-memory)
// order, k'' = rr * 8 + cc  <-  weight[co][(c0 + cc) * KK + rr * TPR + s]; zero where the tap or
// the K padding does not exist. 2 x 147 KB at the benchmark shape.
__global__ void dcn_prep_weights(const float *__restrict__ weight, float *__restrict__ wimg, DcnDims d, BoxPlan pl)
{
    const int per_img = d.Co * pl.Ksp;
    const int nimg = d.dg * pl.ncs * pl.TPR;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nimg * per_img; i += gridDim.x * blockDim.x) {
        const int img = i / per_img, e = i - img * per_img;
        const int s = img % pl.TPR, chunk = img / pl.TPR;
        const int c0 = (chunk / pl.ncs) * d.cpg + (chunk % pl.ncs) * 8;
        const int kk = e & 3, cor = (e >> 2) & 7, rest = e >> 5;
        const int kc = rest % pl.kch, cog = rest / pl.kch;
        const int co = cog * 8 + cor, kp = kc * 4 + kk;
        const int rr = kp / 8, cc = kp - rr * 8, t = rr * pl.TPR + s;
        float hi = 0.f, lo = 0.f;
        if (kp < pl.Ks && t < d.KK)
            umma::split_tf32(__ldg(weight + (size_t)co * d.C * d.KK + (size_t)(c0 + cc) * d.KK + t), hi, lo);
        wimg[(size_t)img * 2 * per_img + e] = hi;
        wimg[(size_t)img * 2 * per_img + per_img + e] = lo;
    }
}

// act_bytes: size of one offset / mask element (4 or 2); it sets the shared-memory planes and the TMA row alignment
bool make_plan(const DcnDims &d, BoxPlan &pl, int act_bytes = 4)
{
    if (d.Co % 16 != 0 || d.Co > 128 || d.cpg % 8 != 0) return false;   // blocked layout: 8-channel chunks
    if ((long)2 * d.KK * d.Ho * d.Wo >= (1L << 31)) return false;        // 32-bit offsets inside one group
    if ((long)d.B * d.C / 8 >= (1L << 31) || (long)d.W * 8 >= (1L << 31)) return false;
    pl.nacc = std::min(3, ACC_COLS / d.Co - 1);
    if (pl.nacc < 1) return false;
    pl.TPR = ceil_div(d.KK, NR);
    if (pl.TPR > 4) return false;                       // kernels up to 12 taps (3x3, 1x1, 3x4, ...)
    pl.ncs = d.cpg / 8;
    pl.Ks = NR * 8;
    pl.Ksp = ebfi::round_up(pl.Ks, 8);
    pl.kch = pl.Ksp / 4;
    pl.a_bytes = TM * pl.Ksp * 4;
    pl.b_bytes = d.Co * pl.Ksp * 4;
    pl.tiles_x = ceil_div(d.Wo, TW);
    pl.tiles_y = ceil_div(d.Ho, TH);
    pl.ntiles = pl.tiles_x * pl.tiles_y;
    // box margins: centre the tile's undeformed sampling footprint (floor coordinates need one extra row / pixel)
    const int fh = (TH - 1) * d.sh + (d.kh - 1) * d.dh + 1, fw = (TW - 1) * d.sw + (d.kw - 1) * d.dw + 1;
    pl.my = std::max(0, (BH - 1 - fh + 1) / 2);
    pl.mx = std::max(0, (BW - 1 - fw + 1) / 2);
    pl.om_bytes = 3 * d.KK * TM * act_bytes;
    pl.use_om_tma = d.Wo % (16 / act_bytes) == 0 && getenv("EBFI_DCN_NO_TMA") == nullptr;
    pl.unit_bytes = pl.TPR * 2 * pl.b_bytes;
    pl.off_w = NS * 2 * pl.a_bytes;
    pl.off_box = pl.off_w + 2 * pl.unit_bytes;
    pl.off_om = pl.off_box + 2 * BOX_BYTES;
    pl.smem = pl.off_om + 2 * pl.om_bytes;
    return pl.smem <= 225 * 1024;
}

}  // namespace

// byte offset of the group-blocked input copy inside the forward workspace (0: this shape has no tensor-core forward)
size_t forward_tc_blocked_offset(const DcnDims &d)
{
    BoxPlan pl{};
    if (!make_plan(d, pl)) return 0;
    return ebfi::round_up((size_t)d.dg * pl.ncs * pl.TPR * 2 * pl.b_bytes, (size_t)256);
}

size_t forward_tc_workspace(const DcnDims &d)
{
    BoxPlan pl{};
    if (!make_plan(d, pl)) return 0;
    return ebfi::round_up((size_t)d.dg * pl.ncs * pl.TPR * 2 * pl.b_bytes, (size_t)256) +
           (size_t)d.B * d.C * d.H * d.W * sizeof(float);
}

template <typename T>
int forward_tc(cudaStream_t st, const DcnDims &d, const T *input, const float *weight, const float *bias,
               const T *offset, const T *mask, T *output, void *workspace, size_t workspace_bytes)
{
    BoxPlan pl{};
    if (!make_plan(d, pl, (int)sizeof(T))) return EBFI_ERR_UNSUPPORTED;
    const size_t wbytes = (size_t)d.dg * pl.ncs * pl.TPR * 2 * pl.b_bytes;
    const size_t need = ebfi::round_up(wbytes, (size_t)256) + (size_t)d.B * d.C * d.H * d.W * sizeof(float);
    // the blocked input copy inside the workspace is read by TMA (16-byte) and by 256-bit loads (32-byte alignment)
    if (!workspace || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 31u)) return EBFI_ERR_UNSUPPORTED;
    float *wimg = static_cast<float *>(workspace);
    float *in_blk = reinterpret_cast<float *>(static_cast<char *>(workspace) + ebfi::round_up(wbytes, (size_t)256));
    dcn_prep_weights<<<ceil_div((int)(wbytes / 8), 256), 256, 0, st>>>(weight, wimg, d, pl);
    EBFI_LAUNCH_OK("dcn_prep_weights");
    if (int rc = launch_nchw_to_blocked(st, input, in_blk, d.B * d.C / 8, d.H * d.W)) return rc;

    CUtensorMap tm_box{}, tm_off{}, tm_mask{};
    {
        const uint64_t dims[3] = {(uint64_t)d.W * 8, (uint64_t)d.H, (uint64_t)d.B * d.C / 8};
        const uint64_t str[2] = {(uint64_t)d.W * 32, (uint64_t)d.H * d.W * 32};
        const uint32_t box[3] = {BW * 8, BH, 1};
        if (int rc = tma::encode_3d(tm_box, in_blk, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dims, str, box)) return rc;
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
    const unsigned grid = (unsigned)std::min(ebfi::sm_count(), d.B * pl.ntiles);
#define EBFI_FWD_BOX(R)                                                                                       \
    do {                                                                                                      \
        if (d.packed) {                                                                                       \
            EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_fwd_box_kernel<R, true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem)); \
            dcn_fwd_box_kernel<R, true, T><<<grid, NTHR, pl.smem, st>>>(in_blk, bias, offset, mask, output, wimg, d, pl, tm_box, tm_off, tm_mask); \
        } else {                                                                                              \
            EBFI_CUDA_OK(cudaFuncSetAttribute(dcn_fwd_box_kernel<R, false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem)); \
            dcn_fwd_box_kernel<R, false, T><<<grid, NTHR, pl.smem, st>>>(in_blk, bias, offset, mask, output, wimg, d, pl, tm_box, tm_off, tm_mask); \
        }                                                                                                     \
    } while (0)
    switch (pl.TPR) {
    case 1: EBFI_FWD_BOX(1); break;
    case 2: EBFI_FWD_BOX(2); break;
    case 3: EBFI_FWD_BOX(3); break;
    default: EBFI_FWD_BOX(4); break;
    }
#undef EBFI_FWD_BOX
    EBFI_LAUNCH_OK("dcn_fwd_box_kernel");
    return EBFI_OK;
}
template int forward_tc<float>(cudaStream_t, const DcnDims &, const float *, const float *, const float *, const float *,
                               const float *, float *, void *, size_t);
template int forward_tc<__nv_bfloat16>(cudaStream_t, const DcnDims &, const __nv_bfloat16 *, const float *, const float *,
                                       const __nv_bfloat16 *, const __nv_bfloat16 *, __nv_bfloat16 *, void *, size_t);
template int forward_tc<__half>(cudaStream_t, const DcnDims &, const __half *, const float *, const float *,
                                const __half *, const __half *, __half *, void *, size_t);

}  // namespace ebfi_dcn
