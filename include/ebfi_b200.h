/*
 * ebfi_b200.h — C ABI of the B200-native event-frame alignment kernels.
 *
 * This is the drop-in boundary for the three hot-path operators of
 * WarranWeng/EBFI-BE (see SURVEY.md §8b):
 *
 *   - DCNv2 modulated deformable convolution, forward + backward
 *       replaces  _ext.dcn_v2_forward / _ext.dcn_v2_backward
 *       (reference: models/DCNv2/src/dcn_v2.h:9-92, vision.cpp:4-9,
 *        src/cuda/dcn_v2_cuda.cu:20-216, src/cuda/dcn_v2_im2col_cuda.cu:125-402)
 *   - FAC KernelConv2D per-pixel K x K filter, forward + backward
 *       replaces  kernelconv2d_cuda.forward / kernelconv2d_cuda.backward
 *       (reference: models/FAC/kernelconv2d/KernelConv2D_cuda.cpp:10-61,
 *        KernelConv2D_kernel.cu:25-204)
 *   - event -> image / voxel / polarity-stack encoders
 *       replaces the index_put_ scatters of dataloader/encodings.py:243-377
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer unless its name ends in `_host`.
 *   - Tensors are dense, row-major NCHW fp32 exactly as the reference's
 *     `data_ptr<float>()` callers hand them over (dcn_v2_cuda.cu:79-86,
 *     KernelConv2D_kernel.cu:68-77).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     Nothing here synchronises the stream or the device.
 *   - Return value: 0 on success, a negative EBFI_ERR_* otherwise; no C++
 *     exception ever crosses this boundary. ebfi_last_error() returns a
 *     thread-local, human readable message for the last failing call.
 *   - There is no CPU fallback anywhere behind this ABI.
 */
#ifndef EBFI_B200_H_
#define EBFI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EBFI_OK               0
#define EBFI_ERR_INVALID     -1   /* bad shape / null pointer / unsupported argument */
#define EBFI_ERR_CUDA        -2   /* a CUDA runtime call or kernel launch failed */
#define EBFI_ERR_WORKSPACE   -3   /* workspace too small (query the *_workspace_bytes fn) */
#define EBFI_ERR_UNSUPPORTED -4   /* valid request this build does not implement */

#define EBFI_ABI_VERSION 3

/* ---- library ---------------------------------------------------------------- */

int         ebfi_abi_version(void);
const char *ebfi_last_error(void);
/* Compute capability major*10+minor of the current device, or a negative error. */
int         ebfi_device_arch(void);

/* ---- DCNv2 modulated deformable convolution --------------------------------- */

/* Geometry of one call; same fields, same meaning and same order as the integer
 * tail of _ext.dcn_v2_forward (models/DCNv2/src/dcn_v2.h:9-23). */
typedef struct ebfi_dcn_geom {
    int batch, channels, height, width;   /* input  (B, C, H, W)                */
    int channels_out;                     /* weight (Cout, C, kernel_h, kernel_w) */
    int kernel_h, kernel_w;
    int stride_h, stride_w;
    int pad_h, pad_w;
    int dilation_h, dilation_w;
    int deformable_group;                 /* offset (B, 2*dg*kh*kw, Ho, Wo); mask (B, dg*kh*kw, Ho, Wo) */
    int flags;                            /* 0, or EBFI_DCN_DETERMINISTIC (new; not in the reference's argument list) */
} ebfi_dcn_geom;

/* Backward only: ALL five gradients bit-reproducible run to run for ANY offsets. The reference's col2im uses float
 * atomicAdd (dcn_v2_im2col_cuda.cu:249) and is not. The DEFAULT mode (no flag) is already bit-reproducible on the
 * box kernel (csrc/dcn_bwd_box.cu: 8, 16 or 32 channels per deformable group, 64 outputs, a tile footprint that fits
 * its box) for every sample whose four corners lie within ~7 pixels of its tile's undeformed footprint: those
 * accumulate in shared-memory fixed point and the per-tile boxes are summed in a fixed order; only samples beyond
 * that ("far" samples) use float red.global.add. With this flag the same box kernel runs, and its far samples add
 * into a 64-bit fixed-point buffer instead (integer atomics are associative): one extra pass over grad_output for the
 * scale, and the same bits as the default mode wherever no sample is far. Shapes the box kernel does not cover
 * accumulate ALL of grad_input in 64-bit fixed point: csrc/dcn_bwd_tc.cu for 8 channels per group and 64 outputs
 * (e.g. stride 2 in W), the CUDA-core kernel otherwise. The fixed-point scale, a power of two derived on the device
 * from max|grad_output|, max|weight| and max|mask| such that no sum can overflow, applies to those 64-bit sums only
 * (on the box kernel: the far samples); its resolution is at least 2^-20 of the largest possible single
 * contribution. A non-finite gradient yields NaN (never a silent zero). */
#define EBFI_DCN_DETERMINISTIC 1

/* Backward only: `input` is not the NCHW tensor but its group-blocked copy [B][C/8][H][W][8 channels] (32-byte aligned)
 * that ebfi_dcnv2_forward left in its workspace at byte offset ebfi_dcnv2_blocked_input_offset(g) — a caller that keeps
 * the forward workspace alive until the backward (an autograd context) saves the re-blocking pass. Only valid when
 * that offset is non-zero (with or without EBFI_DCN_DETERMINISTIC). */
#define EBFI_DCN_INPUT_BLOCKED 2

/* Output spatial size, formula of dcn_v2_cuda.cu:64-65. Returns EBFI_ERR_INVALID
 * when the geometry is inconsistent (non-positive sizes, C % dg != 0, ...). */
int ebfi_dcnv2_output_size(const ebfi_dcn_geom *g, int *height_out, int *width_out);

/* Scratch the backward pass needs: per-CTA grad_weight / grad_bias partials, the group-blocked copy of the input and,
 * on the tensor-core path, one dense 24 x 30-pixel grad_input box per (128-pixel tile, deformable group) — about 5.6x
 * the size of grad_input. 32-byte aligned device memory. The column buffer of the reference (dcn_v2_cuda.cu:68) never
 * exists in HBM in either pass. */
size_t ebfi_dcnv2_backward_workspace_bytes(const ebfi_dcn_geom *g);

/* Scratch for the forward pass: the TF32 hi/lo weight images the tensor-core kernel streams
 * into shared memory (2 x the weight tensor) + the group-blocked input copy. 32-byte aligned device memory. Without it (NULL /
 * too small) the forward falls back to its CUDA-core kernel, which needs none. */
size_t ebfi_dcnv2_forward_workspace_bytes(const ebfi_dcn_geom *g);

/* Byte offset of the group-blocked input copy inside the forward workspace after ebfi_dcnv2_forward, or 0 when this
 * geometry does not produce / the backward cannot consume one, or EBFI_DCN_IMPL=simt is set in the environment (the
 * CUDA-core kernels neither write nor read it) (see EBFI_DCN_INPUT_BLOCKED). */
size_t ebfi_dcnv2_blocked_input_offset(const ebfi_dcn_geom *g);

/* out[b,co,h,w] = bias[co] + sum_{c,i,j} weight[co,c,i,j] * mask * bilinear(input[b,c], ...)
 * Replaces dcn_v2_cuda_forward (dcn_v2_cuda.cu:20-95). `output` is written in
 * full (no pre-zeroing needed). */
int ebfi_dcnv2_forward(void *stream, const ebfi_dcn_geom *g,
                       const float *input, const float *weight, const float *bias,
                       const float *offset, const float *mask,
                       float *output, void *workspace, size_t workspace_bytes);

/* All five gradients of dcn_v2_cuda_backward (dcn_v2_cuda.cu:97-216), every
 * output written in full. grad_offset / grad_mask / grad_weight / grad_bias are
 * reduced in a fixed order (bit-reproducible run to run); grad_input: see EBFI_DCN_DETERMINISTIC.
 * Reference quirk kept on purpose: the grad_input scatter uses pad_h for BOTH
 * paddings (dcn_v2_im2col_cuda.cu:368 passes `pad_h, pad_h`). */
int ebfi_dcnv2_backward(void *stream, const ebfi_dcn_geom *g,
                        const float *input, const float *weight, const float *bias,
                        const float *offset, const float *mask,
                        const float *grad_output,
                        float *grad_input, float *grad_offset, float *grad_mask,
                        float *grad_weight, float *grad_bias,
                        void *workspace, size_t workspace_bytes);

/* Packed variants: the deformable conv fed directly with the raw output of the module's
 * `conv_offset_mask` (models/DCNv2/dcn_v2.py:217-227, DCN.forward :179-187):
 *   offset_mask : (B, 3*dg*kh*kw, Ho, Wo); channels [0, 2*dg*kh*kw) ARE cat(o1, o2) = the offsets,
 *                 the last third are the mask logits; the kernels apply sigmoid() themselves.
 * This folds torch.chunk / torch.cat / torch.sigmoid (and their backward passes) into the kernels:
 * `grad_offset_mask` has the layout of `offset_mask` and already contains
 * grad_mask * m * (1 - m) in its last third. `abs_offset_sum` (nullable, 1 float, device) receives
 * sum |offset| so that the module's `offset_mean > 100` warning needs no separate pass over the
 * offsets (it is a statistic: accumulated with atomics, not bit-reproducible).
 * Workspace sizes are those of the unpacked calls. */
int ebfi_dcnv2_forward_packed(void *stream, const ebfi_dcn_geom *g,
                              const float *input, const float *weight, const float *bias,
                              const float *offset_mask, float *output, float *abs_offset_sum,
                              void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_backward_packed(void *stream, const ebfi_dcn_geom *g,
                               const float *input, const float *weight, const float *bias,
                               const float *offset_mask, const float *grad_output,
                               float *grad_input, float *grad_offset_mask,
                               float *grad_weight, float *grad_bias,
                               void *workspace, size_t workspace_bytes);

/* bf16 activation variants of the five DCNv2 entries above (mixed precision: bf16 activations, fp32 parameters), same
 * argument order and the same workspace queries. input, offset, mask / offset_mask, grad_output, output, grad_input,
 * grad_offset, grad_mask and grad_offset_mask are `__nv_bfloat16*` NCHW; weight, bias, grad_weight, grad_bias and
 * abs_offset_sum stay fp32. With EBFI_DCN_INPUT_BLOCKED, `input` is the fp32 group-blocked copy, as for the fp32 entry.
 * Only the activation loads and stores change: loads widen exactly, results are rounded once (RN) from the fp32 values
 * the fp32 entries store, so on bf16-valued inputs every activation result equals the fp32 entry's result rounded to
 * bf16, and grad_weight / grad_bias are equal.
 * They run only where the tensor-core kernels run: the forward for Cout a multiple of 16 up to 128, channels per group
 * a multiple of 8 and up to 12 taps, with a workspace of ebfi_dcnv2_forward_workspace_bytes; the backward for
 * Cout == 64, 8 / 16 / 32 channels per group, a tile footprint that fits the box and a 16-byte aligned grad_output, in
 * both modes of EBFI_DCN_DETERMINISTIC (the bound of the deterministic scale is taken on the widened values); neither
 * under EBFI_DCN_IMPL=simt. Anything else returns EBFI_ERR_UNSUPPORTED before any work is enqueued: take the fp32 entry
 * on widened copies. ebfi_dcnv2_backward_dp_bf16 is declared with the data-parallel entries below. */
int ebfi_dcnv2_forward_bf16(void *stream, const ebfi_dcn_geom *g,
                            const void *input, const float *weight, const float *bias,
                            const void *offset, const void *mask,
                            void *output, void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_backward_bf16(void *stream, const ebfi_dcn_geom *g,
                             const void *input, const float *weight, const float *bias,
                             const void *offset, const void *mask,
                             const void *grad_output,
                             void *grad_input, void *grad_offset, void *grad_mask,
                             float *grad_weight, float *grad_bias,
                             void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_forward_packed_bf16(void *stream, const ebfi_dcn_geom *g,
                                   const void *input, const float *weight, const float *bias,
                                   const void *offset_mask, void *output, float *abs_offset_sum,
                                   void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_backward_packed_bf16(void *stream, const ebfi_dcn_geom *g,
                                    const void *input, const float *weight, const float *bias,
                                    const void *offset_mask, const void *grad_output,
                                    void *grad_input, void *grad_offset_mask,
                                    float *grad_weight, float *grad_bias,
                                    void *workspace, size_t workspace_bytes);

/* fp16 activation variants (torch.autocast's default dtype): the *_bf16 entries above with `__half*` in place of
 * `__nv_bfloat16*`, same arguments, workspaces, coverage and EBFI_ERR_UNSUPPORTED. On fp16-valued inputs every
 * activation result equals the fp32 entry's result rounded once (RN) to fp16, and grad_weight / grad_bias are equal.
 * An activation result beyond the fp16 range is +-inf, as a cast to fp16 gives; NaN stays NaN.
 * ebfi_dcnv2_backward_dp_fp16 is declared with the data-parallel entries below. */
int ebfi_dcnv2_forward_fp16(void *stream, const ebfi_dcn_geom *g,
                            const void *input, const float *weight, const float *bias,
                            const void *offset, const void *mask,
                            void *output, void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_backward_fp16(void *stream, const ebfi_dcn_geom *g,
                             const void *input, const float *weight, const float *bias,
                             const void *offset, const void *mask,
                             const void *grad_output,
                             void *grad_input, void *grad_offset, void *grad_mask,
                             float *grad_weight, float *grad_bias,
                             void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_forward_packed_fp16(void *stream, const ebfi_dcn_geom *g,
                                   const void *input, const float *weight, const float *bias,
                                   const void *offset_mask, void *output, float *abs_offset_sum,
                                   void *workspace, size_t workspace_bytes);
int ebfi_dcnv2_backward_packed_fp16(void *stream, const ebfi_dcn_geom *g,
                                    const void *input, const float *weight, const float *bias,
                                    const void *offset_mask, const void *grad_output,
                                    void *grad_input, void *grad_offset_mask,
                                    float *grad_weight, float *grad_bias,
                                    void *workspace, size_t workspace_bytes);

/* ---- FAC KernelConv2D ------------------------------------------------------- */

/* input  : (B, C, H+K-1, W+K-1)   already padded by the caller (KernelConv2D.py:82-86)
 * kernel : (B, C*K*K, H, W)       channel order c*K*K + ky*K + kx (KernelConv2D_kernel.cu:47)
 * output : (B, C, H, W)           every element written
 * Replaces KernelConv2D_forward_cuda (KernelConv2D_cuda.cpp:10-30). */
int ebfi_fac_forward(void *stream, const float *input, const float *kernel, float *output,
                     int batch, int channels, int height_out, int width_out, int kernel_size);

/* Scratch for ebfi_fac_backward: the K-1 overhang rows each row segment hands to the
 * segment below it, plus one arrival counter per hand-off. An upper bound for the
 * given shape; 16-byte aligned device memory. */
size_t ebfi_fac_backward_workspace_bytes(int batch, int channels, int height_out, int width_out,
                                         int kernel_size);

/* grad_input  : (B, C, H+K-1, W+K-1), grad_kernel : (B, C*K*K, H, W); both written
 * in full — the caller's zero fill (KernelConv2D.py:50-51) is not relied upon.
 * One fused pass: grad_output and kernel are each read once, and grad_input is
 * reduced in a fixed order (bit-reproducible, no atomics on data).
 * Replaces KernelConv2D_backward_cuda (KernelConv2D_cuda.cpp:32-56). */
int ebfi_fac_backward(void *stream, const float *input, const float *kernel,
                      const float *grad_output, float *grad_input, float *grad_kernel,
                      int batch, int channels, int height_out, int width_out, int kernel_size,
                      void *workspace, size_t workspace_bytes);

/* bf16 storage variants (new; the reference is fp32-only, KernelConv2D_kernel.cu:68 `data<float>()`):
 * every tensor is bfloat16, all arithmetic and the grad_input reduction are fp32, results are
 * rounded once on store. Half the HBM bytes of the fp32 op. Pointers are `__nv_bfloat16*`. */
int ebfi_fac_forward_bf16(void *stream, const void *input, const void *kernel, void *output,
                          int batch, int channels, int height_out, int width_out, int kernel_size);
int ebfi_fac_backward_bf16(void *stream, const void *input, const void *kernel, const void *grad_output,
                           void *grad_input, void *grad_kernel,
                           int batch, int channels, int height_out, int width_out, int kernel_size,
                           void *workspace, size_t workspace_bytes);

/* fp16 storage variants: as the bf16 ones, with every tensor `__half*`. A result beyond the fp16 range is stored as
 * +-inf, as a cast to fp16 gives; NaN stays NaN. */
int ebfi_fac_forward_fp16(void *stream, const void *input, const void *kernel, void *output,
                          int batch, int channels, int height_out, int width_out, int kernel_size);
int ebfi_fac_backward_fp16(void *stream, const void *input, const void *kernel, const void *grad_output,
                           void *grad_input, void *grad_kernel,
                           int batch, int channels, int height_out, int width_out, int kernel_size,
                           void *workspace, size_t workspace_bytes);

/* ReplicationPad2d((K-1)/2) followed by FAC as one op (the KernelConv2D module, KernelConv2D.py:77-87): the
 * arguments of the entries above, except that input and grad_input are the unpadded (B, C, H, W) tensors.
 * The pad is folded into the kernels, so no padded copy is written or read. The forward and grad_kernel are
 * bit-identical to the padded entries on the replication-padded input. grad_input sums the padded cells each
 * input element is replicated to in a fixed order in fp32 (no atomics) and rounds 16-bit results once; an
 * element outside the first and last row and column is bit-identical to its padded counterpart. The backward
 * takes exactly ebfi_fac_backward_workspace_bytes(B, C, H, W, K) bytes of workspace. K = 1 is the plain op. */
int ebfi_fac_replpad_forward(void *stream, const float *input, const float *kernel, float *output,
                             int batch, int channels, int height_out, int width_out, int kernel_size);
int ebfi_fac_replpad_backward(void *stream, const float *input, const float *kernel,
                              const float *grad_output, float *grad_input, float *grad_kernel,
                              int batch, int channels, int height_out, int width_out, int kernel_size,
                              void *workspace, size_t workspace_bytes);
int ebfi_fac_replpad_forward_bf16(void *stream, const void *input, const void *kernel, void *output,
                                  int batch, int channels, int height_out, int width_out, int kernel_size);
int ebfi_fac_replpad_backward_bf16(void *stream, const void *input, const void *kernel, const void *grad_output,
                                   void *grad_input, void *grad_kernel,
                                   int batch, int channels, int height_out, int width_out, int kernel_size,
                                   void *workspace, size_t workspace_bytes);
int ebfi_fac_replpad_forward_fp16(void *stream, const void *input, const void *kernel, void *output,
                                  int batch, int channels, int height_out, int width_out, int kernel_size);
int ebfi_fac_replpad_backward_fp16(void *stream, const void *input, const void *kernel, const void *grad_output,
                                   void *grad_input, void *grad_kernel,
                                   int batch, int channels, int height_out, int width_out, int kernel_size,
                                   void *workspace, size_t workspace_bytes);

/* ---- KernelConv producer -> FAC fusion (forward; SURVEY 8f rank 1) ------------- */

/* models/Ours/model_singleframe.py:145-146,159-162 (class Modification) as ONE op:
 *   Kernel = LeakyReLU(conv3x3(cat([event_feat, frame_feat], 1), conv_weight, conv_bias, pad 1))   (B, Ce*K*K, H, W)
 *   output = KernelConv2D(K)(event_feat, Kernel)      = FAC on the ReplicationPad2d((K-1)/2)-padded event_feat
 * The (B, Ce*K*K, H, W) kernel tensor never exists in HBM. All tensors fp32 NCHW contiguous:
 *   event_feat (B, Ce, H, W); frame_feat (B, Cf, H, W); conv_weight (Ce*K*K, Ce+Cf, 3, 3); conv_bias (Ce*K*K);
 *   output (B, Ce, H, W), every element written.
 * Precision: the convolution's operands are rounded to bf16 for the tcgen05 tensor cores, accumulation and the
 * FAC contraction are fp32 (the reference's conv runs in TF32 under torch's defaults). Shapes: (Ce+Cf) % 32 == 0,
 * Ce+Cf <= 128, odd K <= 5; otherwise EBFI_ERR_UNSUPPORTED. The matching backward is ebfi_kpn_fused_backward. */
size_t ebfi_kpn_fused_workspace_bytes(int batch, int channels_event, int channels_frame, int height, int width,
                                      int kernel_size);
int ebfi_kpn_fused_forward(void *stream, const float *event_feat, const float *frame_feat,
                           const float *conv_weight, const float *conv_bias, float negative_slope,
                           float *output, int batch, int channels_event, int channels_frame,
                           int height, int width, int kernel_size, void *workspace, size_t workspace_bytes);

/* Fused backward of the same block, given grad_output = dL/doutput (B, Ce, H, W). It recomputes the conv's
 * pre-activation P = conv3x3(cat(event_feat, frame_feat)) + conv_bias on the tensor cores exactly as the forward does
 * (same bf16 operands, same accumulation order, so the same LeakyReLU branches) and writes, fp32 NCHW contiguous:
 *   grad_pre       (B, Ce*K*K, H, W)  dL/dP = G * Epad * (P > 0 ? 1 : negative_slope), every element written
 *   grad_event_fac (B, Ce, H, W)      the FAC + ReplicationPad2d part of dL/devent_feat, every element written
 *   grad_bias      (Ce*K*K)           dL/dconv_bias (sum of grad_pre over batch and pixels)
 * Neither the kernel tensor LeakyReLU(P) nor P ever exists in HBM. The caller still computes the conv's weight and
 * input gradients from grad_pre (an ordinary 3x3 pad-1 convolution backward of cat(event_feat, frame_feat)) and adds
 * the event channels of the input gradient to grad_event_fac. Deterministic: no float atomics; results are
 * bit-identical run to run on a device. Shapes, precision and error codes as ebfi_kpn_fused_forward; null pointers
 * return EBFI_ERR_INVALID before any CUDA call. The workspace size does not depend on the device (0 = unsupported). */
size_t ebfi_kpn_fused_backward_workspace_bytes(int batch, int channels_event, int channels_frame,
                                               int height, int width, int kernel_size);
int ebfi_kpn_fused_backward(void *stream, const float *event_feat, const float *frame_feat,
                            const float *conv_weight, const float *conv_bias, float negative_slope,
                            const float *grad_output, float *grad_pre, float *grad_event_fac, float *grad_bias,
                            int batch, int channels_event, int channels_frame, int height, int width,
                            int kernel_size, void *workspace, size_t workspace_bytes);

/* bf16 activation variants of the two entries above (mixed precision: bf16 activations, fp32 parameters), same
 * argument order. event_feat, frame_feat, output, grad_output and grad_pre are `__nv_bfloat16*`; conv_weight,
 * conv_bias, grad_event_fac and grad_bias stay fp32. Only the activation loads and stores change: loads widen
 * exactly, output and grad_pre are rounded once (RN) from the fp32 values the fp32 entries store, so on bf16-valued
 * inputs the results equal the fp32 entries' results rounded to bf16 (grad_event_fac, grad_bias: equal). Workspace
 * sizes are those of ebfi_kpn_fused_workspace_bytes / ebfi_kpn_fused_backward_workspace_bytes. */
int ebfi_kpn_fused_forward_bf16(void *stream, const void *event_feat, const void *frame_feat,
                                const float *conv_weight, const float *conv_bias, float negative_slope,
                                void *output, int batch, int channels_event, int channels_frame,
                                int height, int width, int kernel_size, void *workspace, size_t workspace_bytes);
int ebfi_kpn_fused_backward_bf16(void *stream, const void *event_feat, const void *frame_feat,
                                 const float *conv_weight, const float *conv_bias, float negative_slope,
                                 const void *grad_output, void *grad_pre, float *grad_event_fac, float *grad_bias,
                                 int batch, int channels_event, int channels_frame, int height, int width,
                                 int kernel_size, void *workspace, size_t workspace_bytes);

/* fp16 activation variants: the two *_bf16 entries above with `__half*` in place of `__nv_bfloat16*`, same arguments
 * and workspaces. The conv operands are rounded to bf16 as in the fp32 and bf16 entries, so on fp16-valued inputs
 * output and grad_pre equal the fp32 entries' results rounded once to fp16 (+-inf beyond the fp16 range), and
 * grad_event_fac and grad_bias are equal. */
int ebfi_kpn_fused_forward_fp16(void *stream, const void *event_feat, const void *frame_feat,
                                const float *conv_weight, const float *conv_bias, float negative_slope,
                                void *output, int batch, int channels_event, int channels_frame,
                                int height, int width, int kernel_size, void *workspace, size_t workspace_bytes);
int ebfi_kpn_fused_backward_fp16(void *stream, const void *event_feat, const void *frame_feat,
                                 const float *conv_weight, const float *conv_bias, float negative_slope,
                                 const void *grad_output, void *grad_pre, float *grad_event_fac, float *grad_bias,
                                 int batch, int channels_event, int channels_frame, int height, int width,
                                 int kernel_size, void *workspace, size_t workspace_bytes);

/* ---- event encoders --------------------------------------------------------- */

/* Coordinate / timestamp arrays may be fp32 or fp64, like the tensors the
 * datasets build (dataloader/h5dataset.py:327-349 yields fp64). */
#define EBFI_F32 0
#define EBFI_F64 1

/* events_to_image (dataloader/encodings.py:243-268).
 *   img[(long)ys[i], (long)xs[i]] += ps[i]   for in-range events;
 * out-of-range events get xs=ys=ps=0 written back IN PLACE when `write_back`
 * is non-zero (that is what the reference does to its arguments, :254-256).
 * `img` (H, W) fp32 is ACCUMULATED into; the caller zero-fills it. */
int ebfi_events_to_image(void *stream, void *xs, void *ys, float *ps, int coord_dtype,
                         int64_t n_events, int height, int width,
                         float *img, int write_back);

/* events_to_mask (encodings.py:353-377): img[...] = |ps| with accumulate=False, i.e.
 * the LAST event of a pixel wins (out-of-range events write 0 at pixel (0,0), like the
 * reference). `last_index_scratch` is (H*W) int64 device scratch. */
int ebfi_events_to_mask(void *stream, void *xs, void *ys, float *ps, int coord_dtype,
                        int64_t n_events, int height, int width,
                        float *img, int64_t *last_index_scratch, int write_back);

/* events_to_voxel (encodings.py:271-286): temporal-bilinear voxel grid.
 *   t = ts[i] * (num_bins-1);  voxel[b] += ps[i] * max(0, 1 - |t - b|)
 * xs, ys, ts share `dtype`; ps is fp32. Out-of-range events follow the
 * reference's in-place rule: they are dropped from bin 0 and land on pixel
 * (0,0) for bins >= 1 (a side effect of :254-256 being applied once per bin).
 * voxel : (num_bins, H, W) fp32, accumulated into (caller zero-fills). */
int ebfi_events_to_voxel(void *stream, void *xs, void *ys, const void *ts, const float *ps,
                         int dtype, int64_t n_events, int num_bins, int height, int width,
                         float *voxel, int write_back);

/* flag[0] <- (sum of the n timestamps == 0) ? 1 : 0, on the device, in a fixed summation order: the `ts.sum() == 0`
 * half of events_to_stack's early-out (encodings.py:319-320) as the `skip_flag` of ebfi_events_to_stack.
 * scratch: EBFI_EVENTS_SUM_SCRATCH_BYTES of 8-byte aligned device memory. */
#define EBFI_EVENTS_SUM_SCRATCH_BYTES 4800
int ebfi_events_ts_sum_is_zero(void *stream, const void *ts, int dtype, int64_t n_events, void *scratch,
                               unsigned char *flag);

/* events_to_stack (encodings.py:307-350): per-bin positive / negative counts.
 * The bin boundaries are found on the device with the reference's own binary
 * search (encodings.py:77-99), so boundary-equal timestamps are counted in both
 * adjacent bins exactly like the reference does.
 * stack : (2, num_bins, H, W) fp32, accumulated into (caller zero-fills).
 * bounds : (2*num_bins) int64 scratch, receives [beg_0,end_0,beg_1,end_1,...].
 * skip_flag : optional 1-byte DEVICE flag; non-zero makes the call a no-op. It carries the
 *   reference's early-out `ts.sum() == 0` (:319-320) without a device->host synchronisation
 *   (the `len <= 3` half is decided on the host). */
int ebfi_events_to_stack(void *stream, void *xs, void *ys, const void *ts, const float *ps,
                         int dtype, int64_t n_events, int num_bins, int height, int width,
                         float *stack, int64_t *bounds, int write_back,
                         const unsigned char *skip_flag);

/* The datasets' whole event path in one call: GetEventsIndex + events_to_stack
 * (dataloader/h5dataset.py:327-349) on the ON-DISK dtypes of the HDF5 files
 * (generate_dataset/tools/event_packagers.py:128-131): xs, ys int16; ts float64
 * seconds, non-decreasing; ps int8. The normalisation
 * `ts = (ts - ts[0]) / (ts[-1] - ts[0] + 1e-6)` (h5dataset.py:335) is evaluated in
 * float64 on access, `ps.float()` (:349) in registers; nothing is converted or
 * written back, 13 bytes are read per event instead of 32 (4 x float64).
 * n_events <= 3 (which includes the reference's empty-slice substitute, :332-333) and
 * all-equal timestamps leave `stack` untouched = the zeros early-out (encodings.py:319-320).
 * stack : fp32, accumulated into (caller zero-fills); (2, num_bins, H, W) like the
 *   reference, or (num_bins, 2, H, W) — what the datasets' `.transpose(0, 1)` yields —
 *   when bins_major != 0.
 * bounds : (2*num_bins) int64 scratch. */
int ebfi_events_raw_to_stack(void *stream, const int16_t *xs, const int16_t *ys, const double *ts,
                             const int8_t *ps, int64_t n_events, int num_bins, int height, int width,
                             float *stack, int64_t *bounds, int bins_major);

/* ---- per-frame maps the model computes on the host (SURVEY 8f rank 4) ---------- */

/* Frame2Lap (myutils/utils.py:34-49; model_singleframe.py:311-326): frames (B, 3, H, W) fp32 in [0, 1] ->
 * (im*255).astype(uint8) -> cv2.cvtColor(BGR2GRAY) -> cv2.Laplacian(CV_64F) -> lap (B, 1, H, W) fp32.
 * Integer arithmetic, bit-identical to OpenCV >= 4 (15-bit gray coefficients, BORDER_REFLECT_101). */
int ebfi_frame_to_lap(void *stream, const float *frames, float *lap, int batch, int height, int width);

/* Frame2DCP (myutils/utils.py:15-31): dark channel = min over the 3 channels, then cv2.erode with a
 * window x window rectangle (35 in the reference) = window minimum, pixels outside the image ignored.
 * dark (B, 1, H, W); scratch (B, H, W) fp32. Bit-identical to OpenCV. */
int ebfi_frame_to_dcp(void *stream, const float *frames, float *dark, float *scratch,
                      int batch, int height, int width, int window);

/* ---- data-parallel weight-gradient all-reduce over NVLink peer memory -------------------------------------------
 * SURVEY §8e: batch-sharded training has exactly one exchange on this path, the sum of DCNv2's grad_weight /
 * grad_bias over the ranks (dcn_v2_cuda.cu:203-208 produces them per rank; the reference never reduces them,
 * train_ours.py:250-272 runs every backward under no_sync). Instead of a separate NCCL call the reduction is done by
 * the kernel that produces the gradients: every rank maps one symmetric allocation of each peer (torch symmetric
 * memory, cudaIpc, ... — the host's plumbing), the kernel pushes its local sums into every peer's allocation and raises
 * a flag there; the completing kernel adds the values it received in rank order (identical bits on every rank and run
 * to run) from local memory only. See csrc/dp_comm.cuh.
 *
 * peer_base[q]: this process's mapping of rank q's allocation (peer_base[rank] = the local one), 256-byte aligned,
 * `bytes` >= ebfi_dp_comm_bytes(n) each and THE SAME VALUE ON EVERY RANK (the slot layout derives from it), zero-filled
 * ONCE before the first call (and a host barrier after the fill).
 * Every rank must issue the same sequence of calls on the communicator. world <= 8; world == 1 is a plain copy. */
typedef struct ebfi_dp_comm {
    int world, rank;
    void *peer_base[8];
    size_t bytes;
} ebfi_dp_comm;

/* Symmetric bytes per rank for all-reducing up to n_floats values per call. */
size_t ebfi_dp_comm_bytes(size_t n_floats);

/* In place: a[0, na) and b[0, nb) become the sums over all ranks (one kernel, no NCCL). */
int ebfi_dp_allreduce_sum(void *stream, const ebfi_dp_comm *comm, float *a, size_t na, float *b, size_t nb);

/* The same exchange in two halves, so that the NVLink latency and the skew between the ranks hide behind the work in
 * between: publish stores the local values into every peer's symmetric buffer and signals the peers (does not wait);
 * complete waits for every peer's values of the LAST publish and writes the rank-ordered sums into a / b (same sizes).
 * At most one publish may be outstanding per communicator. */
int ebfi_dp_publish(void *stream, const ebfi_dp_comm *comm, const float *a, size_t na, const float *b, size_t nb);
int ebfi_dp_complete(void *stream, const ebfi_dp_comm *comm, float *a, size_t na, float *b, size_t nb);

/* ebfi_dcnv2_backward whose grad_weight / grad_bias are the sums over all ranks of `comm`; on the tensor-core box path
 * the exchange is fused into the kernel that reduces the per-CTA partials. The other three gradients are per rank.
 * defer != 0: the kernel only publishes — grad_weight / grad_bias hold this rank's sums until the caller runs
 * ebfi_dp_complete(stream, comm, grad_weight, Cout*C*kh*kw, grad_bias, Cout) (e.g. right before the optimizer step). */
int ebfi_dcnv2_backward_dp(void *stream, const ebfi_dcn_geom *g,
                           const float *input, const float *weight, const float *bias,
                           const float *offset, const float *mask, const float *grad_output,
                           float *grad_input, float *grad_offset, float *grad_mask,
                           float *grad_weight, float *grad_bias,
                           void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer);
/* The same with bf16 activations, as ebfi_dcnv2_backward_bf16 (EBFI_ERR_UNSUPPORTED: take ebfi_dcnv2_backward_dp on
 * widened copies). grad_weight / grad_bias are fp32, exchanged exactly as above. */
int ebfi_dcnv2_backward_dp_bf16(void *stream, const ebfi_dcn_geom *g,
                                const void *input, const float *weight, const float *bias,
                                const void *offset, const void *mask, const void *grad_output,
                                void *grad_input, void *grad_offset, void *grad_mask,
                                float *grad_weight, float *grad_bias,
                                void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer);
/* The same with fp16 activations, as ebfi_dcnv2_backward_fp16. */
int ebfi_dcnv2_backward_dp_fp16(void *stream, const ebfi_dcn_geom *g,
                                const void *input, const float *weight, const float *bias,
                                const void *offset, const void *mask, const void *grad_output,
                                void *grad_input, void *grad_offset, void *grad_mask,
                                float *grad_weight, float *grad_bias,
                                void *workspace, size_t workspace_bytes, const ebfi_dp_comm *comm, int defer);

#ifdef __cplusplus
}
#endif
#endif /* EBFI_B200_H_ */
