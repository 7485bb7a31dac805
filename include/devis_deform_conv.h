/*
 * devis_deform_conv.h -- C ABI of the modulated deformable convolution kernels (same library, libdevis_msda.so).
 *
 * DeVIS's mask head evaluates every 3x3 layer with torchvision.ops.deform_conv2d
 * (/root/reference/src/models/deformable_segmentation.py:244-267 ModulatedDeformableConv2d, :323-380 MaskHeadConv;
 * SURVEY.md section 8f-3).  torchvision is a third-party dependency of the reference (pinned at 0.12,
 * docs/INSTALL.md:9); its operator is vision::ops::deform_conv2d (torchvision/csrc/ops/deform_conv2d.cpp) with the CUDA
 * kernels deformable_im2col / deformable_col2im / deformable_col2im_coord (torchvision/csrc/ops/cuda/
 * deform_conv2d_kernel.cu).  The two entry points below replace those three kernels; the matrix products with the
 * convolution weights stay in cuBLAS on the caller's side (torchvision: at::addmm / at::bmm), exactly as the attention
 * library leaves the projection GEMMs to cuBLAS.
 *
 * Layouts.  `input` / `grad_input` are CHANNELS-LAST (N, H, W, C) -- a torch tensor in torch.channels_last memory
 * format, or x.permute(0, 2, 3, 1).contiguous().  `offset` (N, 2*kh*kw, Ho, Wo) and `mask` (N, kh*kw, Ho, Wo) keep
 * torchvision's layout: channel 2k is the row offset and 2k+1 the column offset of kernel position k = ky*kw + kx;
 * mask may be NULL (plain deformable convolution).  Columns: cols[((n*Ho + ho)*Wo + wo) * kh*kw*C + k*C + c], i.e. a
 * row-major (N*Ho*Wo, kh*kw*C) matrix; multiply it with weight.permute(0, 2, 3, 1).reshape(Cout, kh*kw*C)^T.
 * groups = 1 and offset_groups = 1 only.  dtype: DEVIS_MSDA_F32 or DEVIS_MSDA_F64.  Asynchronous on `stream`,
 * no allocation, no synchronisation; returns DEVIS_MSDA_OK or a DEVIS_MSDA_ERR_* code (devis_msda.h).
 */
#ifndef DEVIS_DEFORM_CONV_H_
#define DEVIS_DEFORM_CONV_H_

#include "devis_msda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* cols = modulated deformable im2col(input): cols[pixel, k, c] = mask[k] * bilinear(input[n, :, :, c], sample point k),
 * zero padding (torchvision bilinear_interpolate).  Fully written. */
int devis_dcn_im2col(const void *input_nhwc, const void *offset, const void *mask, void *cols, int batch, int height,
                     int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w, int stride_h,
                     int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int dtype, void *stream);

/* Backward of the gather given grad_cols (same layout as cols):
 *   grad_input_nhwc  like input  -- zero-filled by this call, then accumulated (may be NULL: not needed)
 *   grad_offset      like offset -- fully written
 *   grad_mask        like mask   -- fully written (NULL iff mask is NULL) */
int devis_dcn_col2im(const void *input_nhwc, const void *offset, const void *mask, const void *grad_cols,
                     void *grad_input_nhwc, void *grad_offset, void *grad_mask, int batch, int height, int width,
                     int channels, int out_h, int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w,
                     int pad_h, int pad_w, int dil_h, int dil_w, int dtype, void *stream);

/* ---- deterministic grad_input -----------------------------------------------------------------------------------------
 * The default backward scatters grad_input with floating-point atomics: its last bits change from run to run.  The _ex
 * forms take backward flags (devis_msda.h); with DEVIS_MSDA_FLAG_DETERMINISTIC (float32 only) every grad_input
 * contribution is converted exactly to 64-bit fixed point and summed with integer atomics, so grad_input is
 * bit-identical run to run on a device.  Its resolution is 2^-36 of a bound of the largest possible contribution:
 * max|grad_cols| * max|mask| for col2im, max|grad_out| * max|mask| * out_channels * max|weight| for the fused form
 * (max|mask| = 1 without a mask); the bound and the scale stay on the device (no synchronisation, graph capture is legal).
 * grad_offset / grad_mask are written once per element in every mode and are deterministic anyway.
 * The flag needs a workspace of devis_dcn_backward_workspace_bytes(batch, ...) bytes (8 per grad_input element + 16; 0
 * without the flag).  Checked on the host before any CUDA call: float64 with the flag -> DEVIS_MSDA_ERR_UNSUPPORTED;
 * out_h * out_w * kernel_h * kernel_w >= 2^26 (the int64 sum could overflow) -> DEVIS_MSDA_ERR_TOO_LARGE; a missing or
 * short workspace -> DEVIS_MSDA_ERR_WORKSPACE.  The flag is ignored when grad_input_nhwc is NULL.
 * devis_dcn_col2im / devis_dcn_fused_backward are the _ex forms with flags = 0. */
size_t devis_dcn_backward_workspace_bytes(int batch, int height, int width, int channels, unsigned flags);
int devis_dcn_col2im_ex(const void *input_nhwc, const void *offset, const void *mask, const void *grad_cols,
                        void *grad_input_nhwc, void *grad_offset, void *grad_mask, int batch, int height, int width,
                        int channels, int out_h, int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w,
                        int pad_h, int pad_w, int dil_h, int dil_w, int dtype, unsigned flags, void *workspace,
                        size_t workspace_bytes, void *stream);


/* ---- fused form: gather + contraction with the weights in one kernel; the column matrix is never written ------------
 * For layers with few output channels (the high-resolution half of the mask head) im2col + GEMM is bound by writing and
 * re-reading columns 9x the size of the input.  The fused kernels read input, offsets, mask once and write the output
 * once.  float only; channels % 4 == 0.
 *
 * devis_dcn_fused_form: bit 0 set = devis_dcn_fused_forward serves the layer, bit 1 set = devis_dcn_fused_backward does
 * (0: use devis_dcn_im2col / devis_dcn_col2im + GEMM).  Forward: out_channels in {1, 2, 4, 8, 16} (lane-group kernel) or
 * a multiple of 16 up to 64 with kh*kw*channels <= 1024 (weights held in the constant bank, 16 output channels per
 * launch; calls from different streams are ordered against each other on the device because they share that bank).
 * Backward (data gradients): out_channels in {1, 2, 4, 8, 16}.
 * devis_dcn_pack_weight: rearranges torchvision's weight (out_channels, channels, kh, kw) into the layouts the fused
 * kernels read (devis_dcn_packed_weight_elems floats; deform_conv.cuh "PACKED WEIGHTS").
 * devis_dcn_fused_forward: out[(n*Ho + ho)*Wo + wo][co] (channels-last, (N, Ho, Wo, out_channels)) = bias[co] +
 *   sum_{k, c} weight[co][c][k] * mask[k] * bilinear(input[n, :, :, c], sample point k); bias may be NULL.
 * devis_dcn_fused_backward: data gradients from grad_out (channels-last like out) without materialising grad_cols:
 *   grad_input_nhwc (zero-filled here, then accumulated; may be NULL), grad_offset, grad_mask (fully written).
 *   The weight gradient is cols^T x grad_out: devis_dcn_im2col + GEMM on the caller's side. */
int devis_dcn_fused_form(int channels, int out_channels, int kernel_h, int kernel_w, int dtype);
size_t devis_dcn_packed_weight_elems(int channels, int out_channels, int kernel_h, int kernel_w);
int devis_dcn_pack_weight(const void *weight_oihw, void *packed, int channels, int out_channels, int kernel_h,
                          int kernel_w, void *stream);
int devis_dcn_fused_forward(const void *input_nhwc, const void *offset, const void *mask, const void *packed_weight,
                            const void *bias, void *out_nhwc, int batch, int height, int width, int channels, int out_h,
                            int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                            int dil_h, int dil_w, int out_channels, void *stream);
int devis_dcn_fused_backward(const void *input_nhwc, const void *offset, const void *mask, const void *packed_weight,
                             const void *grad_out_nhwc, void *grad_input_nhwc, void *grad_offset, void *grad_mask,
                             int batch, int height, int width, int channels, int out_h, int out_w, int kernel_h,
                             int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                             int out_channels, void *stream);
int devis_dcn_fused_backward_ex(const void *input_nhwc, const void *offset, const void *mask, const void *packed_weight,
                                const void *grad_out_nhwc, void *grad_input_nhwc, void *grad_offset, void *grad_mask,
                                int batch, int height, int width, int channels, int out_h, int out_w, int kernel_h,
                                int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                                int out_channels, unsigned flags, void *workspace, size_t workspace_bytes, void *stream);

/* devis_dcn_weight_grad: the weight gradient of a narrow layer without a column matrix,
 *   grad_weight[co][k][c] = sum over (n, ho, wo) of mask * bilinear(input[n, .., c]) * grad_out_nhwc[n, ho, wo, co]
 * i.e. (out_channels, kernel_h * kernel_w, channels) row-major, zero-filled here; permute to (Cout, C, kh, kw) on the
 * caller's side.  Replaces torchvision's deformable_im2col + at::addmm pair of the backward
 * (torchvision/csrc/ops/cuda/deform_conv2d_kernel.cu, backward_gradient_parameters) for float32 layers with
 * channels in {16, 32} and out_channels in {1, 2, 4, 8, 16}: devis_dcn_wgrad_supported says so (1 / 0). */
int devis_dcn_wgrad_supported(int channels, int out_channels, int kernel_h, int kernel_w, int dtype);
int devis_dcn_weight_grad(const void *input_nhwc, const void *offset, const void *mask, const void *grad_out_nhwc,
                          void *grad_weight, int batch, int height, int width, int channels, int out_h, int out_w,
                          int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h,
                          int dil_w, int out_channels, void *stream);

/* ---- tensor-core form: the forward of the WIDE layers as an implicit GEMM on tcgen05 (dcn_igemm.cuh) -------------------
 * Replaces deformable_im2col + at::addmm (torchvision/csrc/ops/cuda/deform_conv2d_kernel.cu, forward) for float32 layers
 * with channels % 8 == 0, out_channels % 4 == 0 and out_channels <= 512 -- in DeVIS's mask head the 264 -> 264,
 * 264 -> 128 and 136 -> 64 layers (deformable_segmentation.py:323-380), whose contraction dominates and which round 1 ran
 * as im2col + cuBLAS fp32.  No column matrix: a thread block gathers and interpolates 128 output pixels x 32 channels
 * at a time into shared memory, the weights stream in pre-packed, tcgen05.mma.kind::tf32 accumulates in tensor memory.
 *   precision  DEVIS_DCN_PRECISION_3XTF32 (default): operands split hi + lo, three TF32 products per term, fp32-grade
 *              result (<= 1e-5 against the float64 fixtures); DEVIS_DCN_PRECISION_TF32: one TF32 pass, for callers that
 *              have torch.backends.cuda.matmul.allow_tf32 on (torchvision's addmm honours that switch as well).
 * devis_dcn_igemm_pack_weight: torchvision's weight (out_channels, channels, kh, kw) -> the kernel's swizzled hi / lo
 * slabs (devis_dcn_igemm_packed_weight_elems floats).  out: (N, Ho, Wo, out_channels) channels-last, fully written. */
#define DEVIS_DCN_PRECISION_3XTF32 0
#define DEVIS_DCN_PRECISION_TF32 1
int devis_dcn_igemm_supported(int channels, int out_channels, int kernel_h, int kernel_w, int dtype);
size_t devis_dcn_igemm_packed_weight_elems(int channels, int out_channels, int kernel_h, int kernel_w);
int devis_dcn_igemm_pack_weight(const void *weight_oihw, void *packed, int channels, int out_channels, int kernel_h,
                                int kernel_w, void *stream);
int devis_dcn_igemm_forward(const void *input_nhwc, const void *offset, const void *mask, const void *packed_weight,
                            const void *bias, void *out_nhwc, int batch, int height, int width, int channels, int out_h,
                            int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                            int dil_h, int dil_w, int out_channels, int precision, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DEVIS_DEFORM_CONV_H_ */
