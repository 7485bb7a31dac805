/*
 * devis_msda.h -- C ABI of the B200-native (sm_100a) multi-scale deformable attention library.
 *
 * This is the drop-in boundary for DeVIS's one native component.  The reference exposes
 * two functions through pybind (paths relative to /root/reference/src/models/ops/src):
 *
 *     vision.cpp:14   ms_deform_attn_forward   -> ms_deform_attn.h:20-39  -> cuda/ms_deform_attn_cuda.cu:20-80
 *     vision.cpp:15   ms_deform_attn_backward  -> ms_deform_attn.h:41-61  -> cuda/ms_deform_attn_cuda.cu:83-153
 *
 * devis_msda_forward / devis_msda_backward below are what those two bind to: same operands,
 * same layouts, same semantics; plain pointers and sizes, no torch types.  The caller owns every
 * buffer (the reference allocates its outputs with at::zeros inside the C++ host code,
 * ms_deform_attn_cuda.cu:54,121-123; here the binding allocates and this library fills).
 *
 * devis_tmsda_forward / devis_tmsda_backward are the whole-clip temporal form of the same op: one
 * call replaces the per-frame Python loop of TemporalMSDeformAttn{Encoder,Decoder}.forward
 * (modules/ms_deform_attn.py:325-364, 367-404, 435-460 -- 2*T op calls plus T gather copies of
 * value[temporal_frames]) and reads value (T,S,M,D) in place through a frame table.
 *
 * All pointers are DEVICE pointers unless the parameter name ends in _host.  All tensors are dense
 * row-major ("contiguous") in the shapes given.  Every call is asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream) and never synchronises.
 * Functions return DEVIS_MSDA_OK or a negative error code; nothing is printed.
 * (Deliberate divergence: the reference only printf()s kernel launch failures,
 * cuda/ms_deform_im2col_cuda.cuh:948-952,1321-1325.)
 */
#ifndef DEVIS_MSDA_H_
#define DEVIS_MSDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DEVIS_MSDA_ABI_VERSION 5

/* element types of value / output / grad_output */
#define DEVIS_MSDA_F32 0  /* value, loc, weights, outputs and all gradients float            */
#define DEVIS_MSDA_F64 1  /* everything double (the reference's gradcheck type, test.py:74)   */
#define DEVIS_MSDA_BF16 2 /* extension: value/output/grad_output bf16; sampling locations,    */
                          /* attention weights and ALL gradients (incl. grad_value) float     */
#define DEVIS_MSDA_F16 3  /* extension: value/output/grad_output IEEE half (torch.autocast's  */
                          /* default); everything else float, exactly as for DEVIS_MSDA_BF16 */

/* error codes */
#define DEVIS_MSDA_OK 0
#define DEVIS_MSDA_ERR_NULL_POINTER (-1)
#define DEVIS_MSDA_ERR_BAD_SHAPE (-2)      /* a dimension is negative, or zero where that is meaningless */
#define DEVIS_MSDA_ERR_BAD_DTYPE (-3)
#define DEVIS_MSDA_ERR_BATCH_STEP (-4)     /* batch % min(batch, im2col_step) != 0, ms_deform_attn_cuda.cu:50-52 */
#define DEVIS_MSDA_ERR_TOO_LARGE (-5)      /* a tensor exceeds the 32-bit element indexing the kernels use */
#define DEVIS_MSDA_ERR_WORKSPACE (-6)      /* workspace missing or smaller than *_workspace_bytes() */
#define DEVIS_MSDA_ERR_CUDA (-7)           /* a CUDA runtime call / launch failed; see devis_msda_last_cuda_error */
#define DEVIS_MSDA_ERR_UNSUPPORTED (-8)    /* valid request this build has no kernel for */
#define DEVIS_MSDA_ERR_BAD_FRAME_TABLE (-9)

/* backward flags */
#define DEVIS_MSDA_FLAG_DETERMINISTIC 1u   /* bit-reproducible grad_value (no floating-point atomics) */
#define DEVIS_MSDA_FLAG_NO_GRAD_VALUE 2u   /* skip grad_value (value does not require grad)            */
#define DEVIS_MSDA_FLAG_BF16_GRAD_VALUE 4u /* DEVIS_MSDA_BF16 only, channels 16 or 32, not with DETERMINISTIC: grad_value is a  */
                                           /* bf16 tensor like value, accumulated with packed bf16 reductions (every partial  */
                                           /* sum rounds to bf16, like PyTorch's bf16 atomicAdd scatters); halves the bytes   */
                                           /* the scatter moves.  Default (flag clear): float grad_value, float accumulation. */
                                           /* With DEVIS_MSDA_F16: DEVIS_MSDA_ERR_UNSUPPORTED (fp16's range makes rounding    */
                                           /* every partial sum unsafe).                                                      */

int devis_msda_abi_version(void);
const char *devis_msda_error_string(int code);
/* cudaError_t of the most recent DEVIS_MSDA_ERR_CUDA on the calling thread (0 if none) */
int devis_msda_last_cuda_error(void);
/* number of kernels this library has launched in this process (all threads) */
uint64_t devis_msda_launch_count(void);
/* the same count per kernel family: lets a caller (and the parity tests) verify WHICH kernel served a call -- e.g.
 * that the fused-prologue kernels ran and the module did not silently take the unfused path */
#define DEVIS_MSDA_KERNEL_FWD_GROUPED 0   /* msda_fwd / msda_fwdc / msda_fwd8 (D = 16 | 32 lane-group kernels) */
#define DEVIS_MSDA_KERNEL_FWD_GENERIC 1   /* msda_fwd_generic (any D, fp64) */
#define DEVIS_MSDA_KERNEL_BWD_GROUPED 2   /* msda_bwd */
#define DEVIS_MSDA_KERNEL_BWD_GENERIC 3   /* msda_bwd_generic */
#define DEVIS_MSDA_KERNEL_FUSED_FWD 4     /* tmsda_fused_fwd / tmsda_fused_fwd8 (prologue fused in) */
#define DEVIS_MSDA_KERNEL_FUSED_BWD 5     /* tmsda_fused_bwd */
#define DEVIS_MSDA_KERNEL_BWD_SORTED 6    /* msda_bwds (deterministic, encoder form) */
#define DEVIS_MSDA_KERNEL_AUX 7           /* absmax / fixed-point finalize helpers */
#define DEVIS_MSDA_KERNEL_DCN 8           /* include/devis_deform_conv.h kernels (CUDA-core forms, helpers) */
#define DEVIS_MSDA_KERNEL_DCN_IGEMM 9     /* dcn_igemm_fwd (tcgen05 implicit GEMM) */
#define DEVIS_MSDA_KERNEL_FAMILIES 10
uint64_t devis_msda_kernel_launches(int family);
/* Developer knobs of the benchmarks (launch shapes, kernel A/B selection).  They are inert in a product process:
 * unless the process was started with the environment variable DEVIS_MSDA_TUNING=1 this returns
 * DEVIS_MSDA_ERR_UNSUPPORTED and every key stays at 0 = built-in heuristic.
 * key 0: forward threads per block, 1: forward queries per lane group,
 * key 2: backward threads per block, 3: backward queries per lane group,
 * keys 4, 5: unused since round 2 (they chose between forward kernels that no longer exist),
 * key 6: 1 = deterministic mode uses the direct 64-bit scatter instead of the sorted kernel,
 * key 7: sorted kernel's window margin in pixels (0 = 6), key 9: its first level with a window + 1. */
int devis_msda_set_tuning(int key, int value);

/*
 * Forward.  Replaces ms_deform_attn_forward (vision.cpp:14).
 *   value              (batch, spatial_size, num_heads, channels)
 *   spatial_shapes     (num_levels, 2) int64, rows (H_l, W_l)            -- read on the device
 *   level_start_index  (num_levels)    int64, first row of level l in spatial_size
 *   sampling_loc       (batch, num_query, num_heads, num_levels, num_point, 2), (x, y) in [0,1]
 *   attn_weight        (batch, num_query, num_heads, num_levels, num_point)
 *   output             (batch, num_query, num_heads*channels)            -- fully written
 * im2col_step only has to satisfy the reference's precondition; the batch is never chunked here.
 */
int devis_msda_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                       const void *sampling_loc, const void *attn_weight, void *output, int batch,
                       int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                       int num_point, int im2col_step, int dtype, void *stream);

/*
 * Backward.  Replaces ms_deform_attn_backward (vision.cpp:15).
 *   grad_output        (batch, num_query, num_heads*channels)
 *   grad_value         like value (float for DEVIS_MSDA_BF16 / F16) -- zero-filled by this call, then accumulated
 *   grad_sampling_loc  like sampling_loc                        -- fully written
 *   grad_attn_weight   like attn_weight                         -- fully written
 * flags: DEVIS_MSDA_FLAG_*; the deterministic mode needs a workspace of
 * devis_msda_backward_workspace_bytes() bytes (0 for the default mode).
 */
size_t devis_msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels,
                                           int num_levels, int num_query, int num_point, int dtype,
                                           unsigned flags);
int devis_msda_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                        const void *sampling_loc, const void *attn_weight, const void *grad_output,
                        void *grad_value, void *grad_sampling_loc, void *grad_attn_weight, int batch,
                        int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                        int num_point, int im2col_step, int dtype, unsigned flags, void *workspace,
                        size_t workspace_bytes, void *stream);

/*
 * Whole-clip temporal forward.  Replaces, in one launch, the T x (current call + gather copy +
 * temporal call + add) sequence of modules/ms_deform_attn.py:435-460 (encoder) and :325-404 (decoder).
 *   value            (num_frames, spatial_size, num_heads, channels)   -- value_proj output, read in place
 *   spatial_shapes_host, level_start_index_host   HOST int64 arrays for ONE frame (num_levels rows);
 *                    devis_transformer.py:97,118 builds the repeated temporal copies on the host anyway
 *   frame_table_host HOST int32 (num_frames, t_window): frame_table[t][j] = temporal_offsets[t][j] + t,
 *                    the frame that temporal slot j of query frame t samples (ms_deform_attn.py:339,445)
 *   loc_curr         (num_frames, num_query, num_heads, num_levels, n_curr_points, 2)
 *   aw_curr          (num_frames, num_query, num_heads, num_levels, n_curr_points)
 *   loc_temporal     (num_frames, num_query, num_heads, t_window*num_levels, n_temporal_points, 2)
 *   aw_temporal      (num_frames, num_query, num_heads, t_window*num_levels, n_temporal_points)
 *                    temporal level axis is frame-slot-major, level-minor (ms_deform_attn.py:232-238)
 *   output           (num_frames, num_query, num_heads*channels) = current + temporal (ms_deform_attn.py:459)
 *   query_order      optional DEVICE int32 (num_query): a permutation of the query indices of one frame.
 *                    Queries that are consecutive in this order share a thread block, so an order that
 *                    walks the encoder's pixel grid in 2-D tiles keeps each block's taps in one
 *                    neighbourhood of value (cache locality only -- results do not depend on it).  NULL = identity.
 */
int devis_tmsda_forward(const void *value, const int64_t *spatial_shapes_host,
                        const int64_t *level_start_index_host, const int32_t *frame_table_host,
                        const void *loc_curr, const void *aw_curr, const void *loc_temporal,
                        const void *aw_temporal, void *output, const int32_t *query_order, int num_frames,
                        int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                        int n_curr_points, int n_temporal_points, int t_window, int dtype, void *stream);

size_t devis_tmsda_backward_workspace_bytes(int num_frames, int spatial_size, int num_heads, int channels,
                                            int num_levels, int num_query, int n_curr_points,
                                            int n_temporal_points, int t_window, int dtype, unsigned flags);
int devis_tmsda_backward(const void *value, const int64_t *spatial_shapes_host,
                         const int64_t *level_start_index_host, const int32_t *frame_table_host,
                         const void *loc_curr, const void *aw_curr, const void *loc_temporal,
                         const void *aw_temporal, const void *grad_output, void *grad_value,
                         void *grad_loc_curr, void *grad_aw_curr, void *grad_loc_temporal,
                         void *grad_aw_temporal, const int32_t *query_order, int num_frames, int spatial_size, int num_heads,
                         int channels, int num_levels, int num_query, int n_curr_points,
                         int n_temporal_points, int t_window, int dtype, unsigned flags, void *workspace,
                         size_t workspace_bytes, void *stream);

/*
 * Whole-clip temporal attention with the prologue fused in.  Replaces, besides the per-frame op calls, the elementwise
 * chain that turns the Linear outputs into op operands: the cat + joint softmax over all K = L*Pc + Wt*L*Pt taps
 * (modules/ms_deform_attn.py:240-260) and the sampling-location arithmetic of the encoder (:437-439, :447-452) and of
 * the decoder (:320-404).
 *   ref            (num_frames, num_query, num_levels, ref_dim) float   reference points (x, y) or boxes (x, y, w, h)
 *   off_curr       (num_frames, num_query, num_heads, num_levels, n_curr_points, 2) float      raw sampling_offsets output
 *   logit_curr     (num_frames, num_query, num_heads, num_levels*n_curr_points) float           raw attention_weights output
 *   off_temporal   (num_frames, num_query, num_heads, t_window*num_levels, n_temporal_points, 2) float
 *   logit_temporal (num_frames, num_query, num_heads, t_window*num_levels*n_temporal_points) float
 *   ref_dim 2:  loc = ref + off / (W_level, H_level)                    (:437-439 encoder, :327-330 decoder layer 0)
 *   ref_dim 4:  loc = ref.xy + off / n_points * ref.wh * 0.5            (:369-371, :390-394 decoder with box refinement)
 *   temporal_ref_mode   the reference point a TEMPORAL tap of (frame t, query q, level l, temporal slot j) starts from:
 *       DEVIS_TMSDA_TREF_LEVEL0  ref[t][q][0]                       encoder (:447)
 *       DEVIS_TMSDA_TREF_OWN     ref[t][q][l]                       decoder, dec_instance_aware_att off (:346-347)
 *       DEVIS_TMSDA_TREF_SAMPLED ref[frame_table[t][j]][q][l]       decoder, instance aware (:342-344)
 *   loc_*_out / aw_*_out   optional (NULL = skip): the sampling locations and softmax weights the kernel computed, laid
 *       out like devis_tmsda_forward's operands -- what TemporalMSDeformAttnDecoder.forward returns next to its output
 *       (:414, consumed by visualize_att_maps.py:162-165)
 *   grad_ref       optional (NULL = skip): d/d(ref), like ref; zero-filled by the call, accumulated with float atomics
 * value / output / grad_output: DEVIS_MSDA_F32, DEVIS_MSDA_BF16 or DEVIS_MSDA_F16; channels must be 32 and the point counts multiples of
 * 4 (else DEVIS_MSDA_ERR_UNSUPPORTED and the caller uses devis_tmsda_forward on materialised operands).  The backward
 * writes d/d(off_*) and d/d(logit_*) directly; grad_value (float) is zero-filled by the call; flags:
 * DEVIS_MSDA_FLAG_NO_GRAD_VALUE, DEVIS_MSDA_FLAG_BF16_GRAD_VALUE, DEVIS_MSDA_FLAG_DETERMINISTIC (round 2: grad_value
 * through exact 64-bit fixed point in `workspace` of devis_tmsda_fused_backward_workspace_bytes, bit-identical run to run;
 * with grad_ref or BF16_GRAD_VALUE -> DEVIS_MSDA_ERR_UNSUPPORTED).  workspace may be NULL when the byte count is 0.
 */
#define DEVIS_TMSDA_TREF_LEVEL0 0
#define DEVIS_TMSDA_TREF_OWN 1
#define DEVIS_TMSDA_TREF_SAMPLED 2
int devis_tmsda_fused_forward(const void *value, const int64_t *spatial_shapes_host,
                              const int64_t *level_start_index_host, const int32_t *frame_table_host,
                              const void *ref, const void *off_curr, const void *logit_curr,
                              const void *off_temporal, const void *logit_temporal, void *output,
                              void *loc_curr_out, void *aw_curr_out, void *loc_temporal_out, void *aw_temporal_out,
                              const int32_t *query_order, int num_frames, int spatial_size, int num_heads,
                              int channels, int num_levels, int num_query, int n_curr_points,
                              int n_temporal_points, int t_window, int ref_dim, int temporal_ref_mode, int dtype,
                              void *stream);
size_t devis_tmsda_fused_backward_workspace_bytes(int num_frames, int spatial_size, int num_heads, int channels,
                                                  unsigned flags);
int devis_tmsda_fused_backward(const void *value, const int64_t *spatial_shapes_host,
                               const int64_t *level_start_index_host, const int32_t *frame_table_host,
                               const void *ref, const void *off_curr, const void *logit_curr,
                               const void *off_temporal, const void *logit_temporal, const void *grad_output,
                               void *grad_value, void *grad_off_curr, void *grad_logit_curr,
                               void *grad_off_temporal, void *grad_logit_temporal, void *grad_ref,
                               const int32_t *query_order, int num_frames, int spatial_size, int num_heads,
                               int channels, int num_levels, int num_query, int n_curr_points,
                               int n_temporal_points, int t_window, int ref_dim, int temporal_ref_mode, int dtype,
                               unsigned flags, void *workspace, size_t workspace_bytes, void *stream);

/*
 * The two calls above with an input padding mask.  devis_tmsda_fused_forward / _backward are these with
 * padding_mask = NULL.
 *   padding_mask   optional DEVICE uint8 (num_frames, spatial_size), one byte per value row; nonzero = the row is
 *                  padding.  Exactly equivalent to value.masked_fill(padding_mask[..., None], 0) before the op -- even
 *                  when a masked row holds NaN or Inf: a masked corner contributes nothing to the output, receives no
 *                  grad_value and counts as a zero value in d/d(off_*), d/d(logit_*) and d/d(ref).  The mask is indexed
 *                  by the frame a tap samples, so it also applies to the temporal slots.  NULL = no mask.
 * This is what MSDeformAttn's input_padding_mask needs: its batch of N images is the frame axis (t_window = 0, no frame
 * table), the encoder with points (ref_dim 2), the decoder with points or boxes.
 */
int devis_tmsda_fused_forward_ex(const void *value, const int64_t *spatial_shapes_host,
                                 const int64_t *level_start_index_host, const int32_t *frame_table_host,
                                 const void *ref, const void *off_curr, const void *logit_curr,
                                 const void *off_temporal, const void *logit_temporal, void *output,
                                 void *loc_curr_out, void *aw_curr_out, void *loc_temporal_out, void *aw_temporal_out,
                                 const int32_t *query_order, const uint8_t *padding_mask, int num_frames,
                                 int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                 int n_curr_points, int n_temporal_points, int t_window, int ref_dim,
                                 int temporal_ref_mode, int dtype, void *stream);
int devis_tmsda_fused_backward_ex(const void *value, const int64_t *spatial_shapes_host,
                                  const int64_t *level_start_index_host, const int32_t *frame_table_host,
                                  const void *ref, const void *off_curr, const void *logit_curr,
                                  const void *off_temporal, const void *logit_temporal, const void *grad_output,
                                  void *grad_value, void *grad_off_curr, void *grad_logit_curr,
                                  void *grad_off_temporal, void *grad_logit_temporal, void *grad_ref,
                                  const int32_t *query_order, const uint8_t *padding_mask, int num_frames,
                                  int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                  int n_curr_points, int n_temporal_points, int t_window, int ref_dim,
                                  int temporal_ref_mode, int dtype, unsigned flags, void *workspace,
                                  size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DEVIS_MSDA_H_ */
