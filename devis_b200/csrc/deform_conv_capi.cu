// deform_conv_capi.cu -- C ABI (include/devis_deform_conv.h) of the modulated deformable convolution kernels.
#include "../../include/devis_deform_conv.h"
#include "capi_common.h"
#include "deform_conv.cuh"
#include "dcn_igemm.cuh"

#include <mutex>

using namespace devis;

namespace {

int check_dims(const DcnDims &d, int dtype)
{
    if (dtype != DEVIS_MSDA_F32 && dtype != DEVIS_MSDA_F64) return DEVIS_MSDA_ERR_BAD_DTYPE;
    if (d.N < 0 || d.H <= 0 || d.W <= 0 || d.C <= 0 || d.Ho < 0 || d.Wo < 0 || d.kh <= 0 || d.kw <= 0 || d.sh <= 0 ||
        d.sw <= 0 || d.ph < 0 || d.pw < 0 || d.dh <= 0 || d.dw <= 0 || d.og < 1 || d.C % d.og)
        return DEVIS_MSDA_ERR_BAD_SHAPE;
    if ((long long)d.H * d.W >= (1LL << 31)) return DEVIS_MSDA_ERR_TOO_LARGE;
    return DEVIS_MSDA_OK;
}

// ---- deterministic grad_input (DEVIS_MSDA_FLAG_DETERMINISTIC, deform_conv.cuh "Deterministic form") ---------------------
// workspace: [int64 accumulators, one per grad_input element][4 x u32 bound factors]
size_t det_workspace_bytes(long long batch, long long height, long long width, long long channels)
{
    return (size_t)(batch * height * width * channels) * sizeof(long long) + 4 * sizeof(unsigned);
}

// host-side checks of a deterministic call, before any CUDA call
int check_det(const DcnDims &d, int dtype, const void *workspace, size_t workspace_bytes)
{
    if (dtype != DEVIS_MSDA_F32) return DEVIS_MSDA_ERR_UNSUPPORTED;
    // a tap's live corners are distinct pixels, so one grad_input element receives at most Ho*Wo*kh*kw contributions per
    // image, each below 2^F in magnitude: their int64 sum cannot overflow while that count stays below 2^(62 - F)
    if ((double)d.Ho * d.Wo * d.kh * d.kw >= (double)(1LL << (62 - kDetFracBits))) return DEVIS_MSDA_ERR_TOO_LARGE;
    if (!workspace || workspace_bytes < det_workspace_bytes(d.N, d.H, d.W, d.C)) return DEVIS_MSDA_ERR_WORKSPACE;
    return DEVIS_MSDA_OK;
}

// zero the accumulators and the bound factors; factor 0 = max|grad| (n_grad floats), factor 1 = max|mask| (1 without one;
// N * og * kh * kw * Ho * Wo elements)
int det_begin(void *workspace, const DcnDims &d, const void *grad, size_t n_grad, const void *mask, cudaStream_t st,
              DetScale &det, unsigned *&slots)
{
    const size_t n_acc = (size_t)d.N * d.H * d.W * d.C;
    const cudaError_t e = cudaMemsetAsync(workspace, 0, det_workspace_bytes(d.N, d.H, d.W, d.C), st);
    if (e != cudaSuccess) return devis_capi_cuda_fail(e);
    det.acc = reinterpret_cast<long long *>(workspace);
    slots = reinterpret_cast<unsigned *>(det.acc + n_acc);
    det.max_bits = slots;
    const int blocks = devis_capi_helper_blocks();
    absmax_kernel<Elem::F32><<<blocks, 256, 0, st>>>(grad, n_grad, slots);
    int rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_AUX);
    if (rc) return rc;
    if (mask) absmax_kernel<Elem::F32><<<blocks, 256, 0, st>>>(mask, (size_t)d.N * d.og * d.kh * d.kw * d.Ho * d.Wo, slots + 1);
    else set_word_kernel<<<1, 1, 0, st>>>(slots + 1, 0x3f800000u);
    return devis_capi_check_launch(DEVIS_MSDA_KERNEL_AUX);
}

// fixed point -> grad_input (channel order, every element written)
int det_finish(const DetScale &det, const DcnDims &d, void *grad_input, int n_factors, cudaStream_t st)
{
    det_finalize_kernel<<<devis_capi_helper_blocks(), 256, 0, st>>>(det.acc, (float *)grad_input,
                                                                   (size_t)d.N * d.H * d.W * d.C, det.max_bits, 0, n_factors);
    return devis_capi_check_launch(DEVIS_MSDA_KERNEL_AUX);
}

// lanes per tap: a group covers its offset group's Cg = C / og channels in 16-byte pieces; 8 lanes = one 128-byte line
// per corner row.  Grid: x = output plane (wo fastest), y = virtual kernel position g * K + k, z = batch item (in slices
// of at most 65535).
constexpr int kMaxGridZ = 65535;

// the grid's y dimension of the gather / scatter kernels, checked before any CUDA call
int check_grid_y(const DcnDims &d)
{
    return (long long)d.og * d.kh * d.kw > 65535 ? DEVIS_MSDA_ERR_TOO_LARGE : DEVIS_MSDA_OK;
}

template <class F4, class F8, class S8, class S32>
int dispatch(const DcnDims &d, int dtype, F4 f4, F8 f8, S8 s8, S32 s32)
{
    const long long plane = (long long)d.Ho * d.Wo;
    if (d.N == 0 || plane == 0) return DEVIS_MSDA_OK;
    int G;
    const int Cg = d.C / d.og;
    const bool vec = dtype == DEVIS_MSDA_F32 && Cg % 4 == 0;
    if (vec) G = Cg / 4 >= 8 ? 8 : 4;
    else G = Cg >= 32 ? 32 : 8;
    if (plane * G + 255 >= (1LL << 31)) return DEVIS_MSDA_ERR_TOO_LARGE;     // grid y: check_grid_y, by the callers
    for (int n0 = 0; n0 < d.N; n0 += kMaxGridZ) {
        const dim3 grid((unsigned)((plane * G + 255) / 256), (unsigned)(d.og * d.kh * d.kw),
                        (unsigned)(d.N - n0 < kMaxGridZ ? d.N - n0 : kMaxGridZ));
        if (vec) {
            if (G == 8) f8(grid, n0);
            else f4(grid, n0);
        } else {
            if (G == 32) s32(grid, n0);
            else s8(grid, n0);
        }
        const int rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
        if (rc) return rc;
    }
    return DEVIS_MSDA_OK;
}

}  // namespace

extern "C" {

int devis_dcn_im2col(const void *input, const void *offset, const void *mask, void *cols, int batch, int height,
                     int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w, int stride_h,
                     int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int dtype, void *stream)
{
    return devis_dcn_im2col_og(input, offset, mask, cols, batch, height, width, channels, out_h, out_w, kernel_h,
                               kernel_w, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, 1, dtype, stream);
}

int devis_dcn_im2col_og(const void *input, const void *offset, const void *mask, void *cols, int batch, int height,
                        int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w, int stride_h,
                        int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int offset_groups, int dtype,
                        void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, offset_groups};
    int rc = check_dims(d, dtype);
    if (!rc) rc = check_grid_y(d);
    if (rc) return rc;
    const long long n_taps = (long long)batch * out_h * out_w * kernel_h * kernel_w;
    if (n_taps > 0 && (!input || !offset || !cols)) return DEVIS_MSDA_ERR_NULL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == DEVIS_MSDA_F32) {
        const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask;
        float *co = (float *)cols;
        return dispatch(d, dtype,
                        [&](dim3 b, int n0) { dcn_im2col_kernel<float, 4, 4><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); },
                        [&](dim3 b, int n0) { dcn_im2col_kernel<float, 4, 8><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); },
                        [&](dim3 b, int n0) { dcn_im2col_kernel<float, 1, 8><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); },
                        [&](dim3 b, int n0) { dcn_im2col_kernel<float, 1, 32><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); });
    }
    const double *in = (const double *)input, *of = (const double *)offset, *mk = (const double *)mask;
    double *co = (double *)cols;
    return dispatch(d, dtype, [&](dim3, int) {}, [&](dim3, int) {},
                    [&](dim3 b, int n0) { dcn_im2col_kernel<double, 1, 8><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); },
                    [&](dim3 b, int n0) { dcn_im2col_kernel<double, 1, 32><<<b, 256, 0, st>>>(in, of, mk, co, d, n0); });
}

size_t devis_dcn_backward_workspace_bytes(int batch, int height, int width, int channels, unsigned flags)
{
    if (!(flags & DEVIS_MSDA_FLAG_DETERMINISTIC) || batch < 0 || height < 0 || width < 0 || channels < 0) return 0;
    return det_workspace_bytes(batch, height, width, channels);
}

int devis_dcn_col2im(const void *input, const void *offset, const void *mask, const void *grad_cols, void *grad_input,
                     void *grad_offset, void *grad_mask, int batch, int height, int width, int channels, int out_h,
                     int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h,
                     int dil_w, int dtype, void *stream)
{
    return devis_dcn_col2im_ex(input, offset, mask, grad_cols, grad_input, grad_offset, grad_mask, batch, height, width,
                               channels, out_h, out_w, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
                               dtype, 0u, nullptr, 0, stream);
}

int devis_dcn_col2im_ex(const void *input, const void *offset, const void *mask, const void *grad_cols, void *grad_input,
                        void *grad_offset, void *grad_mask, int batch, int height, int width, int channels, int out_h,
                        int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h,
                        int dil_w, int dtype, unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    return devis_dcn_col2im_og(input, offset, mask, grad_cols, grad_input, grad_offset, grad_mask, batch, height, width,
                               channels, out_h, out_w, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
                               1, dtype, flags, workspace, workspace_bytes, stream);
}

int devis_dcn_col2im_og(const void *input, const void *offset, const void *mask, const void *grad_cols, void *grad_input,
                        void *grad_offset, void *grad_mask, int batch, int height, int width, int channels, int out_h,
                        int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h,
                        int dil_w, int offset_groups, int dtype, unsigned flags, void *workspace, size_t workspace_bytes,
                        void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, offset_groups};
    int rc = check_dims(d, dtype);
    if (!rc) rc = check_grid_y(d);
    if (rc) return rc;
    const bool det_flag = (flags & DEVIS_MSDA_FLAG_DETERMINISTIC) && grad_input;
    if (det_flag) {
        rc = check_det(d, dtype, workspace, workspace_bytes);
        if (rc) return rc;
    }
    const long long n_taps = (long long)batch * out_h * out_w * kernel_h * kernel_w;
    if (n_taps > 0 && (!input || !offset || !grad_cols || !grad_offset || (mask && !grad_mask)))
        return DEVIS_MSDA_ERR_NULL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    const bool det = det_flag && n_taps > 0;        // no taps: grad_input is all zeros, filled below
    if (grad_input && !det) {   // torchvision: at::zeros_like(input)
        const size_t bytes = (size_t)batch * height * width * channels * (dtype == DEVIS_MSDA_F64 ? 8 : 4);
        if (bytes) {
            const cudaError_t e = cudaMemsetAsync(grad_input, 0, bytes, st);
            if (e != cudaSuccess) return devis_capi_cuda_fail(e);
        }
    }
    if (det) {
        DetScale ds{};
        unsigned *slots = nullptr;
        rc = det_begin(workspace, d, grad_cols, (size_t)n_taps * channels, mask, st, ds, slots);
        if (rc) return rc;
        const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask;
        const float *gc = (const float *)grad_cols;
        float *go = (float *)grad_offset, *gm = (float *)grad_mask;
        rc = dispatch(d, dtype,
                      [&](dim3 b, int n0) { dcn_col2im_kernel<float, 4, 4, true><<<b, 256, 0, st>>>(in, of, mk, gc, nullptr, go, gm, d, n0, ds); },
                      [&](dim3 b, int n0) { dcn_col2im_kernel<float, 4, 8, true><<<b, 256, 0, st>>>(in, of, mk, gc, nullptr, go, gm, d, n0, ds); },
                      [&](dim3 b, int n0) { dcn_col2im_kernel<float, 1, 8, true><<<b, 256, 0, st>>>(in, of, mk, gc, nullptr, go, gm, d, n0, ds); },
                      [&](dim3 b, int n0) { dcn_col2im_kernel<float, 1, 32, true><<<b, 256, 0, st>>>(in, of, mk, gc, nullptr, go, gm, d, n0, ds); });
        return rc ? rc : det_finish(ds, d, grad_input, kDcnDetFactorsCol2im, st);
    }
    const DetScale nodet{};
    if (dtype == DEVIS_MSDA_F32) {
        const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask;
        const float *gc = (const float *)grad_cols;
        float *gi = (float *)grad_input, *go = (float *)grad_offset, *gm = (float *)grad_mask;
        return dispatch(d, dtype,
                        [&](dim3 b, int n0) { dcn_col2im_kernel<float, 4, 4><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); },
                        [&](dim3 b, int n0) { dcn_col2im_kernel<float, 4, 8><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); },
                        [&](dim3 b, int n0) { dcn_col2im_kernel<float, 1, 8><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); },
                        [&](dim3 b, int n0) { dcn_col2im_kernel<float, 1, 32><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); });
    }
    const double *in = (const double *)input, *of = (const double *)offset, *mk = (const double *)mask;
    const double *gc = (const double *)grad_cols;
    double *gi = (double *)grad_input, *go = (double *)grad_offset, *gm = (double *)grad_mask;
    return dispatch(d, dtype, [&](dim3, int) {}, [&](dim3, int) {},
                    [&](dim3 b, int n0) { dcn_col2im_kernel<double, 1, 8><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); },
                    [&](dim3 b, int n0) { dcn_col2im_kernel<double, 1, 32><<<b, 256, 0, st>>>(in, of, mk, gc, gi, go, gm, d, n0, nodet); });
}


}  // extern "C"

// ---- fused gather + contraction (no column matrix) -------------------------------------------------------------------

namespace {

// which fused kernels serve a layer, and what the packed weight buffer holds for it
struct FusedPlan {
    int G = 0;                 // lanes per pixel of the lane-group kernels
    bool lanes_fwd = false;    // forward by dcn_fused_fwd_kernel
    bool lanes_bwd = false;    // data backward by dcn_fused_bwd_kernel
    bool constant = false;     // forward by dcn_fusedc_fwd_kernel (weights in the constant bank)
    int CT = 16;               // its output channels per thread
    size_t lanes_elems = 0, const_elems = 0;   // packed buffer = [lane-group layout | constant layout]
    bool any() const { return lanes_fwd || lanes_bwd || constant; }
};

// og offset groups: the lane-group kernels contract each group's Cg = C / og channels (Cg % 4 == 0); the constant-bank
// forward serves og = 1 only (its weight chunking works per kernel position)
FusedPlan fused_plan(int C, int cout, int kh, int kw, int dtype, int og)
{
    FusedPlan p;
    if (dtype != DEVIS_MSDA_F32 || og < 1 || C <= 0 || C % og || (C / og) % 4 || kh <= 0 || kw <= 0 || cout <= 0) return p;
    const long long K = (long long)kh * kw;
    const int Cg = C / og;
    const bool small = cout == 1 || cout == 2 || cout == 4 || cout == 8 || cout == 16;
    p.G = Cg / 4 > 4 ? 8 : 4;
    const bool c_served = C == 16 || C == 32 || C == 40 || C == 64 || C == 72;   // dcn_fusedc_fwd_kernel<C, CT> instantiations
    p.constant = og == 1 && c_served && cout % 16 == 0 && cout <= 64;
    p.CT = cout % 32 == 0 ? 32 : 16;
    p.lanes_bwd = small;
    p.lanes_fwd = small && !p.constant;
    if (p.lanes_fwd || p.lanes_bwd) p.lanes_elems = (size_t)K * og * ((Cg / 4 + p.G - 1) / p.G) * cout * p.G * 4;
    if (p.constant) p.const_elems = (size_t)K * C * cout;
    return p;
}

// the constant bank exists once PER DEVICE and is shared by every stream using that device: calls are serialised by a
// mutex on the host and, per device, by an event (a call on another stream waits for the previous call's kernels before
// it overwrites the bank).  State is indexed by the current device, so single-process multi-GPU callers
// (nn.DataParallel, per-thread devices) never record an event created on another device.
// Stream capture: the cross-stream guard cannot be recorded into a graph, so a captured call is only safe when no eager
// call on ANOTHER stream of the same device touches the bank while the graph replays (INTEGRATION.md section 5).
constexpr int kMaxDevices = 64;
std::mutex g_const_mutex;
struct ConstBankState {
    cudaEvent_t event = nullptr;
    cudaStream_t stream = nullptr;
    bool used = false;
} g_const[kMaxDevices];

bool stream_is_capturing(cudaStream_t st)
{
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &status) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return status != cudaStreamCaptureStatusNone;
}

}  // namespace

extern "C" {

int devis_dcn_fused_form(int channels, int out_channels, int kernel_h, int kernel_w, int dtype)
{
    return devis_dcn_fused_form_og(channels, out_channels, kernel_h, kernel_w, 1, dtype);
}

int devis_dcn_fused_form_og(int channels, int out_channels, int kernel_h, int kernel_w, int offset_groups, int dtype)
{
    const FusedPlan p = fused_plan(channels, out_channels, kernel_h, kernel_w, dtype, offset_groups);
    return ((p.lanes_fwd || p.constant) ? 1 : 0) | (p.lanes_bwd ? 2 : 0);
}

size_t devis_dcn_packed_weight_elems(int channels, int out_channels, int kernel_h, int kernel_w)
{
    return devis_dcn_packed_weight_elems_og(channels, out_channels, kernel_h, kernel_w, 1);
}

size_t devis_dcn_packed_weight_elems_og(int channels, int out_channels, int kernel_h, int kernel_w, int offset_groups)
{
    const FusedPlan p = fused_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32, offset_groups);
    return p.lanes_elems + p.const_elems;
}

int devis_dcn_pack_weight(const void *weight, void *packed, int channels, int out_channels, int kernel_h, int kernel_w,
                          void *stream)
{
    return devis_dcn_pack_weight_og(weight, packed, channels, out_channels, kernel_h, kernel_w, 1, stream);
}

int devis_dcn_pack_weight_og(const void *weight, void *packed, int channels, int out_channels, int kernel_h, int kernel_w,
                             int offset_groups, void *stream)
{
    if (kernel_h <= 0 || kernel_w <= 0 || channels <= 0 || out_channels <= 0 || offset_groups < 1 ||
        channels % offset_groups)
        return DEVIS_MSDA_ERR_BAD_SHAPE;
    const FusedPlan p = fused_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32, offset_groups);
    if (!p.any()) return DEVIS_MSDA_ERR_UNSUPPORTED;
    if (!weight || !packed) return DEVIS_MSDA_ERR_NULL_POINTER;
    const int K = kernel_h * kernel_w;
    cudaStream_t st = (cudaStream_t)stream;
    if (p.lanes_elems) {
        const int nblk = (channels / offset_groups / 4 + p.G - 1) / p.G;
        const unsigned blocks = (unsigned)((p.lanes_elems + 255) / 256 > 1184 ? 1184 : (p.lanes_elems + 255) / 256);
        dcn_pack_weight_kernel<<<blocks, 256, 0, st>>>((const float *)weight, (float *)packed, out_channels, channels, K,
                                                       p.G, nblk, offset_groups);
        const int rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
        if (rc) return rc;
    }
    if (p.const_elems) {
        const unsigned blocks = (unsigned)((p.const_elems + 255) / 256 > 1184 ? 1184 : (p.const_elems + 255) / 256);
        dcn_pack_weight_const_kernel<<<blocks, 256, 0, st>>>((const float *)weight, (float *)packed + p.lanes_elems,
                                                             out_channels, channels, K, p.CT);
        const int rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
        if (rc) return rc;
    }
    return DEVIS_MSDA_OK;
}

// pixels per lane group: the weights fetched for one (position, channel block) serve PPG pixels
#define DCN_FUSED_LAUNCH(KERNEL, COUT, G, PPG, ...)                                                          \
    for (int n0 = 0; n0 < d.N; n0 += kMaxGridZ) {                                                            \
        const dim3 grid((unsigned)((d.Wo + (32 / G) * PPG - 1) / ((32 / G) * PPG)), (unsigned)((d.Ho + 7) / 8), \
                        (unsigned)(d.N - n0 < kMaxGridZ ? d.N - n0 : kMaxGridZ));                            \
        KERNEL<COUT, G, PPG><<<grid, 256, 0, st>>>(__VA_ARGS__, d, n0);                                      \
        const int rc_ = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);                                                           \
        if (rc_) return rc_;                                                                                 \
    }
#define DCN_FUSED_CASES(KERNEL, G, PPG, ...)                                     \
    switch (out_channels) {                                                      \
    case 1: DCN_FUSED_LAUNCH(KERNEL, 1, G, PPG, __VA_ARGS__) break;              \
    case 2: DCN_FUSED_LAUNCH(KERNEL, 2, G, PPG, __VA_ARGS__) break;              \
    case 4: DCN_FUSED_LAUNCH(KERNEL, 4, G, PPG, __VA_ARGS__) break;              \
    case 8: DCN_FUSED_LAUNCH(KERNEL, 8, G, PPG, __VA_ARGS__) break;              \
    default: DCN_FUSED_LAUNCH(KERNEL, 16, G, PPG, __VA_ARGS__) break;            \
    }

int devis_dcn_fused_forward(const void *input, const void *offset, const void *mask, const void *packed_weight,
                            const void *bias, void *out, int batch, int height, int width, int channels, int out_h,
                            int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                            int dil_h, int dil_w, int out_channels, void *stream)
{
    return devis_dcn_fused_forward_og(input, offset, mask, packed_weight, bias, out, batch, height, width, channels, out_h,
                                      out_w, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, 1,
                                      out_channels, stream);
}

int devis_dcn_fused_forward_og(const void *input, const void *offset, const void *mask, const void *packed_weight,
                               const void *bias, void *out, int batch, int height, int width, int channels, int out_h,
                               int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                               int dil_h, int dil_w, int offset_groups, int out_channels, void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, offset_groups};
    const int rc = check_dims(d, DEVIS_MSDA_F32);
    if (rc) return rc;
    const FusedPlan plan = fused_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32, offset_groups);
    if (!plan.lanes_fwd && !plan.constant) return DEVIS_MSDA_ERR_UNSUPPORTED;
    const long long n_pixels = (long long)batch * out_h * out_w;
    if (n_pixels == 0) return DEVIS_MSDA_OK;
    if (!input || !offset || !packed_weight || !out) return DEVIS_MSDA_ERR_NULL_POINTER;
    if ((long long)out_h * out_w >= (1LL << 31) || (long long)height * width * channels >= (1LL << 31))
        return DEVIS_MSDA_ERR_TOO_LARGE;
    cudaStream_t st = (cudaStream_t)stream;
    const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask;
    const float *bs = (const float *)bias;
    float *o = (float *)out;
    if (plan.constant) {
        const float *wc = (const float *)packed_weight + plan.lanes_elems;
        const int K = kernel_h * kernel_w, CT = plan.CT;
        const int k_fit = kDcnConstFloats / (channels * CT);                    // kernel positions the bank holds
        const int n_chunks = (K + k_fit - 1) / k_fit, k_step = (K + n_chunks - 1) / n_chunks;
        const size_t smem = (((size_t)channels * kDcnCStride + 3) / 4 + 512) * 16;
        typedef void (*Kernel)(const float *, const float *, const float *, const float *, float *, DcnDims, int, int, int, int, int);
        Kernel kernel = nullptr;
#define DCN_CONST_PICK(CC)                                                                  \
        if (channels == CC) kernel = CT == 16 ? (Kernel)dcn_fusedc_fwd_kernel<CC, 16> : (Kernel)dcn_fusedc_fwd_kernel<CC, 32>;
        DCN_CONST_PICK(16) DCN_CONST_PICK(32) DCN_CONST_PICK(40) DCN_CONST_PICK(64) DCN_CONST_PICK(72)
#undef DCN_CONST_PICK
        if (!kernel) return DEVIS_MSDA_ERR_UNSUPPORTED;
        std::lock_guard<std::mutex> lock(g_const_mutex);
        {
            const cudaError_t e = cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return devis_capi_cuda_fail(e);
        }
        const bool capturing = stream_is_capturing(st);
        int dev = 0;
        {
            const cudaError_t e = cudaGetDevice(&dev);
            if (e != cudaSuccess) return devis_capi_cuda_fail(e);
            if (dev < 0 || dev >= kMaxDevices) return DEVIS_MSDA_ERR_UNSUPPORTED;
        }
        ConstBankState &bank = g_const[dev];
        if (!capturing) {
            if (!bank.event) {
                const cudaError_t e = cudaEventCreateWithFlags(&bank.event, cudaEventDisableTiming);
                if (e != cudaSuccess) return devis_capi_cuda_fail(e);
            }
            if (bank.used && bank.stream != st) {
                const cudaError_t e = cudaStreamWaitEvent(st, bank.event, 0);
                if (e != cudaSuccess) return devis_capi_cuda_fail(e);
            }
        }
        for (int t = 0; t < out_channels / CT; ++t) {
            for (int k0 = 0; k0 < K; k0 += k_step) {
                const int k1 = k0 + k_step < K ? k0 + k_step : K;
                const cudaError_t e = cudaMemcpyToSymbolAsync(dcn_cw, wc + ((size_t)t * K + k0) * channels * CT,
                                                              (size_t)(k1 - k0) * channels * CT * sizeof(float), 0,
                                                              cudaMemcpyDeviceToDevice, st);
                if (e != cudaSuccess) return devis_capi_cuda_fail(e);
                for (int n0 = 0; n0 < d.N; n0 += kMaxGridZ) {
                    const dim3 grid((unsigned)((d.Wo + kDcnCTileW - 1) / kDcnCTileW), (unsigned)((d.Ho + kDcnCTileH - 1) / kDcnCTileH),
                                    (unsigned)(d.N - n0 < kMaxGridZ ? d.N - n0 : kMaxGridZ));
                    kernel<<<grid, 256, smem, st>>>(in, of, mk, bs, o, d, n0, out_channels, CT * t, k0, k1);
                    const int rc_ = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
                    if (rc_) return rc_;
                }
            }
        }
        if (!capturing) {
            const cudaError_t e = cudaEventRecord(bank.event, st);
            if (e != cudaSuccess) return devis_capi_cuda_fail(e);
            bank.used = true;
            bank.stream = st;
        }
        return DEVIS_MSDA_OK;
    }
    const float4 *wp = (const float4 *)packed_weight;
    if (plan.G == 8) { DCN_FUSED_CASES(dcn_fused_fwd_kernel, 8, 2, in, of, mk, wp, bs, o) }
    else { DCN_FUSED_CASES(dcn_fused_fwd_kernel, 4, 2, in, of, mk, wp, bs, o) }
    return DEVIS_MSDA_OK;
}

int devis_dcn_fused_backward(const void *input, const void *offset, const void *mask, const void *packed_weight,
                             const void *grad_out, void *grad_input, void *grad_offset, void *grad_mask, int batch,
                             int height, int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w,
                             int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int out_channels,
                             void *stream)
{
    return devis_dcn_fused_backward_og(input, offset, mask, packed_weight, grad_out, grad_input, grad_offset, grad_mask,
                                       batch, height, width, channels, out_h, out_w, kernel_h, kernel_w, stride_h, stride_w,
                                       pad_h, pad_w, dil_h, dil_w, 1, out_channels, 0u, nullptr, 0, stream);
}

int devis_dcn_fused_backward_ex(const void *input, const void *offset, const void *mask, const void *packed_weight,
                                const void *grad_out, void *grad_input, void *grad_offset, void *grad_mask, int batch,
                                int height, int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w,
                                int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int out_channels,
                                unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    return devis_dcn_fused_backward_og(input, offset, mask, packed_weight, grad_out, grad_input, grad_offset, grad_mask,
                                       batch, height, width, channels, out_h, out_w, kernel_h, kernel_w, stride_h, stride_w,
                                       pad_h, pad_w, dil_h, dil_w, 1, out_channels, flags, workspace, workspace_bytes,
                                       stream);
}

}  // extern "C"

// the deterministic data backward, launched through the same DCN_FUSED_CASES switch as the default one
template <int COUT, int G, int PPG>
constexpr auto dcn_fused_bwd_det_kernel = dcn_fused_bwd_kernel<COUT, G, PPG, true>;

extern "C" {

int devis_dcn_fused_backward_og(const void *input, const void *offset, const void *mask, const void *packed_weight,
                                const void *grad_out, void *grad_input, void *grad_offset, void *grad_mask, int batch,
                                int height, int width, int channels, int out_h, int out_w, int kernel_h, int kernel_w,
                                int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int offset_groups,
                                int out_channels, unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, offset_groups};
    int rc = check_dims(d, DEVIS_MSDA_F32);
    if (rc) return rc;
    const FusedPlan plan = fused_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32, offset_groups);
    if (!plan.lanes_bwd) return DEVIS_MSDA_ERR_UNSUPPORTED;
    const bool det_flag = (flags & DEVIS_MSDA_FLAG_DETERMINISTIC) && grad_input;
    if (det_flag) {
        rc = check_det(d, DEVIS_MSDA_F32, workspace, workspace_bytes);
        if (rc) return rc;
    }
    const long long n_pixels = (long long)batch * out_h * out_w;
    if (n_pixels > 0 && (!input || !offset || !packed_weight || !grad_out || !grad_offset || (mask && !grad_mask)))
        return DEVIS_MSDA_ERR_NULL_POINTER;
    if (n_pixels > 0 && ((long long)out_h * out_w >= (1LL << 31) || (long long)height * width * channels >= (1LL << 31)))
        return DEVIS_MSDA_ERR_TOO_LARGE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool det = det_flag && n_pixels > 0;      // no pixels: grad_input is all zeros, filled below
    if (grad_input && !det) {
        const size_t bytes = (size_t)batch * height * width * channels * 4;
        if (bytes) {
            const cudaError_t e = cudaMemsetAsync(grad_input, 0, bytes, st);
            if (e != cudaSuccess) return devis_capi_cuda_fail(e);
        }
    }
    if (n_pixels == 0) return DEVIS_MSDA_OK;
    const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask;
    const float4 *wp = (const float4 *)packed_weight;
    const float *go = (const float *)grad_out;
    float *gi = (float *)grad_input, *gof = (float *)grad_offset, *gm = (float *)grad_mask;
    if (det) {
        DetScale ds{};
        unsigned *slots = nullptr;
        rc = det_begin(workspace, d, grad_out, (size_t)n_pixels * out_channels, mask, st, ds, slots);
        if (rc) return rc;
        // factors 2, 3: max|W| over the lane-group layout (zero padded: same maximum) and Cout
        absmax_kernel<Elem::F32><<<devis_capi_helper_blocks(), 256, 0, st>>>(packed_weight, plan.lanes_elems, slots + 2);
        rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_AUX);
        if (rc) return rc;
        const float cout_f = (float)out_channels;
        set_word_kernel<<<1, 1, 0, st>>>(slots + 3, *reinterpret_cast<const unsigned *>(&cout_f));
        rc = devis_capi_check_launch(DEVIS_MSDA_KERNEL_AUX);
        if (rc) return rc;
        if (plan.G == 8) { DCN_FUSED_CASES(dcn_fused_bwd_det_kernel, 8, 1, in, of, mk, wp, go, nullptr, gof, gm, ds) }
        else { DCN_FUSED_CASES(dcn_fused_bwd_det_kernel, 4, 1, in, of, mk, wp, go, nullptr, gof, gm, ds) }
        return det_finish(ds, d, grad_input, kDcnDetFactorsFused, st);
    }
    const DetScale nodet{};
    if (plan.G == 8) { DCN_FUSED_CASES(dcn_fused_bwd_kernel, 8, 1, in, of, mk, wp, go, gi, gof, gm, nodet) }
    else { DCN_FUSED_CASES(dcn_fused_bwd_kernel, 4, 1, in, of, mk, wp, go, gi, gof, gm, nodet) }
    return DEVIS_MSDA_OK;
}

/* devis_dcn_wgrad: 1 if devis_dcn_weight_grad serves the layer (float32, C in {16, 32}, out_channels in {1, 2, 4, 8, 16}) */
int devis_dcn_wgrad_supported(int channels, int out_channels, int kernel_h, int kernel_w, int dtype)
{
    if (dtype != DEVIS_MSDA_F32 || kernel_h <= 0 || kernel_w <= 0 || kernel_h * kernel_w > 65535) return 0;
    if (channels != 16 && channels != 32) return 0;
    return out_channels == 1 || out_channels == 2 || out_channels == 4 || out_channels == 8 || out_channels == 16;
}

int devis_dcn_weight_grad(const void *input, const void *offset, const void *mask, const void *grad_out, void *grad_weight,
                          int batch, int height, int width, int channels, int out_h, int out_w, int kernel_h,
                          int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                          int out_channels, void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w};
    const int rc = check_dims(d, DEVIS_MSDA_F32);
    if (rc) return rc;
    if (!devis_dcn_wgrad_supported(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32)) return DEVIS_MSDA_ERR_UNSUPPORTED;
    if (!grad_weight) return DEVIS_MSDA_ERR_NULL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t wbytes = (size_t)out_channels * kernel_h * kernel_w * channels * 4;
    const cudaError_t e = cudaMemsetAsync(grad_weight, 0, wbytes, st);
    if (e != cudaSuccess) return devis_capi_cuda_fail(e);
    const long long plane = (long long)out_h * out_w;
    if ((long long)batch * plane == 0) return DEVIS_MSDA_OK;
    if (!input || !offset || !grad_out) return DEVIS_MSDA_ERR_NULL_POINTER;
    if (plane >= (1LL << 30) || (long long)height * width * channels >= (1LL << 31)) return DEVIS_MSDA_ERR_TOO_LARGE;
    const int G = channels / 4, gpb = 256 / G;
    // pixels per lane group: long runs amortise the block reduction, but keep >= ~4 blocks per SM in flight
    int run = 64;
    while (run > 8 && ((plane + (long long)gpb * run - 1) / ((long long)gpb * run)) * kernel_h * kernel_w * batch < devis_capi_helper_blocks()) run /= 2;
    const unsigned gx = (unsigned)((plane + (long long)gpb * run - 1) / ((long long)gpb * run));
    const float *in = (const float *)input, *of = (const float *)offset, *mk = (const float *)mask, *go = (const float *)grad_out;
    float *gw = (float *)grad_weight;
    for (int n0 = 0; n0 < batch; n0 += kMaxGridZ) {
        const dim3 grid(gx, (unsigned)(kernel_h * kernel_w), (unsigned)(batch - n0 < kMaxGridZ ? batch - n0 : kMaxGridZ));
#define DCN_WGRAD(CO, GG) dcn_wgrad_kernel<CO, GG><<<grid, 256, 0, st>>>(in, of, mk, go, gw, d, n0, run)
#define DCN_WGRAD_G(CO)                      \
    do {                                     \
        if (G == 8) DCN_WGRAD(CO, 8);        \
        else DCN_WGRAD(CO, 4);               \
    } while (0)
        switch (out_channels) {
        case 1: DCN_WGRAD_G(1); break;
        case 2: DCN_WGRAD_G(2); break;
        case 4: DCN_WGRAD_G(4); break;
        case 8: DCN_WGRAD_G(8); break;
        default: DCN_WGRAD_G(16); break;
        }
#undef DCN_WGRAD_G
#undef DCN_WGRAD
        const int rc2 = devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
        if (rc2) return rc2;
    }
    return DEVIS_MSDA_OK;
}


// ---- tensor-core implicit GEMM forward (dcn_igemm.cuh) -----------------------------------------------------------------
namespace {

struct IgPlan {
    bool ok = false;
    int Npad = 0, nchunks = 0, n0 = 0, n1 = 0, tmem_cols = 0;
    // blocks per SM the launch aims for: the shared-memory budget of a block is 227 KB / blocks
    int blocks(int split) const
    {
#ifdef DEVIS_IG_BLOCKS
        (void)split;
        return DEVIS_IG_BLOCKS;
#else
        const int stage = (split ? 2 : 1) * (devis::kIgATile + Npad * 128);
        return (2 * stage + devis::kIgGeomBytes + 2048) * 2 <= 227 * 1024 ? 2 : 1;
#endif
    }
    int stages(int split) const
    {
        const int stage = (split ? 2 : 1) * (devis::kIgATile + Npad * 128);
        int s = (227 * 1024 / blocks(split) - devis::kIgGeomBytes - 256 - 1024 - 1024) / stage;
        return s > devis::kIgMaxStages ? devis::kIgMaxStages : s;
    }
    size_t smem(int split) const
    {
        return (size_t)stages(split) * (split ? 2 : 1) * (devis::kIgATile + Npad * 128) + devis::kIgGeomBytes + 256 + 1024;
    }
};

IgPlan igemm_plan(int channels, int out_channels, int kernel_h, int kernel_w, int dtype)
{
    IgPlan p;
    if (dtype != DEVIS_MSDA_F32 || channels <= 0 || out_channels <= 0 || kernel_h <= 0 || kernel_w <= 0) return p;
    if (channels % 8 != 0 || out_channels % 4 != 0) return p;
    p.Npad = (out_channels + 15) / 16 * 16;
    if (p.Npad > 512) return p;
    p.nchunks = (channels + devis::kIgBK - 1) / devis::kIgBK;
    if (p.Npad <= 256) {
        p.n0 = p.Npad;
    } else {                                  // two MMAs along N, both multiples of 16 and <= 256
        p.n0 = (p.Npad / 2 + 15) / 16 * 16;
        p.n1 = p.Npad - p.n0;
    }
    p.tmem_cols = 32;
    while (p.tmem_cols < p.Npad) p.tmem_cols *= 2;
    p.ok = p.stages(1) >= 2;
    return p;
}

}  // namespace

int devis_dcn_igemm_supported(int channels, int out_channels, int kernel_h, int kernel_w, int dtype)
{
    return igemm_plan(channels, out_channels, kernel_h, kernel_w, dtype).ok ? 1 : 0;
}

size_t devis_dcn_igemm_packed_weight_elems(int channels, int out_channels, int kernel_h, int kernel_w)
{
    const IgPlan p = igemm_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32);
    return p.ok ? (size_t)kernel_h * kernel_w * p.nchunks * 2 * p.Npad * devis::kIgBK : 0;
}

int devis_dcn_igemm_pack_weight(const void *weight, void *packed, int channels, int out_channels, int kernel_h, int kernel_w,
                                void *stream)
{
    if (kernel_h <= 0 || kernel_w <= 0 || channels <= 0 || out_channels <= 0) return DEVIS_MSDA_ERR_BAD_SHAPE;
    const IgPlan p = igemm_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32);
    if (!p.ok) return DEVIS_MSDA_ERR_UNSUPPORTED;
    if (!weight || !packed) return DEVIS_MSDA_ERR_NULL_POINTER;
    const long long total = (long long)kernel_h * kernel_w * p.nchunks * p.Npad * devis::kIgBK;
    const long long want = (total + 255) / 256;
    const unsigned blocks = (unsigned)(want > devis_capi_helper_blocks() ? devis_capi_helper_blocks() : want);
    devis::dcn_igemm_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float *)weight, (float *)packed, out_channels,
                                                                          channels, kernel_h * kernel_w, p.Npad, p.nchunks);
    return devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN);
}

int devis_dcn_igemm_forward(const void *input, const void *offset, const void *mask, const void *packed_weight,
                            const void *bias, void *out, int batch, int height, int width, int channels, int out_h,
                            int out_w, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                            int dil_h, int dil_w, int out_channels, int precision, void *stream)
{
    const DcnDims d{batch, height, width, channels, out_h, out_w, kernel_h, kernel_w,
                    stride_h, stride_w, pad_h, pad_w, dil_h, dil_w};
    const int rc = check_dims(d, DEVIS_MSDA_F32);
    if (rc) return rc;
    if (precision != DEVIS_DCN_PRECISION_3XTF32 && precision != DEVIS_DCN_PRECISION_TF32) return DEVIS_MSDA_ERR_BAD_SHAPE;
    const IgPlan p = igemm_plan(channels, out_channels, kernel_h, kernel_w, DEVIS_MSDA_F32);
    if (!p.ok) return DEVIS_MSDA_ERR_UNSUPPORTED;
    const long long P = (long long)batch * out_h * out_w;
    if (P == 0) return DEVIS_MSDA_OK;
    if (!input || !offset || !packed_weight || !out) return DEVIS_MSDA_ERR_NULL_POINTER;
    // the producers address the input with 32-bit element offsets
    if ((long long)batch * height * width * channels >= (1LL << 31) || (long long)out_h * out_w >= (1LL << 30) ||
        (P + devis::kIgBM - 1) / devis::kIgBM > 0x7fffffffLL)
        return DEVIS_MSDA_ERR_TOO_LARGE;
    const int split = precision == DEVIS_DCN_PRECISION_3XTF32 ? 1 : 0;
    devis::IgArgs a{};
    a.input = (const float *)input;
    a.offset = (const float *)offset;
    a.mask = (const float *)mask;
    a.wpacked = (const float *)packed_weight;
    a.bias = (const float *)bias;
    a.out = (float *)out;
    a.d = d;
    a.Cout = out_channels;
    a.Npad = p.Npad;
    a.nchunks = p.nchunks;
    a.stages = p.stages(split);
    a.split = split;
    a.n0 = p.n0;
    a.n1 = p.n1;
    a.tmem_cols = p.tmem_cols;
    a.P = P;
    const size_t smem = p.smem(split);
    const unsigned grid = (unsigned)((P + devis::kIgBM - 1) / devis::kIgBM);
    const int blocks = p.blocks(split);
    auto launch = [&](auto kernel) -> int {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return devis_capi_cuda_fail(e);
        kernel<<<grid, devis::kIgThreads, smem, (cudaStream_t)stream>>>(a);
        return DEVIS_MSDA_OK;
    };
    const int lrc = blocks >= 3 ? launch(devis::dcn_igemm_fwd_kernel<3>)
                                : blocks == 2 ? launch(devis::dcn_igemm_fwd_kernel<2>) : launch(devis::dcn_igemm_fwd_kernel<1>);
    if (lrc) return lrc;
    return devis_capi_check_launch(DEVIS_MSDA_KERNEL_DCN_IGEMM);
}

}  // extern "C"
