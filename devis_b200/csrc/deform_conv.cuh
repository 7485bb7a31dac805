// deform_conv.cuh -- modulated deformable convolution (DCNv2) gather / scatter kernels for sm_100a.
//
// DeVIS's mask head (src/models/deformable_segmentation.py:244-267, MaskHeadConv :323-380) calls
// torchvision.ops.deform_conv2d for every 3x3 layer.  torchvision's CUDA op (torchvision/csrc/ops/cuda/
// deform_conv2d_kernel.cu, a third-party dependency of the reference, pinned at torchvision 0.12 in docs/INSTALL.md)
// is the 2017 im2col design: NCHW input, one thread per (channel, output pixel) column element, scalar 4-byte gathers
// whose 4 corners are (H*W) floats apart from the next channel's, scalar atomicAdd scatter in the backward, a
// 5x5-neighbourhood search per column element for grad_input and a serial loop over channels for grad_offset.
//
// Here the same arithmetic (bilinear_interpolate with zero padding, deform_conv2d_kernel.cu `bilinear_interpolate`,
// `deformable_im2col_kernel`, `deformable_col2im_kernel`, `deformable_col2im_coord_kernel`) is laid out like the
// attention kernels of this library:
//   * the input is read CHANNELS-LAST (N, H, W, C): a bilinear corner is one contiguous row of C channels, gathered
//     with 16-byte loads by a group of G lanes (G = 4..32 by channel count);
//   * a TAP is one (output pixel, kernel position, offset group): the tap's geometry is computed once per lane group,
//     its column slice (the group's Cg = C / offset_groups channels) is written contiguously:
//     cols[(pixel * K + k) * C + g * Cg + c] -- the GEMM with the weights stays in cuBLAS (as torchvision's does,
//     at::addmm), it is not part of this file;
//   * backward: ONE pass per tap gathers the four corner rows again, forms the four dot products
//     A_c = sum_ch grad_col[ch] * corner_c[ch] (reduced over the group with shuffles) from which grad_mask and
//     grad_offset follow in closed form, and scatters grad_input with 16-byte vector reductions
//     (red.global.add.v4.f32) -- replacing torchvision's three kernels and its scalar atomics;
//   * grad_offset / grad_mask are written exactly once (no zero fill); only grad_input is zero-filled by the launcher.
// Offset groups (torchvision's offset_groups, DCNv2's deformable groups): group g of G reads offset channels
// 2 * (g * K + k) (+1) and mask channel g * K + k, and covers input channels [g * Cg, (g + 1) * Cg).  A kernel position
// of a group is a VIRTUAL position v = g * K + k with its own channel window; with G = 1, v = k and every kernel computes
// what it computed before offset groups existed.  The im2col / col2im kernels and the lane-group fused kernels serve
// any G; the constant-bank forward, the tcgen05 forward (dcn_igemm.cuh) and dcn_wgrad_kernel serve G = 1 only.
// groups = 1 (no weight grouping); any kernel size, stride, padding, dilation.
//
// Deterministic form (DET = true, float only).  The float scatter of grad_input sums in arrival order, so its last bits
// change from run to run.  The DET kernels convert every grad_input contribution m * w_corner * gc[c] exactly to a 64-bit
// fixed-point integer and add it with integer atomics (associative), with the machinery of the attention's deterministic
// grad_value (msda_common.cuh: DetScale, det_exponent, det_add4, det_finalize_kernel).  The scale is 2^(F - e),
// F = kDetFracBits, 2^e > 2 * bound, where the bound of every contribution |m * w_corner * gc| (|w_corner| <= 1) is the
// product of the factors in det.max_bits:
//   col2im        max|grad_cols| * max|mask|                      (kDcnDetFactorsCol2im)
//   fused bwd     max|grad_out|  * max|mask| * max|W| * Cout      (kDcnDetFactorsFused; gc = sum_co grad_out[co] * W[co][c][k]
//                 is never stored: Cout * max|W| bounds sum_co |W| and costs at most log2(Cout) <= 4 bits of resolution)
// (max|mask| is 1 without a mask).  The accumulators are in channel order, the input's channels-last layout: a lane's
// four channels are four consecutive 8-byte words (one full 32-byte sector), so no permutation is needed and
// det_finalize_kernel runs with lpg = 0.  The launcher rejects shapes whose Ho * Wo * kh * kw contributions per element
// and image could overflow int64 (DEVIS_MSDA_ERR_TOO_LARGE).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "msda_common.cuh"

namespace devis {

constexpr int kDcnDetFactorsCol2im = 2, kDcnDetFactorsFused = 4;

// one fixed-point contribution (sh is a power of two: the product and its conversion are exact)
__device__ __forceinline__ void dcn_det_add(long long *p, float sh, float v)
{
    atomicAdd(reinterpret_cast<unsigned long long *>(p), (unsigned long long)__float2ll_rn(v * sh));
}

__device__ __forceinline__ float dcn_det_scale(const DetScale &det, int n_factors)
{
    return ldexpf(1.f, kDetFracBits - det_exponent(det.max_bits, n_factors));
}

// one 16-byte vector reduction (SASS REDG.E.ADD.F32x4) instead of four scalar atomics
__device__ __forceinline__ void dcn_red_add_f4(float *p, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

struct DcnDims {
    int N, H, W, C;       // input, channels-last
    int Ho, Wo;           // output size
    int kh, kw, sh, sw, ph, pw, dh, dw;
    int og = 1;           // offset groups: C % og == 0
};

// geometry of one tap, torchvision's bilinear_interpolate: the sample is void unless -1 < h < H and -1 < w < W; corners
// outside the map contribute zero.  Rows are clamped in-bounds and their weights zeroed, but a corner outside the map
// (ok == false) must never contribute its value: the clamped row is some other pixel, and 0 * Inf = NaN would carry a
// non-finite value there into taps that never sample it.  The gathers load corners through dcn_corner / dcn_corner4
// (not read, value 0 when dead); the scatter kernels use them only in dot products zeroed by ok afterwards.
template <typename T>
struct DcnTap {
    T w[4];          // bilinear weights of TL, TR, BL, BR with outside corners zeroed
    T hh, hw, lh, lw;
    int row[4];      // (y * W + x) of the clamped corners
    bool ok[4];
    bool inside;
};

template <typename T>
__device__ __forceinline__ DcnTap<T> dcn_tap(T h, T w, int H, int W)
{
    DcnTap<T> t;
    t.inside = h > (T)-1 && w > (T)-1 && h < (T)H && w < (T)W;
    const T hf = floor(h), wf = floor(w);
    const int h0 = t.inside ? (int)hf : 0, w0 = t.inside ? (int)wf : 0;
    t.lh = h - hf;
    t.lw = w - wf;
    t.hh = (T)1 - t.lh;
    t.hw = (T)1 - t.lw;
    const bool top = t.inside && h0 >= 0, bot = t.inside && h0 + 1 <= H - 1;
    const bool lef = t.inside && w0 >= 0, rig = t.inside && w0 + 1 <= W - 1;
    t.ok[0] = top && lef;
    t.ok[1] = top && rig;
    t.ok[2] = bot && lef;
    t.ok[3] = bot && rig;
    t.w[0] = t.ok[0] ? t.hh * t.hw : (T)0;
    t.w[1] = t.ok[1] ? t.hh * t.lw : (T)0;
    t.w[2] = t.ok[2] ? t.lh * t.hw : (T)0;
    t.w[3] = t.ok[3] ? t.lh * t.lw : (T)0;
    const int h0c = max(h0, 0), h1c = min(h0 + 1, H - 1), w0c = max(w0, 0), w1c = min(w0 + 1, W - 1);
    t.row[0] = h0c * W + w0c;
    t.row[1] = h0c * W + w1c;
    t.row[2] = h1c * W + w0c;
    t.row[3] = h1c * W + w1c;
    return t;
}

// one corner value of a gather: the load is predicated off for a corner outside the map, whose value is 0.  (Loading the
// clamped row unconditionally and selecting 0 afterwards needs fewer registers in dcn_wgrad_kernel, but measured slower
// on every mask-head layer, 7 to 33 % for the tensor-core forward: the dead corners of border taps then cost memory
// traffic.)
template <typename T>
__device__ __forceinline__ T dcn_corner(const T *p, bool ok)
{
    return ok ? *p : (T)0;
}

__device__ __forceinline__ float4 dcn_corner4(const float4 *p, bool ok)
{
    return ok ? __ldg(p) : make_float4(0.f, 0.f, 0.f, 0.f);
}

// A tap is addressed by the launch grid: blockIdx.z (+ n_base) = batch item, blockIdx.y = virtual kernel position
// v = g * K + k (offset group g, kernel position k), and the
// x dimension runs over the output plane with wo fastest: the groups of a warp work on neighbouring output pixels for
// the same kernel position, so their offset / mask reads are coalesced and their gathers share a neighbourhood of the
// input.  (32-bit arithmetic only: a 64-bit division per index component cost more than the gather itself.)
struct DcnTapId {
    int n, k, ho, wo;
    int v;             // g * K + k: the tap's offset / mask channel (offset group g)
    long long pixel;   // (n * Ho + ho) * Wo + wo
};

__device__ __forceinline__ DcnTapId dcn_tap_id(int plane_pixel, int n, int k, const DcnDims &d)
{
    DcnTapId id;
    id.n = n;
    id.k = k;
    id.v = k;
    id.ho = plane_pixel / d.Wo;
    id.wo = plane_pixel - id.ho * d.Wo;
    id.pixel = (long long)n * d.Ho * d.Wo + plane_pixel;
    return id;
}

template <typename T>
__device__ __forceinline__ void dcn_sample_point(const T *offset, const T *mask, const DcnTapId &id, const DcnDims &d,
                                                 T &h, T &w, T &m)
{
    const int GK = d.og * d.kh * d.kw;
    const long long plane = (long long)d.Ho * d.Wo;
    const long long at = (long long)id.ho * d.Wo + id.wo;
    const T off_h = offset[((long long)id.n * 2 * GK + 2 * id.v) * plane + at];
    const T off_w = offset[((long long)id.n * 2 * GK + 2 * id.v + 1) * plane + at];
    m = mask ? mask[((long long)id.n * GK + id.v) * plane + at] : (T)1;
    const int ky = id.k / d.kw, kx = id.k - ky * d.kw;
    h = (T)(id.ho * d.sh - d.ph + ky * d.dh) + off_h;
    w = (T)(id.wo * d.sw - d.pw + kx * d.dw) + off_w;
}

// ---------------------------------------------------------------------------------------------------------------------
// forward gather: cols[(pixel * K + k) * C + g * Cg + c] = mask * bilinear(input[n, :, :, g * Cg + c], h, w)
// V = channels per lane and load (4: float4, Cg % 4 == 0; 1: any Cg / double)
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int V, int G>
__global__ void __launch_bounds__(256) dcn_im2col_kernel(const T *__restrict__ input, const T *__restrict__ offset,
                                                         const T *__restrict__ mask, T *__restrict__ cols, DcnDims d,
                                                         int n_base)
{
    const int j = threadIdx.x % G;
    const int pp = (int)((blockIdx.x * blockDim.x + threadIdx.x) / G);
    if (pp >= d.Ho * d.Wo) return;
    const int K = d.kh * d.kw, v = (int)blockIdx.y, grp = d.og > 1 ? v / K : 0, Cg = d.C / d.og;
    DcnTapId id = dcn_tap_id(pp, n_base + (int)blockIdx.z, v - grp * K, d);
    id.v = v;
    T h, w, m;
    dcn_sample_point(offset, mask, id, d, h, w, m);
    const DcnTap<T> t = dcn_tap(h, w, d.H, d.W);
    const T *img = input + (long long)id.n * d.H * d.W * d.C + grp * Cg;
    T *out = cols + (id.pixel * K + id.k) * (long long)d.C + grp * Cg;
    const T f0 = m * t.w[0], f1 = m * t.w[1], f2 = m * t.w[2], f3 = m * t.w[3];
    if (V == 4) {
        const float4 *r0 = reinterpret_cast<const float4 *>(img + (long long)t.row[0] * d.C);
        const float4 *r1 = reinterpret_cast<const float4 *>(img + (long long)t.row[1] * d.C);
        const float4 *r2 = reinterpret_cast<const float4 *>(img + (long long)t.row[2] * d.C);
        const float4 *r3 = reinterpret_cast<const float4 *>(img + (long long)t.row[3] * d.C);
        float4 *o = reinterpret_cast<float4 *>(out);
        for (int c = j; c < Cg / 4; c += G) {
            const float4 a = dcn_corner4(r0 + c, t.ok[0]), b = dcn_corner4(r1 + c, t.ok[1]);
            const float4 e = dcn_corner4(r2 + c, t.ok[2]), f = dcn_corner4(r3 + c, t.ok[3]);
            float4 s;
            s.x = f0 * a.x + f1 * b.x + f2 * e.x + f3 * f.x;
            s.y = f0 * a.y + f1 * b.y + f2 * e.y + f3 * f.y;
            s.z = f0 * a.z + f1 * b.z + f2 * e.z + f3 * f.z;
            s.w = f0 * a.w + f1 * b.w + f2 * e.w + f3 * f.w;
            o[c] = s;
        }
    } else {
        const T *r0 = img + (long long)t.row[0] * d.C, *r1 = img + (long long)t.row[1] * d.C;
        const T *r2 = img + (long long)t.row[2] * d.C, *r3 = img + (long long)t.row[3] * d.C;
        for (int c = j; c < Cg; c += G)
            out[c] = f0 * dcn_corner(r0 + c, t.ok[0]) + f1 * dcn_corner(r1 + c, t.ok[1]) + f2 * dcn_corner(r2 + c, t.ok[2]) +
                     f3 * dcn_corner(r3 + c, t.ok[3]);
    }
}

__device__ __forceinline__ void dcn_red_add(float *p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void dcn_red_add(double *p, double v) { atomicAdd(p, v); }

// ---------------------------------------------------------------------------------------------------------------------
// backward: grad_input (scatter), grad_offset, grad_mask from grad_cols, one pass per tap (the offset / mask gradients of
// a tap are reduced over its group's Cg channels only)
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int V, int G, bool DET = false>
__global__ void __launch_bounds__(256) dcn_col2im_kernel(const T *__restrict__ input, const T *__restrict__ offset,
                                                         const T *__restrict__ mask, const T *__restrict__ grad_cols,
                                                         T *__restrict__ grad_input, T *__restrict__ grad_offset,
                                                         T *__restrict__ grad_mask, DcnDims d, int n_base, DetScale det)
{
    static_assert(!DET || sizeof(T) == 4, "the fixed-point form is float only");
    const int j = threadIdx.x % G;
    int pp = (int)((blockIdx.x * blockDim.x + threadIdx.x) / G);
    const bool live = pp < d.Ho * d.Wo;
    if (!live) pp = d.Ho * d.Wo - 1;   // keep the whole warp in the shuffles below; results of dead groups are dropped
    const int K = d.kh * d.kw, v = (int)blockIdx.y, grp = d.og > 1 ? v / K : 0, Cg = d.C / d.og;
    DcnTapId id = dcn_tap_id(pp, n_base + (int)blockIdx.z, v - grp * K, d);
    id.v = v;
    T h, w, m;
    dcn_sample_point(offset, mask, id, d, h, w, m);
    const DcnTap<T> t = dcn_tap(h, w, d.H, d.W);
    const T *img = input + (long long)id.n * d.H * d.W * d.C + grp * Cg;
    T *gimg = grad_input ? grad_input + (long long)id.n * d.H * d.W * d.C + grp * Cg : nullptr;
    const T *gc = grad_cols + (id.pixel * K + id.k) * (long long)d.C + grp * Cg;
    const T f0 = m * t.w[0], f1 = m * t.w[1], f2 = m * t.w[2], f3 = m * t.w[3];
    long long *gacc = nullptr;
    float det_sh = 0.f;
    if constexpr (DET) {
        gacc = det.acc + (long long)id.n * d.H * d.W * d.C + grp * Cg;
        det_sh = dcn_det_scale(det, kDcnDetFactorsCol2im);
    }
    T A0 = 0, A1 = 0, A2 = 0, A3 = 0;
    if (V == 4) {
        const float4 *r0 = reinterpret_cast<const float4 *>(img + (long long)t.row[0] * d.C);
        const float4 *r1 = reinterpret_cast<const float4 *>(img + (long long)t.row[1] * d.C);
        const float4 *r2 = reinterpret_cast<const float4 *>(img + (long long)t.row[2] * d.C);
        const float4 *r3 = reinterpret_cast<const float4 *>(img + (long long)t.row[3] * d.C);
        const float4 *g4 = reinterpret_cast<const float4 *>(gc);
        for (int c = j; c < Cg / 4; c += G) {
            const float4 g = __ldg(g4 + c);
            const float4 a = __ldg(r0 + c), b = __ldg(r1 + c), e = __ldg(r2 + c), f = __ldg(r3 + c);
            A0 += g.x * a.x + g.y * a.y + g.z * a.z + g.w * a.w;
            A1 += g.x * b.x + g.y * b.y + g.z * b.z + g.w * b.w;
            A2 += g.x * e.x + g.y * e.y + g.z * e.z + g.w * e.w;
            A3 += g.x * f.x + g.y * f.y + g.z * f.z + g.w * f.w;
            if constexpr (DET) {
                if (live) {
                    if (f0 != 0.f) det_add4<1>(gacc + (long long)t.row[0] * d.C + 4 * c, det_sh, f0 * g.x, f0 * g.y, f0 * g.z, f0 * g.w);
                    if (f1 != 0.f) det_add4<1>(gacc + (long long)t.row[1] * d.C + 4 * c, det_sh, f1 * g.x, f1 * g.y, f1 * g.z, f1 * g.w);
                    if (f2 != 0.f) det_add4<1>(gacc + (long long)t.row[2] * d.C + 4 * c, det_sh, f2 * g.x, f2 * g.y, f2 * g.z, f2 * g.w);
                    if (f3 != 0.f) det_add4<1>(gacc + (long long)t.row[3] * d.C + 4 * c, det_sh, f3 * g.x, f3 * g.y, f3 * g.z, f3 * g.w);
                }
            }
            if (live && gimg) {
                float *q = reinterpret_cast<float *>(gimg);
                if (f0 != 0.f) dcn_red_add_f4(q + (long long)t.row[0] * d.C + 4 * c, f0 * g.x, f0 * g.y, f0 * g.z, f0 * g.w);
                if (f1 != 0.f) dcn_red_add_f4(q + (long long)t.row[1] * d.C + 4 * c, f1 * g.x, f1 * g.y, f1 * g.z, f1 * g.w);
                if (f2 != 0.f) dcn_red_add_f4(q + (long long)t.row[2] * d.C + 4 * c, f2 * g.x, f2 * g.y, f2 * g.z, f2 * g.w);
                if (f3 != 0.f) dcn_red_add_f4(q + (long long)t.row[3] * d.C + 4 * c, f3 * g.x, f3 * g.y, f3 * g.z, f3 * g.w);
            }
        }
    } else {
        const T *r0 = img + (long long)t.row[0] * d.C, *r1 = img + (long long)t.row[1] * d.C;
        const T *r2 = img + (long long)t.row[2] * d.C, *r3 = img + (long long)t.row[3] * d.C;
        for (int c = j; c < Cg; c += G) {
            const T g = gc[c];
            A0 += g * r0[c];
            A1 += g * r1[c];
            A2 += g * r2[c];
            A3 += g * r3[c];
            if constexpr (DET) {
                if (live) {
                    if (f0 != (T)0) dcn_det_add(gacc + (long long)t.row[0] * d.C + c, det_sh, f0 * g);
                    if (f1 != (T)0) dcn_det_add(gacc + (long long)t.row[1] * d.C + c, det_sh, f1 * g);
                    if (f2 != (T)0) dcn_det_add(gacc + (long long)t.row[2] * d.C + c, det_sh, f2 * g);
                    if (f3 != (T)0) dcn_det_add(gacc + (long long)t.row[3] * d.C + c, det_sh, f3 * g);
                }
            }
            if (live && gimg) {
                if (f0 != (T)0) dcn_red_add(gimg + (long long)t.row[0] * d.C + c, f0 * g);
                if (f1 != (T)0) dcn_red_add(gimg + (long long)t.row[1] * d.C + c, f1 * g);
                if (f2 != (T)0) dcn_red_add(gimg + (long long)t.row[2] * d.C + c, f2 * g);
                if (f3 != (T)0) dcn_red_add(gimg + (long long)t.row[3] * d.C + c, f3 * g);
            }
        }
    }
#pragma unroll
    for (int o = G / 2; o >= 1; o >>= 1) {
        A0 += __shfl_xor_sync(0xffffffffu, A0, o, G);
        A1 += __shfl_xor_sync(0xffffffffu, A1, o, G);
        A2 += __shfl_xor_sync(0xffffffffu, A2, o, G);
        A3 += __shfl_xor_sync(0xffffffffu, A3, o, G);
    }
    if (live && j == 0) {
        // outside corners carry garbage from their clamped rows: zero them like the zero padding does
        A0 = t.ok[0] ? A0 : (T)0;
        A1 = t.ok[1] ? A1 : (T)0;
        A2 = t.ok[2] ? A2 : (T)0;
        A3 = t.ok[3] ? A3 : (T)0;
        const int GK = d.og * K;
        const long long plane = (long long)d.Ho * d.Wo, at = (long long)id.ho * d.Wo + id.wo;
        const T val = t.hh * (t.hw * A0 + t.lw * A1) + t.lh * (t.hw * A2 + t.lw * A3);
        const T gh = t.hw * (A2 - A0) + t.lw * (A3 - A1);      // d/dh of the interpolated value
        const T gw = t.hh * (A1 - A0) + t.lh * (A3 - A2);      // d/dw
        grad_offset[((long long)id.n * 2 * GK + 2 * v) * plane + at] = t.inside ? m * gh : (T)0;
        grad_offset[((long long)id.n * 2 * GK + 2 * v + 1) * plane + at] = t.inside ? m * gw : (T)0;
        if (grad_mask) grad_mask[((long long)id.n * GK + v) * plane + at] = t.inside ? val : (T)0;
    }
}

// =====================================================================================================================
// Fused kernels: gather + contraction with the convolution weights in one pass, the column matrix is never written.
//
// For the high-resolution layers of the mask head (few output channels: 72->32 at 45x80, 32->16 and 16->1 at 90x160)
// the column matrix is 9x the input and the GEMM is a thin one, so im2col + cuBLAS spends its time writing and
// re-reading columns (995 MB per direction for 60 instances at 90x160).  Here a group of G lanes owns one output pixel;
// a lane owns the channel pieces c = j, j+G, ... (4 channels each), interpolates them for kernel position k and
// immediately multiplies by the weights of (k, piece), accumulating COUT partial outputs in registers; after the 9
// positions the partials are combined over the group with a reduce-scatter butterfly and each lane stores COUT/G
// outputs.  HBM traffic = input + offsets + mask + output, once each.
//
// With offset groups the kernel positions become the G_off * K virtual positions v = g * K + k, each contracting its
// group's Cg = C / G_off channels (Cg % 4 == 0).
//
// PACKED WEIGHTS (devis_dcn_pack_weight_og): wp[((v * nblk + b) * COUT + co) * G + jj], v = g * K + k, is a float4
// holding weight[co][g*Cg + (b*G + jj)*4 + 0..3][ky][kx] (zero beyond the group's Cg channels), nblk = ceil(Cg / (4*G)):
// the slabs follow the virtual positions in the order the kernels walk them (with G_off = 1, v = k).  For a fixed
// (v, b, co) the G lanes of a group read 16*G contiguous bytes and all groups of a warp read the same bytes (one L1
// wavefront, broadcast).
// =====================================================================================================================
__global__ void dcn_pack_weight_kernel(const float *__restrict__ w /* (Cout, C, kh, kw) */, float *__restrict__ wp,
                                       int cout, int C, int K, int G, int nblk, int og)
{
    const long long total = (long long)K * og * nblk * cout * G * 4;
    const int Cg = C / og;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int e = (int)(i & 3);
        long long r = i >> 2;
        const int jj = (int)(r % G);
        r /= G;
        const int co = (int)(r % cout);
        r /= cout;
        const int b = (int)(r % nblk);
        const int v = (int)(r / nblk);
        const int g = v / K, k = v - g * K;
        const int c = (b * G + jj) * 4 + e;
        wp[i] = c < Cg ? w[((long long)co * C + g * Cg + c) * K + k] : 0.f;
    }
}

// sum of v[0..N) over the G lanes of a group.  N >= G: reduce-scatter, lane j ends with the totals of
// v[j*N/G .. (j+1)*N/G) in v[0 .. N/G).  N < G: every lane ends with all totals.
template <int N, int G>
__device__ __forceinline__ void dcn_group_sum(float (&v)[N], int j)
{
    if (N >= G) {
        int half = N / 2;
#pragma unroll
        for (int o = G / 2; o >= 1; o >>= 1, half >>= 1) {
            const bool up = (j & o) != 0;
#pragma unroll
            for (int i = 0; i < N / 2; ++i) {
                if (i < half) {
                    const float send = up ? v[i] : v[i + half];
                    const float keep = up ? v[i + half] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o, G);
                }
            }
        }
    } else {
#pragma unroll
        for (int o = G / 2; o >= 1; o >>= 1)
#pragma unroll
            for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o, G);
    }
}

// Work split of the fused kernels.  A block of 32*WARPS threads owns a tile of WARPS rows x TW = (32/G)*PPG columns of
// one output plane (blockIdx.z + n_base = batch item): warp w works on tile row w, a group of G lanes on PPG pixels next
// to each other -- the weights fetched for a (kernel position, channel block) are used for PPG pixels, and the tile's
// gathers stay in one neighbourhood of the input (L1 hits).  Pixels beyond the plane are computed on clamped
// coordinates (their lanes must take part in the group shuffles) and never stored.
template <int G, int PPG>
struct DcnTile {
    int j, n, ho, wo[PPG];
    bool row_live, live[PPG];
    long long at[PPG];     // ho * Wo + wo on clamped coordinates
    __device__ __forceinline__ DcnTile(const DcnDims &d, int n_base)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        j = lane % G;
        n = n_base + (int)blockIdx.z;
        const int h = (int)blockIdx.y * (int)(blockDim.x >> 5) + warp;
        row_live = h < d.Ho;
        ho = min(h, d.Ho - 1);
#pragma unroll
        for (int i = 0; i < PPG; ++i) {
            const int w = ((int)blockIdx.x * (32 / G) + lane / G) * PPG + i;
            live[i] = row_live && w < d.Wo;
            wo[i] = min(w, d.Wo - 1);
            at[i] = (long long)ho * d.Wo + wo[i];
        }
    }
};

struct DcnPoint {
    float oh, ow, m;
};

__device__ __forceinline__ DcnPoint dcn_load_point(const float *offset_n, const float *mask_n, int k, long long plane,
                                                   long long at)
{
    DcnPoint p;
    p.oh = __ldg(offset_n + (2 * k) * plane + at);
    p.ow = __ldg(offset_n + (2 * k + 1) * plane + at);
    p.m = mask_n ? __ldg(mask_n + k * plane + at) : 1.f;
    return p;
}

template <int COUT, int G, int PPG>
__global__ void __launch_bounds__(256, 2) dcn_fused_fwd_kernel(const float *__restrict__ input, const float *__restrict__ offset,
                                                            const float *__restrict__ mask, const float4 *__restrict__ wp,
                                                            const float *__restrict__ bias, float *__restrict__ out,
                                                            DcnDims d, int n_base)
{
    const DcnTile<G, PPG> tile(d, n_base);
    if (!tile.row_live) return;          // whole warp
    const int j = tile.j;
    const int K = d.kh * d.kw, GK = d.og * K, C4 = d.C / 4, Cg4 = C4 / d.og, nblk = (Cg4 + G - 1) / G;
    const long long plane = (long long)d.Ho * d.Wo;
    const float4 *img = reinterpret_cast<const float4 *>(input + (long long)tile.n * d.H * d.W * d.C);
    const float *offset_n = offset + (long long)tile.n * 2 * GK * plane;
    const float *mask_n = mask ? mask + (long long)tile.n * GK * plane : nullptr;
    float acc[PPG][COUT];
#pragma unroll
    for (int i = 0; i < PPG; ++i)
#pragma unroll
        for (int co = 0; co < COUT; ++co) acc[i][co] = 0.f;
    DcnPoint nxt[PPG];
#pragma unroll
    for (int i = 0; i < PPG; ++i) nxt[i] = dcn_load_point(offset_n, mask_n, 0, plane, tile.at[i]);
    // virtual position v = grp * K + k: kernel position k of offset group grp, channel pieces [grp * Cg4, (grp + 1) * Cg4)
    for (int v = 0, grp = 0, k = 0; v < GK; ++v) {
        const int ky = k / d.kw, kx = k - ky * d.kw;
        float fw[PPG][4];
        int row[PPG][4];
        bool ok[PPG][4];
#pragma unroll
        for (int i = 0; i < PPG; ++i) {
            const float h = (float)(tile.ho * d.sh - d.ph + ky * d.dh) + nxt[i].oh;
            const float w = (float)(tile.wo[i] * d.sw - d.pw + kx * d.dw) + nxt[i].ow;
            const DcnTap<float> t = dcn_tap(h, w, d.H, d.W);      // a sample outside the map has four dead corners
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                fw[i][q] = nxt[i].m * t.w[q];
                row[i][q] = t.row[q] * C4 + grp * Cg4;
                ok[i][q] = t.ok[q];
            }
        }
        if (v + 1 < GK) {    // next position's offsets and mask: in flight while this one is gathered and contracted
#pragma unroll
            for (int i = 0; i < PPG; ++i) nxt[i] = dcn_load_point(offset_n, mask_n, v + 1, plane, tile.at[i]);
        }
        for (int b = 0; b < nblk; ++b) {
            const int c = b * G + j;
            if (c >= Cg4) break;
            float4 s[PPG];
#pragma unroll
            for (int i = 0; i < PPG; ++i) {
                const float4 a = dcn_corner4(img + row[i][0] + c, ok[i][0]), bb = dcn_corner4(img + row[i][1] + c, ok[i][1]);
                const float4 e = dcn_corner4(img + row[i][2] + c, ok[i][2]), f = dcn_corner4(img + row[i][3] + c, ok[i][3]);
                s[i].x = fw[i][0] * a.x + fw[i][1] * bb.x + fw[i][2] * e.x + fw[i][3] * f.x;
                s[i].y = fw[i][0] * a.y + fw[i][1] * bb.y + fw[i][2] * e.y + fw[i][3] * f.y;
                s[i].z = fw[i][0] * a.z + fw[i][1] * bb.z + fw[i][2] * e.z + fw[i][3] * f.z;
                s[i].w = fw[i][0] * a.w + fw[i][1] * bb.w + fw[i][2] * e.w + fw[i][3] * f.w;
            }
            const float4 *wk = wp + ((long long)(v * nblk + b) * COUT) * G + j;
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const float4 w4 = __ldg(wk + co * G);
#pragma unroll
                for (int i = 0; i < PPG; ++i)
                    acc[i][co] = fmaf(s[i].x, w4.x, fmaf(s[i].y, w4.y, fmaf(s[i].z, w4.z, fmaf(s[i].w, w4.w, acc[i][co]))));
            }
        }
        if (++k == K) k = 0, ++grp;
    }
#pragma unroll
    for (int i = 0; i < PPG; ++i) {
        dcn_group_sum<COUT, G>(acc[i], j);
        if (!tile.live[i]) continue;
        float *o = out + ((long long)tile.n * plane + tile.at[i]) * COUT;
        if (COUT >= G) {
            constexpr int PER = COUT >= G ? COUT / G : 1;
#pragma unroll
            for (int q = 0; q < PER; ++q) o[j * PER + q] = acc[i][q] + (bias ? bias[j * PER + q] : 0.f);
        } else if (j < COUT) {
            float mine = acc[i][0];
#pragma unroll
            for (int q = 1; q < COUT; ++q) mine = j == q ? acc[i][q] : mine;
            o[j] = mine + (bias ? bias[j] : 0.f);
        }
    }
}

// Backward of the fused form with respect to the data: grad_cols is never materialised.  Per (pixel, k) the lane
// forms its slice of the column gradient on the fly, gc[c] = sum_co grad_out[pixel][co] * weight[co][c][k], and uses it
// exactly like dcn_col2im_kernel uses grad_cols: corner dot products -> grad_offset / grad_mask, 16-byte vector
// reductions -> grad_input.  The weight gradient (cols^T x grad_out) is computed by the caller from recomputed columns.
template <int COUT, int G, int PPG, bool DET = false>
__global__ void __launch_bounds__(256, 2) dcn_fused_bwd_kernel(const float *__restrict__ input, const float *__restrict__ offset,
                                                            const float *__restrict__ mask, const float4 *__restrict__ wp,
                                                            const float *__restrict__ grad_out /* (pixels, COUT) */,
                                                            float *__restrict__ grad_input, float *__restrict__ grad_offset,
                                                            float *__restrict__ grad_mask, DetScale det, DcnDims d, int n_base)
{
    const DcnTile<G, PPG> tile(d, n_base);
    if (!tile.row_live) return;
    const int j = tile.j;
    const int K = d.kh * d.kw, GK = d.og * K, C4 = d.C / 4, Cg4 = C4 / d.og, nblk = (Cg4 + G - 1) / G;
    const long long plane = (long long)d.Ho * d.Wo;
    const float4 *img = reinterpret_cast<const float4 *>(input + (long long)tile.n * d.H * d.W * d.C);
    float *gimg = grad_input ? grad_input + (long long)tile.n * d.H * d.W * d.C : nullptr;
    long long *gacc = nullptr;
    float det_sh = 0.f;
    if constexpr (DET) {
        gacc = det.acc + (long long)tile.n * d.H * d.W * d.C;
        det_sh = dcn_det_scale(det, kDcnDetFactorsFused);
    }
    const float *offset_n = offset + (long long)tile.n * 2 * GK * plane;
    const float *mask_n = mask ? mask + (long long)tile.n * GK * plane : nullptr;
    float *goff_n = grad_offset + (long long)tile.n * 2 * GK * plane;
    float *gmask_n = grad_mask ? grad_mask + (long long)tile.n * GK * plane : nullptr;
    float g[PPG][COUT];
#pragma unroll
    for (int i = 0; i < PPG; ++i) {
        const float *go = grad_out + ((long long)tile.n * plane + tile.at[i]) * COUT;
#pragma unroll
        for (int co = 0; co < COUT; ++co) g[i][co] = __ldg(go + co);
    }
    DcnPoint nxt[PPG];
#pragma unroll
    for (int i = 0; i < PPG; ++i) nxt[i] = dcn_load_point(offset_n, mask_n, 0, plane, tile.at[i]);
    for (int v = 0, grp = 0, k = 0; v < GK; ++v) {      // virtual positions, as in dcn_fused_fwd_kernel
        const int ky = k / d.kw, kx = k - ky * d.kw, cb = grp * Cg4;
        DcnTap<float> t[PPG];
        float fw[PPG][4], m[PPG], A[PPG][4];
#pragma unroll
        for (int i = 0; i < PPG; ++i) {
            const float h = (float)(tile.ho * d.sh - d.ph + ky * d.dh) + nxt[i].oh;
            const float w = (float)(tile.wo[i] * d.sw - d.pw + kx * d.dw) + nxt[i].ow;
            t[i] = dcn_tap(h, w, d.H, d.W);
            m[i] = nxt[i].m;
#pragma unroll
            for (int q = 0; q < 4; ++q) fw[i][q] = m[i] * t[i].w[q], A[i][q] = 0.f;
        }
        if (v + 1 < GK) {
#pragma unroll
            for (int i = 0; i < PPG; ++i) nxt[i] = dcn_load_point(offset_n, mask_n, v + 1, plane, tile.at[i]);
        }
        for (int b = 0; b < nblk; ++b) {
            const int cl = b * G + j;
            if (cl >= Cg4) break;
            const int c = cb + cl;
            float4 corner[PPG][4];
#pragma unroll
            for (int i = 0; i < PPG; ++i)
#pragma unroll
                for (int q = 0; q < 4; ++q) corner[i][q] = __ldg(img + (long long)t[i].row[q] * C4 + c);
            const float4 *wk = wp + ((long long)(v * nblk + b) * COUT) * G + j;
            float4 gc[PPG];
#pragma unroll
            for (int i = 0; i < PPG; ++i) gc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const float4 w4 = __ldg(wk + co * G);
#pragma unroll
                for (int i = 0; i < PPG; ++i) {
                    gc[i].x = fmaf(g[i][co], w4.x, gc[i].x);
                    gc[i].y = fmaf(g[i][co], w4.y, gc[i].y);
                    gc[i].z = fmaf(g[i][co], w4.z, gc[i].z);
                    gc[i].w = fmaf(g[i][co], w4.w, gc[i].w);
                }
            }
#pragma unroll
            for (int i = 0; i < PPG; ++i) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 r = corner[i][q];
                    A[i][q] += gc[i].x * r.x + gc[i].y * r.y + gc[i].z * r.z + gc[i].w * r.w;
                    const float f = fw[i][q];
                    if constexpr (DET) {
                        if (tile.live[i] && f != 0.f)
                            det_add4<1>(gacc + ((long long)t[i].row[q] * C4 + c) * 4, det_sh, f * gc[i].x, f * gc[i].y, f * gc[i].z, f * gc[i].w);
                    } else if (gimg && tile.live[i] && f != 0.f)
                        dcn_red_add_f4(gimg + ((long long)t[i].row[q] * C4 + c) * 4, f * gc[i].x, f * gc[i].y, f * gc[i].z, f * gc[i].w);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < PPG; ++i) {
#pragma unroll
            for (int o = G / 2; o >= 1; o >>= 1)
#pragma unroll
                for (int q = 0; q < 4; ++q) A[i][q] += __shfl_xor_sync(0xffffffffu, A[i][q], o, G);
            if (tile.live[i] && j == 0) {
                // outside corners carry garbage from their clamped rows: zero them like the zero padding does
                const float A0 = t[i].ok[0] ? A[i][0] : 0.f, A1 = t[i].ok[1] ? A[i][1] : 0.f;
                const float A2 = t[i].ok[2] ? A[i][2] : 0.f, A3 = t[i].ok[3] ? A[i][3] : 0.f;
                const float val = t[i].hh * (t[i].hw * A0 + t[i].lw * A1) + t[i].lh * (t[i].hw * A2 + t[i].lw * A3);
                const float gh = t[i].hw * (A2 - A0) + t[i].lw * (A3 - A1);
                const float gw = t[i].hh * (A1 - A0) + t[i].lh * (A3 - A2);
                goff_n[(2 * v) * plane + tile.at[i]] = t[i].inside ? m[i] * gh : 0.f;
                goff_n[(2 * v + 1) * plane + tile.at[i]] = t[i].inside ? m[i] * gw : 0.f;
                if (gmask_n) gmask_n[v * plane + tile.at[i]] = t[i].inside ? val : 0.f;
            }
        }
        if (++k == K) k = 0, ++grp;
    }
}

// =====================================================================================================================
// Fused forward with the weights in CONSTANT memory (layers with 16, 32, 48 or 64 output channels and kh*kw*C <= 1024).
//
// The lane-group kernel above fetches a float4 of weights per lane for every 4 (x PPG) multiply-adds: the register-file
// delivery of those loads (4 data-pipe wavefronts per LDG.128, broadcast or not) costs more than the arithmetic they
// feed.  Here the contraction is turned around: a THREAD owns one output pixel and 16 output channels, so the weight of
// (k, c, co) is the same for every lane of the warp and comes straight out of the constant bank as an operand of the
// FFMA -- no load instruction, no data-pipe traffic.  A block owns a tile of 8 x 32 output pixels and alternates, per
// kernel position k:
//   gather      groups of 8 lanes interpolate the C channels of one (pixel, k) each -- coalesced 16-byte gathers exactly
//               like dcn_im2col_kernel -- and park them in shared memory as cols_s[c][pixel] (row stride 257: the 32
//               lanes of a warp hit 32 different banks on the way in, consecutive pixels on the way out);
//   contract    thread p: acc[co] += cols_s[c][p] * W[k][c][co] for all c, 16 FFMAs per shared-memory word.
// Several blocks per SM overlap one block's gathers with another's arithmetic.  Output channels beyond 16 are served by
// further launches (one 16-channel tile of the weights in the constant bank at a time).
// =====================================================================================================================
constexpr int kDcnConstFloats = 16384;                 // 64 KB
__constant__ __align__(16) float dcn_cw[kDcnConstFloats];            // [k][c][16] of the current 16-channel tile
constexpr int kDcnCTileW = 32, kDcnCTileH = 8, kDcnCStride = kDcnCTileW * kDcnCTileH + 1;
constexpr int kDcnCOutside = -0x7fffffff - 1;         // gather record of a pixel outside the output plane

// packed layout for this form: wc[((t * K + k) * C + c) * CT + q] = weight[CT t + q][c][k], CT = output channels per thread
__global__ void dcn_pack_weight_const_kernel(const float *__restrict__ w /* (Cout, C, K) */, float *__restrict__ wc, int cout,
                                             int C, int K, int CT)
{
    const int total = cout * C * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int q = i % CT;
        int r = i / CT;
        const int c = r % C;
        r /= C;
        const int k = r % K, t = r / K;
        wc[i] = w[((long long)(CT * t + q) * C + c) * K + k];
    }
}

// One launch covers kernel positions [k0, k1) for output channels [co0, co0 + CT); the constant bank holds
// W[k0..k1)[c][CT].  k0 > 0: the partial sums of the earlier positions are read back from `out` (layers whose weights
// exceed the bank are served by several launches over k; the gathers are not repeated).
template <int C, int CT>
__global__ void __launch_bounds__(256, CT == 16 ? 3 : 2)
    dcn_fusedc_fwd_kernel(const float *__restrict__ input, const float *__restrict__ offset, const float *__restrict__ mask,
                          const float *__restrict__ bias, float *__restrict__ out, DcnDims d, int n_base, int cout, int co0,
                          int k0, int k1)
{
    extern __shared__ float4 dcn_smem4[];
    float *cols_s = reinterpret_cast<float *>(dcn_smem4);                    // [C][kDcnCStride]
    float4 *rec_f = dcn_smem4 + (C * kDcnCStride + 3) / 4;                   // [8 warps][32 taps] corner factors
    int4 *rec_r = reinterpret_cast<int4 *>(rec_f + 256);                     // [8 warps][32 taps] corner rows (x C/4)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, j = lane & 7, grp = lane >> 3;
    const int n = n_base + (int)blockIdx.z;
    const int ty0 = (int)blockIdx.y * kDcnCTileH, tx0 = (int)blockIdx.x * kDcnCTileW;
    constexpr int C4 = C / 4, nblk = (C4 + 7) / 8;
    const int K = d.kh * d.kw;
    const long long plane = (long long)d.Ho * d.Wo;
    const float4 *img = reinterpret_cast<const float4 *>(input + (long long)n * d.H * d.W * C);
    const float *offset_n = offset + (long long)n * 2 * K * plane;
    const float *mask_n = mask ? mask + (long long)n * K * plane : nullptr;

    // gather role: the group (warp, grp) serves tile column warp*4+grp, rows it = 0..7.  The 32 taps of a warp and
    // kernel position are prepared ONCE, one per lane (lane = grp*8 + row), and handed to the groups through shared
    // memory as two 16-byte records (corner factors with the mask folded in; corner rows).
    const int gx = tx0 + warp * 4 + grp;
    const int my_y = ty0 + j;
    const bool my_live = my_y < d.Ho && gx < d.Wo;
    const long long my_at = (long long)min(my_y, d.Ho - 1) * d.Wo + min(gx, d.Wo - 1);
    // contract role: thread owns tile pixel threadIdx.x = row warp, column lane
    const int oy = ty0 + warp, ox = tx0 + lane;
    const bool out_live = oy < d.Ho && ox < d.Wo;
    float *o = out + ((long long)n * plane + (long long)min(oy, d.Ho - 1) * d.Wo + min(ox, d.Wo - 1)) * cout + co0;
    float acc[CT];
    if (k0 > 0 && out_live) {
#pragma unroll
        for (int q = 0; q < CT / 4; ++q) {
            const float4 v = reinterpret_cast<const float4 *>(o)[q];
            acc[4 * q] = v.x, acc[4 * q + 1] = v.y, acc[4 * q + 2] = v.z, acc[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < CT; ++q) acc[q] = 0.f;
    }

    DcnPoint nxt = dcn_load_point(offset_n, mask_n, k0, plane, my_at);
    int wbase = 0;     // its own induction variable: untouched by the divergent gather code, it stays in a uniform register
    for (int k = k0; k < k1; ++k, wbase += C * (CT / 4)) {
        const int ky = k / d.kw, kx = k - ky * d.kw;
        {
            const float h = (float)(my_y * d.sh - d.ph + ky * d.dh) + nxt.oh;
            const float w = (float)(gx * d.sw - d.pw + kx * d.dw) + nxt.ow;
            const DcnTap<float> t = dcn_tap(h, w, d.H, d.W);
            const float m = nxt.m;
            if (k + 1 < k1) nxt = dcn_load_point(offset_n, mask_n, k + 1, plane, my_at);
            rec_f[warp * 32 + lane] = make_float4(m * t.w[0], m * t.w[1], m * t.w[2], m * t.w[3]);
            // corner rows; -1 = corner outside the map (value 0, never read), kDcnCOutside = pixel outside the plane
            const int r0 = t.ok[0] ? t.row[0] * C4 : -1;
            rec_r[warp * 32 + lane] = make_int4(my_live ? r0 : kDcnCOutside, t.ok[1] ? t.row[1] * C4 : -1,
                                                t.ok[2] ? t.row[2] * C4 : -1, t.ok[3] ? t.row[3] * C4 : -1);
        }
        if (k > k0) __syncthreads();                     // everyone is done reading the previous position's columns
        else __syncwarp();
#pragma unroll 2
        for (int it = 0; it < kDcnCTileH; ++it) {
            const int4 rr = rec_r[warp * 32 + grp * 8 + it];
            if (rr.x == kDcnCOutside) continue;          // pixel outside the plane: its columns are never read
            const float4 ff = rec_f[warp * 32 + grp * 8 + it];
            const bool ok0 = rr.x >= 0, ok1 = rr.y >= 0, ok2 = rr.z >= 0, ok3 = rr.w >= 0;
            const float4 *r0 = img + max(rr.x, 0), *r1 = img + max(rr.y, 0), *r2 = img + max(rr.z, 0), *r3 = img + max(rr.w, 0);
            float *dst = cols_s + it * 32 + warp * 4 + grp;
#pragma unroll
            for (int b = 0; b < nblk; ++b) {
                const int c = b * 8 + j;
                if (c >= C4) break;
                const float4 a = dcn_corner4(r0 + c, ok0), bb = dcn_corner4(r1 + c, ok1);
                const float4 e = dcn_corner4(r2 + c, ok2), f = dcn_corner4(r3 + c, ok3);
                dst[(4 * c + 0) * kDcnCStride] = ff.x * a.x + ff.y * bb.x + ff.z * e.x + ff.w * f.x;
                dst[(4 * c + 1) * kDcnCStride] = ff.x * a.y + ff.y * bb.y + ff.z * e.y + ff.w * f.y;
                dst[(4 * c + 2) * kDcnCStride] = ff.x * a.z + ff.y * bb.z + ff.z * e.z + ff.w * f.z;
                dst[(4 * c + 3) * kDcnCStride] = ff.x * a.w + ff.y * bb.w + ff.z * e.w + ff.w * f.w;
            }
        }
        __syncthreads();
        // C is a compile-time constant and the loop is unrolled: the weight addresses are (uniform base + immediate), the
        // compiler fetches them with uniform constant loads (LDCU into uniform registers) and feeds the FFMAs from
        // there -- no per-thread load, nothing on the L1 data pipe
        const float *col = cols_s + threadIdx.x;
        const float4 *wk = reinterpret_cast<const float4 *>(dcn_cw) + wbase;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float v = col[c * kDcnCStride];
#pragma unroll
            for (int q = 0; q < CT / 4; ++q) {
                const float4 w4 = wk[c * (CT / 4) + q];
                acc[4 * q + 0] = fmaf(v, w4.x, acc[4 * q + 0]);
                acc[4 * q + 1] = fmaf(v, w4.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(v, w4.z, acc[4 * q + 2]);
                acc[4 * q + 3] = fmaf(v, w4.w, acc[4 * q + 3]);
            }
        }
    }
    if (!out_live) return;
    const bool last = k1 == K;
#pragma unroll
    for (int q = 0; q < CT / 4; ++q) {
        float4 v = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
        if (bias && last) {
            v.x += bias[co0 + 4 * q], v.y += bias[co0 + 4 * q + 1], v.z += bias[co0 + 4 * q + 2], v.w += bias[co0 + 4 * q + 3];
        }
        reinterpret_cast<float4 *>(o)[q] = v;
    }
}

// =====================================================================================================================
// Weight gradient without the column matrix (narrow layers: C = 4 * G channels, COUT <= 16):
//     grad_w[co][k][c] = sum over output pixels of  mask * bilinear(input[.., c])  *  grad_out[pixel][co]
// torchvision (and the im2col route here) writes the columns -- K x the input, 995 MB for 60 instances at 90 x 160 x 32 --
// and multiplies them with grad_out^T in a GEMM whose reduction dimension is the pixel count.  Here a lane group of G
// lanes owns kernel position k = blockIdx.y and a strided run of output pixels; a lane gathers and interpolates its four
// channels of a pixel exactly like dcn_im2col_kernel, multiplies them with the pixel's COUT output gradients (one
// broadcast load per four) and keeps the 4 x COUT partial sums in registers for the whole run.  The groups of a block are
// then added up (shuffles inside a warp, shared memory across warps) and ONE atomic per (k, c, co) and block goes to
// grad_w.  Nothing of column size exists at any point.
// =====================================================================================================================
template <int COUT, int G>
__global__ void __launch_bounds__(256) dcn_wgrad_kernel(const float *__restrict__ input, const float *__restrict__ offset,
                                                        const float *__restrict__ mask, const float *__restrict__ grad_out,
                                                        float *__restrict__ grad_w, DcnDims d, int n_base, int run)
{
    constexpr int GPB = 256 / G;                    // lane groups per block
    constexpr int C = 4 * G;
    __shared__ float red_s[8][C * COUT];
    const int j = threadIdx.x % G, grp = threadIdx.x / G, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = n_base + (int)blockIdx.z, k = (int)blockIdx.y;
    const int plane = d.Ho * d.Wo;
    const float4 *img = reinterpret_cast<const float4 *>(input + (long long)n * d.H * d.W * C);
    float acc[4][COUT];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int co = 0; co < COUT; ++co) acc[i][co] = 0.f;

    // pixel of iteration r: consecutive groups take consecutive pixels (coalesced offsets, shared gather neighbourhoods);
    // the sampling point of iteration r + 1 is loaded while iteration r gathers (one dependent latency less per pixel)
    const int K_ = d.kh * d.kw;
    const float *off_h = offset + ((long long)n * 2 * K_ + 2 * k) * plane, *off_w = off_h + plane;
    const float *msk = mask ? mask + ((long long)n * K_ + k) * plane : nullptr;
    const int ky = k / d.kw, kx = k - ky * d.kw;
    const int pp0 = (int)blockIdx.x * run * GPB + grp;
    float n_oh = 0.f, n_ow = 0.f, n_m = 1.f;
    if (pp0 < plane) {
        n_oh = __ldg(off_h + pp0);
        n_ow = __ldg(off_w + pp0);
        if (msk) n_m = __ldg(msk + pp0);
    }
    for (int r = 0; r < run; ++r) {
        const int pp = pp0 + r * GPB;
        const float c_oh = n_oh, c_ow = n_ow, m = n_m;
        if (r + 1 < run && pp + GPB < plane) {
            n_oh = __ldg(off_h + pp + GPB);
            n_ow = __ldg(off_w + pp + GPB);
            if (msk) n_m = __ldg(msk + pp + GPB);
        }
        if (pp < plane) {
            const DcnTapId id = dcn_tap_id(pp, n, k, d);
            const float h = (float)(id.ho * d.sh - d.ph + ky * d.dh) + c_oh;
            const float w = (float)(id.wo * d.sw - d.pw + kx * d.dw) + c_ow;
            const DcnTap<float> t = dcn_tap(h, w, d.H, d.W);
            const float f0 = m * t.w[0], f1 = m * t.w[1], f2 = m * t.w[2], f3 = m * t.w[3];
            const float4 a = dcn_corner4(img + (long long)t.row[0] * G + j, t.ok[0]);
            const float4 b = dcn_corner4(img + (long long)t.row[1] * G + j, t.ok[1]);
            const float4 e = dcn_corner4(img + (long long)t.row[2] * G + j, t.ok[2]);
            const float4 f = dcn_corner4(img + (long long)t.row[3] * G + j, t.ok[3]);
            float v[4];
            v[0] = f0 * a.x + f1 * b.x + f2 * e.x + f3 * f.x;
            v[1] = f0 * a.y + f1 * b.y + f2 * e.y + f3 * f.y;
            v[2] = f0 * a.z + f1 * b.z + f2 * e.z + f3 * f.z;
            v[3] = f0 * a.w + f1 * b.w + f2 * e.w + f3 * f.w;
            const float *g = grad_out + id.pixel * COUT;
            if (COUT % 4 == 0) {
#pragma unroll
                for (int q = 0; q < COUT / 4; ++q) {
                    const float4 gq = __ldg(reinterpret_cast<const float4 *>(g) + q);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        acc[i][4 * q + 0] = fmaf(v[i], gq.x, acc[i][4 * q + 0]);
                        acc[i][4 * q + 1] = fmaf(v[i], gq.y, acc[i][4 * q + 1]);
                        acc[i][4 * q + 2] = fmaf(v[i], gq.z, acc[i][4 * q + 2]);
                        acc[i][4 * q + 3] = fmaf(v[i], gq.w, acc[i][4 * q + 3]);
                    }
                }
            } else {
#pragma unroll
                for (int co = 0; co < COUT; ++co) {
                    const float gc = __ldg(g + co);
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[i][co] = fmaf(v[i], gc, acc[i][co]);
                }
            }
        }
    }
    // groups of a warp (same lane index j, 32 / G of them) by xor shuffles; every lane ends up with the warp's sum
#pragma unroll
    for (int o = G; o < 32; o <<= 1)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int co = 0; co < COUT; ++co) acc[i][co] += __shfl_xor_sync(0xffffffffu, acc[i][co], o);
    if (lane < G) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int co = 0; co < COUT; ++co) red_s[warp][co * C + 4 * j + i] = acc[i][co];
    }
    __syncthreads();
    const int K = d.kh * d.kw;
    for (int idx = threadIdx.x; idx < C * COUT; idx += 256) {
        float sum = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) sum += red_s[wv][idx];
        const int co = idx / C, c = idx - co * C;
        atomicAdd(grad_w + ((long long)co * K + k) * C + c, sum);
    }
}

}  // namespace devis
