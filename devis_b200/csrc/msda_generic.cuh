// msda_generic.cuh -- any-channel-count, any-dtype (fp32 / fp64 / bf16 / fp16) kernels.
//
// The reference instantiates its kernels for float and double and for every channel count
// (cuda/ms_deform_attn_cuda.cu:64,134; the backward picks one of six kernels by D,
// cuda/ms_deform_im2col_cuda.cuh:975-1320; test.py:83 sweeps D = 30,32,64,71,1025,2048,3096 in
// double).  The grouped-lane kernels in msda_fwd.cuh / msda_bwd.cuh cover the shapes DeVIS uses
// (D = 32, 16); everything else lands here: one WARP per (query, head), lanes stride the channels,
// so loads are coalesced for any D, the per-tap channel reduction is a warp shuffle tree (no shared
// memory, no barriers, no serial thread-0 loop), and a single kernel replaces the reference's six.
// Arithmetic follows the reference's per-channel formulation (cuh:33-84, 87-159) in the compute type.
#pragma once
#include "msda_common.cuh"

namespace devis {

template <typename T> struct Scalar;
template <> struct Scalar<float> {
    using C = float;   // compute / location / gradient type
    static __device__ __forceinline__ float load(const void *p, size_t i) { return __ldg(reinterpret_cast<const float *>(p) + i); }
    static __device__ __forceinline__ void store(void *p, size_t i, float v) { reinterpret_cast<float *>(p)[i] = v; }
    static __device__ __forceinline__ float coord(float l, int n) { return __fadd_rn(__fmul_rn(l, (float)n), -0.5f); }
};
template <> struct Scalar<double> {
    using C = double;
    static __device__ __forceinline__ double load(const void *p, size_t i) { return __ldg(reinterpret_cast<const double *>(p) + i); }
    static __device__ __forceinline__ void store(void *p, size_t i, double v) { reinterpret_cast<double *>(p)[i] = v; }
    static __device__ __forceinline__ double coord(double l, int n) { return __dadd_rn(__dmul_rn(l, (double)n), -0.5); }
};
template <> struct Scalar<__nv_bfloat16> {
    using C = float;
    static __device__ __forceinline__ float load(const void *p, size_t i)
    {
        return __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(p)[i]);
    }
    static __device__ __forceinline__ void store(void *p, size_t i, float v)
    {
        reinterpret_cast<__nv_bfloat16 *>(p)[i] = __float2bfloat16_rn(v);
    }
    static __device__ __forceinline__ float coord(float l, int n) { return __fadd_rn(__fmul_rn(l, (float)n), -0.5f); }
};

template <> struct Scalar<__half> {
    using C = float;
    static __device__ __forceinline__ float load(const void *p, size_t i) { return __half2float(reinterpret_cast<const __half *>(p)[i]); }
    static __device__ __forceinline__ void store(void *p, size_t i, float v) { reinterpret_cast<__half *>(p)[i] = __float2half_rn(v); }
    static __device__ __forceinline__ float coord(float l, int n) { return __fadd_rn(__fmul_rn(l, (float)n), -0.5f); }
};

template <typename C>
struct TapC {
    C lh, lw, hh, hw;
    long long r00, r01, r10, r11;  // value rows of the 4 corners (only meaningful where ok bit set)
    unsigned ok;
};

template <typename T>
__device__ __forceinline__ TapC<typename Scalar<T>::C> tap_generic(typename Scalar<T>::C x, typename Scalar<T>::C y,
                                                                    const int4 sl)
{
    using C = typename Scalar<T>::C;
    TapC<C> g;
    const int H = sl.x, W = sl.y;
    const C h = Scalar<T>::coord(y, H), w = Scalar<T>::coord(x, W);
    const bool inb = h > (C)-1 && w > (C)-1 && h < (C)H && w < (C)W;
    const C hf = floor(h), wf = floor(w);
    const int h0 = inb ? (int)hf : 0, w0 = inb ? (int)wf : 0;
    g.lh = h - hf;
    g.lw = w - wf;
    g.hh = (C)1 - g.lh;
    g.hw = (C)1 - g.lw;
    const bool t_ok = h0 >= 0, b_ok = h0 + 1 <= H - 1, l_ok = w0 >= 0, r_ok = w0 + 1 <= W - 1;
    g.ok = inb ? ((t_ok && l_ok) | ((t_ok && r_ok) << 1) | ((b_ok && l_ok) << 2) | ((b_ok && r_ok) << 3)) : 0u;
    const long long base = (long long)sl.z + (long long)h0 * W + w0;
    g.r00 = base;
    g.r01 = base + 1;
    g.r10 = base + W;
    g.r11 = base + W + 1;
    return g;
}

// ---------------------------------------------------------------------------------------------
template <typename T, class SlotSrc>
__global__ void __launch_bounds__(128) msda_fwd_generic_kernel(const FwdArgs<SlotSrc> a)
{
    using C = typename Scalar<T>::C;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);

    const int M = a.d.M, D = a.d.D, Lq = a.d.Lq;
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long long)Lq * M) return;
    const int q = (int)(item / M), m = (int)(item - (long long)q * M);
    const size_t row = ((size_t)outer * Lq + q) * M + m;
    const size_t ps = (size_t)M * D;

    for (int c0 = 0; c0 < D; c0 += 32) {
        const int c = c0 + lane;
        const bool clive = c < D;
        const size_t ch = (size_t)m * D + (clive ? c : 0);
        C col = 0;
        int slot_base = 0;
        for (int sg = 0; sg < a.n_seg; ++sg) {
            const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P;
            const C *loc = reinterpret_cast<const C *>(a.seg[sg].loc) + row * K * 2;
            const C *aw = reinterpret_cast<const C *>(a.seg[sg].aw) + row * K;
            for (int k = 0; k < K; ++k) {
                const TapC<C> g = tap_generic<T>(__ldg(loc + 2 * k), __ldg(loc + 2 * k + 1), s_slot[slot_base + k / P]);
                if (g.ok == 0u || !clive) continue;
                const C v00 = (g.ok & 1u) ? Scalar<T>::load(a.value, g.r00 * ps + ch) : (C)0;
                const C v01 = (g.ok & 2u) ? Scalar<T>::load(a.value, g.r01 * ps + ch) : (C)0;
                const C v10 = (g.ok & 4u) ? Scalar<T>::load(a.value, g.r10 * ps + ch) : (C)0;
                const C v11 = (g.ok & 8u) ? Scalar<T>::load(a.value, g.r11 * ps + ch) : (C)0;
                const C val = g.hh * g.hw * v00 + g.hh * g.lw * v01 + g.lh * g.hw * v10 + g.lh * g.lw * v11;
                col += val * __ldg(aw + k);
            }
            slot_base += a.seg[sg].n_slots;
        }
        if (clive) Scalar<T>::store(a.out, row * D + c, col);
    }
}

// GV: grad_value element type (float, or double for fp64)
template <typename T, class SlotSrc>
__global__ void __launch_bounds__(128) msda_bwd_generic_kernel(const BwdArgs<SlotSrc> a)
{
    using C = typename Scalar<T>::C;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);

    const int M = a.d.M, D = a.d.D, Lq = a.d.Lq;
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long long)Lq * M) return;  // whole warps leave together
    const int q = (int)(item / M), m = (int)(item - (long long)q * M);
    const size_t row = ((size_t)outer * Lq + q) * M + m;
    const size_t ps = (size_t)M * D;
    C *gv = reinterpret_cast<C *>(a.grad_value);  // float for fp32/bf16/fp16, double for fp64
    long long *det = a.det.acc;                    // deterministic fixed-point accumulators (never with fp64)
    const float det_sh = det ? ldexpf(1.f, kDetFracBits - det_exponent(a.det.max_bits)) : 0.f;
    auto scatter = [&](long long r, C v) {
        if (det) atomicAdd(reinterpret_cast<unsigned long long *>(det) + r, (unsigned long long)__float2ll_rn((float)v * det_sh));
        else if (gv) atomicAdd(gv + r, v);
    };

    for (int c0 = 0; c0 < D; c0 += 32) {
        const int c = c0 + lane;
        const bool clive = c < D;
        const size_t ch = (size_t)m * D + (clive ? c : 0);
        const C top = clive ? Scalar<T>::load(a.grad_out, row * D + c) : (C)0;
        int slot_base = 0;
        for (int sg = 0; sg < a.n_seg; ++sg) {
            const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P;
            const C *loc = reinterpret_cast<const C *>(a.seg[sg].loc) + row * K * 2;
            const C *aw = reinterpret_cast<const C *>(a.seg[sg].aw) + row * K;
            C *gloc = reinterpret_cast<C *>(a.seg[sg].grad_loc) + row * K * 2;
            C *gaw = reinterpret_cast<C *>(a.seg[sg].grad_aw) + row * K;
            for (int k = 0; k < K; ++k) {
                const int4 sl = s_slot[slot_base + k / P];
                const TapC<C> g = tap_generic<T>(__ldg(loc + 2 * k), __ldg(loc + 2 * k + 1), sl);
                const C attn = __ldg(aw + k);
                C p_a = 0, p_x = 0, p_y = 0;
                if (g.ok != 0u && clive) {
                    const C tv = top * attn;
                    C gh = 0, gw = 0, v00 = 0, v01 = 0, v10 = 0, v11 = 0;
                    if (g.ok & 1u) {
                        v00 = Scalar<T>::load(a.value, g.r00 * ps + ch);
                        gh -= g.hw * v00;
                        gw -= g.hh * v00;
                        scatter(g.r00 * ps + ch, g.hh * g.hw * tv);
                    }
                    if (g.ok & 2u) {
                        v01 = Scalar<T>::load(a.value, g.r01 * ps + ch);
                        gh -= g.lw * v01;
                        gw += g.hh * v01;
                        scatter(g.r01 * ps + ch, g.hh * g.lw * tv);
                    }
                    if (g.ok & 4u) {
                        v10 = Scalar<T>::load(a.value, g.r10 * ps + ch);
                        gh += g.hw * v10;
                        gw -= g.lh * v10;
                        scatter(g.r10 * ps + ch, g.lh * g.hw * tv);
                    }
                    if (g.ok & 8u) {
                        v11 = Scalar<T>::load(a.value, g.r11 * ps + ch);
                        gh += g.lw * v11;
                        gw += g.lh * v11;
                        scatter(g.r11 * ps + ch, g.lh * g.lw * tv);
                    }
                    const C val = g.hh * g.hw * v00 + g.hh * g.lw * v01 + g.lh * g.hw * v10 + g.lh * g.lw * v11;
                    p_a = top * val;
                    p_x = (C)sl.y * gw * tv;
                    p_y = (C)sl.x * gh * tv;
                }
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) {
                    p_a += __shfl_xor_sync(0xffffffffu, p_a, o);
                    p_x += __shfl_xor_sync(0xffffffffu, p_x, o);
                    p_y += __shfl_xor_sync(0xffffffffu, p_y, o);
                }
                if (lane == 0) {  // same lane revisits the same address for later channel chunks
                    if (c0 == 0) {
                        gaw[k] = p_a;
                        gloc[2 * k] = p_x;
                        gloc[2 * k + 1] = p_y;
                    } else {
                        gaw[k] += p_a;
                        gloc[2 * k] += p_x;
                        gloc[2 * k + 1] += p_y;
                    }
                }
            }
            slot_base += a.seg[sg].n_slots;
        }
    }
}

}  // namespace devis
