// msda_bwd.cuh -- backward of multi-scale deformable attention, grouped-lane kernel for sm_100a.
//
// Replaces ms_deformable_col2im_gpu_kernel_shm_blocksize_aware_reduce_v1<32>
// (cuda/ms_deform_im2col_cuda.cuh:301-403) and ms_deform_attn_col2im_bilinear (:87-159), where a
// one-warp block owns one (query, head), every lane redoes the tap geometry, each tap costs two
// __syncthreads() plus a serial 32-element reduction on thread 0, and grad_value is scattered with
// 4 scalar atomics per (tap, channel).
//
// Here (same work split as msda_fwd.cuh: LPG lanes x 4 channels per (query, head), tap geometry
// prepared by one lane per tap and handed over through the shared-memory TapExchange):
//   * per tap each lane forms the 4 corner dot products  A_c = sum_ch grad_out[ch] * value_c[ch]
//     over its own 4 channels only (16 FMA); everything else about grad_attn / grad_loc is linear in
//     those four numbers, so it is done AFTER the channel reduction, once per tap, by the lane that
//     prepared the tap:
//         grad_attn = hh*hw*A00 + hh*lw*A01 + lh*hw*A10 + lh*lw*A11
//         grad_x    = W * attn * (hh*(A01-A00) + lh*(A11-A10))
//         grad_y    = H * attn * (hw*(A10-A00) + lw*(A11-A01))
//     (algebraically the sums the reference accumulates per channel at :123-158);
//   * the channel reduction is a reduce-scatter butterfly across the group (LPG taps x 4 numbers in,
//     tap j's 4 totals land on lane j): 3.5 shuffles per tap for LPG=8 instead of 12 for four
//     xor-reductions, no shared memory, no barriers;
//   * grad_value: one 16-byte vector reduction per lane and corner
//     (red.global.add.v4.f32, SASS REDG.E.ADD.F32x4) instead of 4 scalar atomics, skipped for
//     corners with zero weight.  Shared-memory float atomics are CAS loops on sm_100a
//     (ATOMS.CAST.SPIN), which is why the accumulation is not staged in shared memory.
//   * grad_sampling_loc / grad_attn_weight are written exactly once per tap with plain coalesced
//     stores -- no zero-fill pass, no atomics (out-of-range taps write 0 like the reference's zeros()).
#pragma once
#include "msda_common.cuh"

// 3 blocks of 256 threads (6 of 128) per SM caps the kernel at 80 registers; uncapped, ptxas takes 84 - 115 and the
// default 128-thread launch loses a block per SM (1428 -> 1440 us at 256 threads, equal at 128: sweep of round 1f)
#ifndef DEVIS_BWD_MIN_BLOCKS
#define DEVIS_BWD_MIN_BLOCKS 3
#endif

namespace devis {

template <class SlotSrc>
struct BwdArgs {
    const void *value;
    const void *grad_out;
    void *grad_value;   // fp32 accumulation target (also for 16-bit value; bf16 under HALF_ACC); nullptr = skip
    DetScale det;       // deterministic mode: det.acc != nullptr replaces the float reductions
    Segment seg[2];
    int n_seg;
    int n_slots_total;
    SlotSrc src;
    OpDims d;
    const int *q_perm;
};

// d[t][c]: partial sums of tap t, corner c held by this lane.  On return r[c] is the group total of
// corner c for tap j (j = this lane's index in the group).
template <int LPG>
__device__ __forceinline__ void reduce_scatter_taps(float (&d)[LPG][4], int j, float (&r)[4])
{
#pragma unroll
    for (int half = LPG / 2; half >= 1; half >>= 1) {
        const bool upper = (j & half) != 0;
#pragma unroll
        for (int t = 0; t < half; ++t) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float send = upper ? d[t][c] : d[t + half][c];
                const float keep = upper ? d[t + half][c] : d[t][c];
                d[t][c] = keep + __shfl_xor_sync(0xffffffffu, send, half, LPG);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) r[c] = d[0][c];
}

// HALF_ACC (bf16 value only, DEVIS_MSDA_FLAG_BF16_GRAD_VALUE): grad_value is a bf16 tensor laid out like value and
// the scatter uses 8-byte packed reductions (red.global.add.noftz.v2.bf16x2, SASS REDG.E.ADD.BF16x4.RN): a row leaves
// the SM as 2 sectors instead of 4, which is what the backward is bound by (DESIGN.md 3.6).
template <Elem E, int LPG, int QPG, class SlotSrc, bool HALF_ACC = false>
__global__ void __launch_bounds__(256, DEVIS_BWD_MIN_BLOCKS) msda_bwd_kernel(const BwdArgs<SlotSrc> a)
{
    using X = TapExchange<LPG>;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + a.n_slots_total) + (threadIdx.x >> 5) * (2 * X::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x % LPG;
    const int g = (threadIdx.x & 31) / LPG;
    const int grp = threadIdx.x / LPG;
    const int QC = blockDim.x / LPG;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;
    const L2Policy pol = make_l2_policy();

    int q[QPG];
    bool qlive[QPG];
    float4 go[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        const int qi = (qchunk * QPG + i) * QC + grp;
        qlive[i] = qi < Lq;
        q[i] = qlive[i] ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
        go[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (qlive[i]) {
            const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
            if constexpr (E != Elem::F32) go[i] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(a.grad_out) + row * LPG + j);
            else go[i] = ld_stream_f4(reinterpret_cast<const float4 *>(a.grad_out) + row * LPG + j, pol);
        }
    }

    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kQuadBytes;
    // keep the per-lane base as ONE 64-bit register pair: each corner address is then base + u32 offset
    // (IADD3 + IADD3.X) instead of a re-derived IMAD.WIDE chain (5 instructions per address in round 1a)
    asm volatile("" : "+l"(vbase));
    // grad_value is fp32 unless HALF_ACC: 16 bytes per channel quad; offsets published for `value` scale by 16/kQuadBytes
    static_assert(!HALF_ACC || E == Elem::BF16, "bf16 accumulation needs bf16 value");
    constexpr unsigned kGvQuadBytes = HALF_ACC ? 8u : 16u;
    char *gvb = a.grad_value ? reinterpret_cast<char *>(a.grad_value) + (size_t)(m * LPG + j) * kGvQuadBytes : nullptr;
    constexpr unsigned kGvShift = (E != Elem::F32 && !HALF_ACC) ? 1u : 0u;
    // deterministic mode: 8-byte fixed-point accumulators, same row pitch in elements -> offsets scale by
    // 2 * 16 / kQuadBytes; within a (row, head) the channels are permuted (det_add4): lane j starts at word j
    char *detb = a.det.acc ? reinterpret_cast<char *>(a.det.acc) + (size_t)(m * LPG) * 32u + (size_t)j * 8u : nullptr;
    const float det_sh = a.det.acc ? ldexpf(1.f, kDetFracBits - det_exponent(a.det.max_bits)) : 0.f;

    int slot_base = 0, parity = 0;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P, pshift = pow2_shift(P);
        const float *loc = reinterpret_cast<const float *>(a.seg[sg].loc);
        const float *aw = reinterpret_cast<const float *>(a.seg[sg].aw);
        float *gloc = reinterpret_cast<float *>(a.seg[sg].grad_loc);
        float *gaw = reinterpret_cast<float *>(a.seg[sg].grad_aw);
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;
            const bool klive = k < K;
            const int4 sl = s_slot[slot_base + (klive ? div_p(k, P, pshift) : 0)];
#pragma unroll
            for (int i = 0; i < QPG; ++i) {
                const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
                const bool live = klive && qlive[i];
                float2 xy = make_float2(0.f, 0.f);
                float w = 0.f;
                if (live) {
                    xy = ld_stream_f2(reinterpret_cast<const float2 *>(loc + row * K * 2) + k, pol);
                    w = ld_stream_f(aw + row * K + k, pol);
                }
                const TapGeom t = tap_geometry(xy.x, xy.y, sl, live);
                float *buf = xbuf + parity * X::kWordsPerWarpBuf;
                parity ^= 1;
                X::publish(buf, j, g, t, w, rowbytes);
                __syncwarp();

                const float4 gg = go[i];
                float dsum[LPG][4];
#pragma unroll
                for (int jj = 0; jj < LPG; ++jj) {
                    uint4 off;
                    float4 c;
                    X::fetch(buf, jj, g, off, c);
                    float4 v00, v01, v10, v11;
                    if constexpr (E != Elem::F32) {
                        v00 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.x));
                        v01 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.y));
                        v10 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.z));
                        v11 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.w));
                    } else {
                        v00 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.x), pol);
                        v01 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.y), pol);
                        v10 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.z), pol);
                        v11 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.w), pol);
                    }
                    dsum[jj][0] = fmaf(v00.w, gg.w, fmaf(v00.z, gg.z, fmaf(v00.y, gg.y, v00.x * gg.x)));
                    dsum[jj][1] = fmaf(v01.w, gg.w, fmaf(v01.z, gg.z, fmaf(v01.y, gg.y, v01.x * gg.x)));
                    dsum[jj][2] = fmaf(v10.w, gg.w, fmaf(v10.z, gg.z, fmaf(v10.y, gg.y, v10.x * gg.x)));
                    dsum[jj][3] = fmaf(v11.w, gg.w, fmaf(v11.z, gg.z, fmaf(v11.y, gg.y, v11.x * gg.x)));
                    if (detb) {
                        if (c.x != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.x << (kGvShift + 1))), det_sh, c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w);
                        if (c.y != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.y << (kGvShift + 1))), det_sh, c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w);
                        if (c.z != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.z << (kGvShift + 1))), det_sh, c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w);
                        if (c.w != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.w << (kGvShift + 1))), det_sh, c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w);
                    } else if (gvb) {
                        if (c.x != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.x << kGvShift), c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w, pol);
                        if (c.y != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.y << kGvShift), c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w, pol);
                        if (c.z != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.z << kGvShift), c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w, pol);
                        if (c.w != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.w << kGvShift), c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w, pol);
                    }
                }

                float A[4];
                reduce_scatter_taps<LPG>(dsum, j, A);
                if (live) {
                    const bool hit = t.ok != 0u;  // out-of-range taps write the reference's zero fill
                    const float hh = (t.ok & 1u) ? t.hh : 0.f, lh = (t.ok & 2u) ? t.lh : 0.f;
                    const float hw = (t.ok & 4u) ? t.hw : 0.f, lw = (t.ok & 8u) ? t.lw : 0.f;
                    // masked bilinear factors make every term of an outside corner vanish (its A is garbage
                    // from the clamped row): d/dx = sum_rows rowfac * (right*[r_ok] - left*[l_ok]) etc.
                    const float l_in = (t.ok & 4u) ? 1.f : 0.f, r_in = (t.ok & 8u) ? 1.f : 0.f;
                    const float t_in = (t.ok & 1u) ? 1.f : 0.f, b_in = (t.ok & 2u) ? 1.f : 0.f;
                    const float val = hh * (hw * A[0] + lw * A[1]) + lh * (hw * A[2] + lw * A[3]);
                    const float gx = hh * (r_in * A[1] - l_in * A[0]) + lh * (r_in * A[3] - l_in * A[2]);
                    const float gy = hw * (b_in * A[2] - t_in * A[0]) + lw * (b_in * A[3] - t_in * A[1]);
                    st_stream_f(gaw + row * K + k, hit ? val : 0.f, pol);
                    st_stream_f2(reinterpret_cast<float2 *>(gloc + row * K * 2) + k,
                                 hit ? make_float2((float)sl.y * gx * w, (float)sl.x * gy * w) : make_float2(0.f, 0.f), pol);
                }
            }
        }
        slot_base += a.seg[sg].n_slots;
    }
}

}  // namespace devis
