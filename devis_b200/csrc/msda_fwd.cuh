// msda_fwd.cuh -- forward of multi-scale deformable attention, grouped-lane kernel for sm_100a.
//
// Replaces ms_deformable_im2col_gpu_kernel (cuda/ms_deform_im2col_cuda.cuh:237-299), which maps one
// thread to one output channel and therefore recomputes each tap's floor/weights D times and gathers
// with 4-byte loads.  Here:
//   * a GROUP of LPG lanes owns one (query, head); each lane owns 4 consecutive channels, so a value
//     row of one head (D = 4*LPG channels) is fetched by the group as one 16*LPG-byte line
//     (128 B for D=32 fp32): 4 corner loads per tap are 4 fully used L1 wavefronts per warp;
//   * tap geometry is computed ONCE per tap: lane j of the group reads location / weight of tap
//     k0+j (coalesced over the group), does the floor / range test / bilinear weights with the
//     attention weight folded in, and publishes a 32-byte record (4 byte offsets, 4 weight factors)
//     in a per-warp shared-memory exchange; the group then walks the LPG records with two broadcast
//     LDS.128 each (TapExchange in msda_common.cuh; shuffles were measured to cost 3x the L1 wavefronts);
//   * a CTA works on ONE head and QC*QPG queries, and walks slots in order, so that its working set
//     at any time is one (frame, level, head) neighbourhood of value -- the L1/L2 locality that the
//     whole-clip op relies on; QPG queries per group are interleaved (accumulators in registers).
//
// The same kernel serves the per-call op (SlotSrc = DeviceLevels, one segment) and the whole-clip
// temporal op (SlotSrc = ClipTable, two segments, value indexed through the frame table).
#pragma once
#include "msda_common.cuh"

#ifndef DEVIS_FWD_TAP_BATCH
#define DEVIS_FWD_TAP_BATCH 2
#endif
// 3 blocks of 256 threads per SM caps the kernel at 80 registers; without a cap ptxas hoists all 32 corner loads of
// an 8-tap exchange (182 registers, 1 block/SM: 787 us instead of 580 us at the DeVIS shape)
#ifndef DEVIS_FWD_MIN_BLOCKS
#define DEVIS_FWD_MIN_BLOCKS 3
#endif

namespace devis {

template <class SlotSrc>
struct FwdArgs {
    const void *value;
    void *out;
    Segment seg[2];
    int n_seg;
    int n_slots_total;
    SlotSrc src;
    OpDims d;
    const int *q_perm;  // optional query visiting order (length Lq), nullptr = identity
};

template <Elem E, int LPG, int QPG, class SlotSrc>
__global__ void __launch_bounds__(256, DEVIS_FWD_MIN_BLOCKS) msda_fwd_kernel(const FwdArgs<SlotSrc> a)
{
    using X = TapExchange<LPG>;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + a.n_slots_total) + (threadIdx.x >> 5) * (2 * X::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x % LPG;          // channel quad owned by this lane == tap it prepares
    const int g = (threadIdx.x & 31) / LPG;   // group within the warp
    const int grp = threadIdx.x / LPG;        // group within the CTA
    const int QC = blockDim.x / LPG;          // (query, head) pairs in flight per CTA
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;

    int q[QPG];
    bool qlive[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        const int qi = (qchunk * QPG + i) * QC + grp;
        qlive[i] = qi < Lq;
        q[i] = qlive[i] ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
    }

    // value row = M*LPG channel quads; this lane reads quad (m*LPG + j) of every row it touches
    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kQuadBytes;
    // keep the per-lane base as ONE 64-bit register pair: each corner address is then base + u32 offset
    // (IADD3 + IADD3.X) instead of a re-derived IMAD.WIDE chain (5 instructions per address in round 1a)
    asm volatile("" : "+l"(vbase));

    float4 acc[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    int slot_base = 0, parity = 0;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P, pshift = pow2_shift(P);
        const float *loc = reinterpret_cast<const float *>(a.seg[sg].loc);
        const float *aw = reinterpret_cast<const float *>(a.seg[sg].aw);
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
                    xy = ld_stream_f2(reinterpret_cast<const float2 *>(loc + row * K * 2) + k);
                    w = ld_stream_f(aw + row * K + k);
                }
                const TapGeom t = tap_geometry(xy.x, xy.y, sl, live);
                float *buf = xbuf + parity * X::kWordsPerWarpBuf;
                parity ^= 1;
                X::publish(buf, j, g, t, w, rowbytes);
                __syncwarp();
                // TB taps are fetched together so that 4*TB corner loads are in flight before the first FFMA needs one
                constexpr int TB = DEVIS_FWD_TAP_BATCH;
#pragma unroll
                for (int j0 = 0; j0 < LPG; j0 += TB) {
                    uint4 off[TB];
                    float4 c[TB];
                    float4 v[TB][4];
#pragma unroll
                    for (int u = 0; u < TB; ++u) X::fetch(buf, j0 + u, g, off[u], c[u]);
#pragma unroll
                    for (int u = 0; u < TB; ++u) {
                        if constexpr (E != Elem::F32) {
                            v[u][0] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off[u].x));
                            v[u][1] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off[u].y));
                            v[u][2] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off[u].z));
                            v[u][3] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off[u].w));
                        } else {
                            v[u][0] = ldg_f4(reinterpret_cast<const float4 *>(vbase + off[u].x));
                            v[u][1] = ldg_f4(reinterpret_cast<const float4 *>(vbase + off[u].y));
                            v[u][2] = ldg_f4(reinterpret_cast<const float4 *>(vbase + off[u].z));
                            v[u][3] = ldg_f4(reinterpret_cast<const float4 *>(vbase + off[u].w));
                        }
                    }
#pragma unroll
                    for (int u = 0; u < TB; ++u) {
                        acc[i].x = fmaf(c[u].w, v[u][3].x, fmaf(c[u].z, v[u][2].x, fmaf(c[u].y, v[u][1].x, fmaf(c[u].x, v[u][0].x, acc[i].x))));
                        acc[i].y = fmaf(c[u].w, v[u][3].y, fmaf(c[u].z, v[u][2].y, fmaf(c[u].y, v[u][1].y, fmaf(c[u].x, v[u][0].y, acc[i].y))));
                        acc[i].z = fmaf(c[u].w, v[u][3].z, fmaf(c[u].z, v[u][2].z, fmaf(c[u].y, v[u][1].z, fmaf(c[u].x, v[u][0].z, acc[i].z))));
                        acc[i].w = fmaf(c[u].w, v[u][3].w, fmaf(c[u].z, v[u][2].w, fmaf(c[u].y, v[u][1].w, fmaf(c[u].x, v[u][0].w, acc[i].w))));
                    }
                }
            }
        }
        slot_base += a.seg[sg].n_slots;
    }

#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        if (!qlive[i]) continue;
        const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
        if constexpr (E != Elem::F32)
            reinterpret_cast<uint2 *>(a.out)[row * LPG + j] = pack_16x4<E>(acc[i]);
        else
            st_stream_f4(reinterpret_cast<float4 *>(a.out) + row * LPG + j, acc[i]);
    }
}


// =================================================================================================
// Exchange layout of the 16-byte tap records, eight taps x four lane groups per warp and buffer
// =================================================================================================
struct Tap16x8 {
    static constexpr int kWordsPerWarpBuf = 8 * 4 * 4;  // 8 taps x 4 groups x 4 words
    static constexpr int kBytesPerWarp = 2 * kWordsPerWarpBuf * 4;
    // readers: fixed tap, 4 groups -> 4 consecutive 16-B records; writers (fixed group, 8 taps): 8 lanes of a
    // quarter-warp write records 64 B apart -> swizzle the group slot with the tap index to spread the banks
    __device__ static __forceinline__ int word(int j, int g) { return (j * 4 + (g ^ (j & 3))) * 4; }
};

// =================================================================================================
// msda_fwdv_kernel (round 2; default for D = 32, P % 4 == 0) -- eight lanes per (query, head) like msda_fwd_kernel, ONE
// 16-byte record per tap (one LDS.128 instead of two), operands prefetched one exchange ahead, DEAD CORNERS SKIPPED.
//   record = { signed byte offset of the footprint's top-left cell | 4 live bits,  w*hh,  w*lh,  lw }
// (tap_geometry_v).  The consumer forms TL = base + offset and BL = TL + map-row pitch (two 64-bit adds); TR and BR are
// the same two registers with an IMMEDIATE of one value row when the row size is a compile-time constant (ROWB: 8 heads
// x 32 channels = 1024 B fp32 / 512 B bf16 -- every DeVIS configuration), so a tap costs 4 address instructions
// instead of 8 and none of the clamp / mask selects the zero-factor form needs.  The four gathers and their 16 FFMA are predicated
// on the live bits: a corner outside its map costs no L1 wavefront (28 % of all corners at the DeVIS layer-clip, where
// most taps into the 6 x 10 and 12 x 20 maps of the other frames leave the map) and, unlike the zero-factor form, can
// not leak a non-finite value of a neighbouring pixel into the result.  Offsets are signed 32-bit: value < 2 GiB.
// =================================================================================================
#ifndef DEVIS_FWDV_MIN_BLOCKS
#define DEVIS_FWDV_MIN_BLOCKS 3
#endif
#ifndef DEVIS_FWDV_MAXT
#define DEVIS_FWDV_MAXT 256
#endif
#ifndef DEVIS_FWDV_TB
#define DEVIS_FWDV_TB 1
#endif
// Predicated gather / accumulate as straight-line PTX: written as C++ `if (live) v = load; ... if (live) acc += c * v;`
// the front end merges the two regions and the load is followed at once by its first use -- one gather in flight per
// warp.  As PTX the gathers of a tap (pair) are issued back to back like unpredicated ones.
// A predicated-off gather keeps the previous content of its destination ("+f": ptxas treats a predicated write as a
// read-modify-write anyway, and with write-only operands it kept all 128 destinations of an exchange live from kernel
// entry -- 1.4 KB of spills); the 32 destination registers therefore live in the kernel's scope, zeroed once.  Only the
// equally predicated FFMAs read them.
__device__ __forceinline__ void ldg_f4_if(float4 &v, const char *p, unsigned live)
{
#if DEVIS_HINTS & 4
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0;\n\t@p ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];\n\t}"
#else
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0;\n\t@p ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];\n\t}"
#endif
        : "+f"(v.x), "+f"(v.y), "+f"(v.z), "+f"(v.w)
        : "l"(p), "r"(live));
}
// four consecutive bf16 channels, widened (bf16 -> fp32 is a shift, so the conversion needs no predicate)
__device__ __forceinline__ void ldg_bf16x4_if(float4 &v, const char *p, unsigned live)
{
    unsigned lo = __float_as_uint(v.x), hi = __float_as_uint(v.z);
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p ld.global.nc.v2.u32 {%0,%1}, [%2];\n\t}" : "+r"(lo), "+r"(hi) : "l"(p), "r"(live));
    v.x = __uint_as_float(lo << 16);
    v.y = __uint_as_float(lo & 0xffff0000u);
    v.z = __uint_as_float(hi << 16);
    v.w = __uint_as_float(hi & 0xffff0000u);
}
// four consecutive fp16 channels, widened (the conversion is exact and cannot fault; only the FFMAs carry the predicate)
__device__ __forceinline__ void ldg_f16x4_if(float4 &v, const char *p, unsigned live)
{
    unsigned lo = __float_as_uint(v.x), hi = __float_as_uint(v.z);
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p ld.global.nc.v2.u32 {%0,%1}, [%2];\n\t}" : "+r"(lo), "+r"(hi) : "l"(p), "r"(live));
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&lo));
    const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&hi));
    v = make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void fma4_if(float4 &acc, float c, const float4 &v, unsigned live)
{
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %9, 0;\n\t"
        "@p fma.rn.f32 %0, %4, %5, %0;\n\t@p fma.rn.f32 %1, %4, %6, %1;\n\t@p fma.rn.f32 %2, %4, %7, %2;\n\t@p fma.rn.f32 %3, %4, %8, %3;\n\t}"
        : "+f"(acc.x), "+f"(acc.y), "+f"(acc.z), "+f"(acc.w)
        : "f"(c), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(live));
}

// TB = taps whose gathers are in flight together (v: their destinations, owned by the kernel)
template <Elem E, int ROWB, int TB>
__device__ __forceinline__ void consume_tap16v(const float *buf, int g, unsigned rowbytes_rt, unsigned pitch_lo,
                                               unsigned pitch_hi, const char *vbase, float4 &acc, float4 (&v)[TB][4])
{
    const unsigned rowb = ROWB ? (unsigned)ROWB : rowbytes_rt;
#pragma unroll
    for (int j0 = 0; j0 < 8; j0 += TB) {
        const char *pt[TB], *pb[TB];
        float c[TB][4];
        unsigned flags[TB];
#pragma unroll
        for (int u = 0; u < TB; ++u) {
            const uint4 r = *reinterpret_cast<const uint4 *>(buf + Tap16x8::word(j0 + u, g));
            flags[u] = r.x;
            pt[u] = vbase + (ptrdiff_t)(int)(r.x & ~15u);
            pb[u] = pt[u] + ((j0 + u) < 4 ? pitch_lo : pitch_hi);
            const float lw = __uint_as_float(r.w), hw = 1.f - lw;
            const float whh = __uint_as_float(r.y), wlh = __uint_as_float(r.z);
            c[u][0] = whh * hw;
            c[u][1] = whh * lw;
            c[u][2] = wlh * hw;
            c[u][3] = wlh * lw;
        }
#pragma unroll
        for (int u = 0; u < TB; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const char *addr = ((e & 2) ? pb[u] : pt[u]) + ((e & 1) ? rowb : 0u);
                if (E == Elem::BF16) ldg_bf16x4_if(v[u][e], addr, flags[u] & (1u << e));
                else if (E == Elem::F16) ldg_f16x4_if(v[u][e], addr, flags[u] & (1u << e));
                else ldg_f4_if(v[u][e], addr, flags[u] & (1u << e));
            }
#pragma unroll
        for (int u = 0; u < TB; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) fma4_if(acc, c[u][e], v[u][e], flags[u] & (1u << e));
    }
}

__device__ __forceinline__ uint4 make_tap16v(const TapGeomV &t, float w, unsigned rowbytes)
{
    uint4 rec;
    rec.x = (unsigned)(t.rowv * (int)rowbytes) | t.live;
    rec.y = __float_as_uint(w * t.hh);
    rec.z = __float_as_uint(w * t.lh);
    rec.w = __float_as_uint(t.lw);
    return rec;
}

template <Elem E, int QPG, class SlotSrc, int ROWB>
__global__ void __launch_bounds__(DEVIS_FWDV_MAXT, DEVIS_FWDV_MIN_BLOCKS) msda_fwdv_kernel(const FwdArgs<SlotSrc> a)
{
    constexpr int LPG = 8;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + a.n_slots_total) + (threadIdx.x >> 5) * (2 * Tap16x8::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x & 7, g = (threadIdx.x & 31) >> 3, grp = threadIdx.x >> 3, QC = blockDim.x >> 3;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;

    int q[QPG];
    bool qlive[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        const int qi = (qchunk * QPG + i) * QC + grp;
        qlive[i] = qi < Lq;
        q[i] = qlive[i] ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
    }

    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = ROWB ? (unsigned)ROWB : (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kQuadBytes;
    asm volatile("" : "+l"(vbase));

    float4 acc[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    struct TapIn {
        float2 xy;
        float w;
    };
    auto load_taps = [&](int sg, int k0, TapIn (&in)[QPG]) {
        const int K = a.seg[sg].n_slots * a.seg[sg].P;
        const float *loc = reinterpret_cast<const float *>(a.seg[sg].loc);
        const float *aw = reinterpret_cast<const float *>(a.seg[sg].aw);
        const int k = k0 + j;
#pragma unroll
        for (int i = 0; i < QPG; ++i) {
            const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
            in[i].xy = make_float2(0.f, 0.f);
            in[i].w = 0.f;
            if (k < K && qlive[i]) {
                in[i].xy = ld_stream_f2(reinterpret_cast<const float2 *>(loc + row * K * 2) + k);
                in[i].w = ld_stream_f(aw + row * K + k);
            }
        }
    };

    float4 v[DEVIS_FWDV_TB][4];             // gather destinations (see ldg_f4_if)
#pragma unroll
    for (int u = 0; u < DEVIS_FWDV_TB; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) v[u][e] = make_float4(0.f, 0.f, 0.f, 0.f);

    int slot_base = 0, parity = 0;
    TapIn nxt[QPG];
    load_taps(0, 0, nxt);
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P, pshift = pow2_shift(P);   // P % 4 == 0, hence K % 4 == 0
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;
            const bool klive = k < K;
            const int4 sl = s_slot[slot_base + (klive ? div_p(k, P, pshift) : 0)];
            const unsigned my_pitch = (unsigned)sl.y * rowbytes;
            const unsigned pitch_lo = __shfl_sync(0xffffffffu, my_pitch, 0, 8);   // slot of taps k0 .. k0+3
            const unsigned pitch_hi = __shfl_sync(0xffffffffu, my_pitch, 4, 8);   // slot of taps k0+4 .. k0+7
            TapIn cur[QPG];
#pragma unroll
            for (int i = 0; i < QPG; ++i) cur[i] = nxt[i];
            if (k0 + LPG < K) load_taps(sg, k0 + LPG, nxt);
            else if (sg + 1 < a.n_seg) load_taps(sg + 1, 0, nxt);
#pragma unroll
            for (int i = 0; i < QPG; ++i) {
                const TapGeomV t = tap_geometry_v(cur[i].xy.x, cur[i].xy.y, sl, klive && qlive[i]);
                float *buf = xbuf + parity * Tap16x8::kWordsPerWarpBuf;
                parity ^= 1;
                *reinterpret_cast<uint4 *>(buf + Tap16x8::word(j, g)) = make_tap16v(t, cur[i].w, rowbytes);
                __syncwarp();
                consume_tap16v<E, ROWB, DEVIS_FWDV_TB>(buf, g, rowbytes, pitch_lo, pitch_hi, vbase, acc[i], v);
            }
        }
        slot_base += a.seg[sg].n_slots;
    }

#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        if (!qlive[i]) continue;
        const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
        if constexpr (E != Elem::F32)
            reinterpret_cast<uint2 *>(a.out)[row * LPG + j] = pack_16x4<E>(acc[i]);
        else
            st_stream_f4(reinterpret_cast<float4 *>(a.out) + row * LPG + j, acc[i]);
    }
}

// =================================================================================================
// Four lanes per (query, head), 8 channels per lane: the shape of the bf16 forward.  A head's bf16 row is 64 B = 4 lanes
// x 16 B, 8 rows per LDG.128 (measured 0.75 data-pipe cycles per row against 1.0 for 8 lanes x 8 bytes), and the record
// shrinks the exchange to ONE LDS.128 per tap for 8 groups.  Requires P % 4 == 0 so that the 4 taps a group exchanges at a
// time belong to one slot (DeVIS: P = 4 everywhere, config.py:52-53,108-109).
// =================================================================================================
struct Tap16 {
    static constexpr int kWordsPerWarpBuf = 4 * 8 * 4;  // 4 taps x 8 groups x 4 words
    static constexpr int kBytesPerWarp = 2 * kWordsPerWarpBuf * 4;
    __device__ static __forceinline__ int word(int j, int g) { return (j * 8 + (g ^ (2 * j))) * 4; }
};

// =================================================================================================
// msda_fwd8v_kernel (round 2; default for bf16 value) -- that shape with the dead corners skipped: the record and the
// addressing of msda_fwdv_kernel (virtual top-left cell, live bits, row size as an immediate), four lanes x 8 channels per
// (query, head), 16-byte gathers predicated on the live bits.  The bf16 forward is the kernel closest to the data-pipe
// limit (87 % busy), so the 28 % of rows that need not be fetched show up in the time.
// =================================================================================================
__device__ __forceinline__ void ldg_u4_if(uint4 &v, const char *p, unsigned live)
{
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0;\n\t@p ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
        : "+r"(v.x), "+r"(v.y), "+r"(v.z), "+r"(v.w)
        : "l"(p), "r"(live));
}
template <Elem E>
__device__ __forceinline__ void fma8_16_if(float (&acc)[8], float c, const uint4 &raw, unsigned live)
{
    // the widening is done unconditionally (cheap, exact, no faults), only the FFMAs carry the predicate
    float u[8];
    unpack_16x8<E>(raw, u);
    const float v0 = u[0], v1 = u[1], v2 = u[2], v3 = u[3], v4 = u[4], v5 = u[5], v6 = u[6], v7 = u[7];
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %17, 0;\n\t"
        "@p fma.rn.f32 %0, %8, %9, %0;\n\t@p fma.rn.f32 %1, %8, %10, %1;\n\t@p fma.rn.f32 %2, %8, %11, %2;\n\t"
        "@p fma.rn.f32 %3, %8, %12, %3;\n\t@p fma.rn.f32 %4, %8, %13, %4;\n\t@p fma.rn.f32 %5, %8, %14, %5;\n\t"
        "@p fma.rn.f32 %6, %8, %15, %6;\n\t@p fma.rn.f32 %7, %8, %16, %7;\n\t}"
        : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3]), "+f"(acc[4]), "+f"(acc[5]), "+f"(acc[6]), "+f"(acc[7])
        : "f"(c), "f"(v0), "f"(v1), "f"(v2), "f"(v3), "f"(v4), "f"(v5), "f"(v6), "f"(v7), "r"(live));
}

// one exchange of 4 published records (4 lanes x 8 16-bit channels per row), dead corners skipped
template <Elem E, int ROWB>
__device__ __forceinline__ void consume_tap16x4v(const float *buf, int g, unsigned rowbytes_rt, unsigned pitch,
                                                 const char *vbase, float (&acc)[8], uint4 (&v)[4])
{
    const unsigned rowb = ROWB ? (unsigned)ROWB : rowbytes_rt;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const uint4 r = *reinterpret_cast<const uint4 *>(buf + Tap16::word(jj, g));
        const char *pt = vbase + (ptrdiff_t)(int)(r.x & ~15u);
        const char *pb = pt + pitch;
        const float lw = __uint_as_float(r.w), hw = 1.f - lw;
        const float whh = __uint_as_float(r.y), wlh = __uint_as_float(r.z);
        const float c[4] = {whh * hw, whh * lw, wlh * hw, wlh * lw};
#pragma unroll
        for (int e = 0; e < 4; ++e) ldg_u4_if(v[e], ((e & 2) ? pb : pt) + ((e & 1) ? rowb : 0u), r.x & (1u << e));
#pragma unroll
        for (int e = 0; e < 4; ++e) fma8_16_if<E>(acc, c[e], v[e], r.x & (1u << e));
    }
}

// (no minimum-blocks hint: ptxas settles at 62-64 registers, 359 us; a hint of 1 made it unroll to 184 registers and 711 us.
// The fp32 form of this shape -- 32-byte predicated gathers, LDG.E.256 -- was measured at 527-543 us against 478 us for
// msda_fwdv_kernel and is not kept, profiles/r2s_fwd_wide_f32_variants.json)
// E: BF16 or F16 (64-byte rows of a head either way)
template <Elem E, int QPG, class SlotSrc, int ROWB>
__global__ void __launch_bounds__(256) msda_fwd8v_kernel(const FwdArgs<SlotSrc> a)
{
    static_assert(E != Elem::F32, "16-bit value only");
    constexpr int LPG = 4;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y;
    build_slots(s_slot, a.src, a.d, outer, a.n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + a.n_slots_total) + (threadIdx.x >> 5) * (2 * Tap16::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x & 3, g = (threadIdx.x & 31) >> 2, grp = threadIdx.x >> 2, QC = blockDim.x >> 2;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;

    int q[QPG];
    bool qlive[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        const int qi = (qchunk * QPG + i) * QC + grp;
        qlive[i] = qi < Lq;
        q[i] = qlive[i] ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
    }

    constexpr unsigned kLaneBytes = 16u;                       // 8 16-bit channels
    const unsigned rowbytes = ROWB ? (unsigned)ROWB : (unsigned)(M * LPG) * kLaneBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kLaneBytes;
    asm volatile("" : "+l"(vbase));

    float acc[QPG][8];
#pragma unroll
    for (int i = 0; i < QPG; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
    uint4 v[4];                                                // gather destinations (see ldg_f4_if): 8 raw channels per corner
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = make_uint4(0u, 0u, 0u, 0u);

    int slot_base = 0, parity = 0;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.seg[sg].P, K = a.seg[sg].n_slots * P, pshift = pow2_shift(P);   // P % 4 == 0 (checked by the launcher)
        const float *loc = reinterpret_cast<const float *>(a.seg[sg].loc);
        const float *aw = reinterpret_cast<const float *>(a.seg[sg].aw);
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;                                // always < K
            const int4 sl = s_slot[slot_base + div_p(k0, P, pshift)];          // one slot for the whole exchange
            const unsigned pitch = (unsigned)sl.y * rowbytes;
#pragma unroll
            for (int i = 0; i < QPG; ++i) {
                const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
                float2 xy = make_float2(0.f, 0.f);
                float w = 0.f;
                if (qlive[i]) {
                    xy = ld_stream_f2(reinterpret_cast<const float2 *>(loc + row * K * 2) + k);
                    w = ld_stream_f(aw + row * K + k);
                }
                const TapGeomV t = tap_geometry_v(xy.x, xy.y, sl, qlive[i]);
                float *buf = xbuf + parity * Tap16::kWordsPerWarpBuf;
                parity ^= 1;
                *reinterpret_cast<uint4 *>(buf + Tap16::word(j, g)) = make_tap16v(t, w, rowbytes);
                __syncwarp();
                consume_tap16x4v<E, ROWB>(buf, g, rowbytes, pitch, vbase, acc[i], v);
            }
        }
        slot_base += a.seg[sg].n_slots;
    }

#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        if (!qlive[i]) continue;
        const size_t row = ((size_t)outer * Lq + q[i]) * M + m;
        const uint2 lo = pack_16x4<E>(make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
        const uint2 hi = pack_16x4<E>(make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
        reinterpret_cast<uint4 *>(a.out)[row * LPG + j] = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
}

}  // namespace devis
