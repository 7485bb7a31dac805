// msda_common.cuh -- shared definitions for the sm_100a multi-scale deformable attention kernels.
//
// Vocabulary (follows the reference, modules/ms_deform_attn.py and cuda/ms_deform_im2col_cuda.cuh):
//   value row   one pixel of one level of one batch item / frame: M heads x D channels, contiguous
//   slot        one (frame, level) map a query can sample: {H, W, first value row}.  For the per-call op a
//               slot is a level (ms_deform_attn_cuda.cu:67-68); for the whole-clip temporal op slots
//               [0,L) are the query frame's own levels and slot L + j*L + l is level l of temporal
//               frame j (ms_deform_attn.py:232-238: temporal "levels" are frame-major, level-minor)
//   segment     a (sampling_loc, attn_weight) tensor pair covering a contiguous run of slots with a fixed
//               number of points per slot: one segment per call for the plain op, two (current, temporal)
//               for the whole-clip op
//   tap         one sampling point of one (query, head): a bilinear read of 4 value rows
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace devis {

constexpr int kMaxLevels = 16;        // host-side table of the whole-clip op
constexpr int kMaxFrameTable = 2048;  // T * t_window entries (uint8 each)
constexpr int kMaxSlots = 1024;       // slots per query (dynamic smem: 16 B each)

// Element type of value / output / grad_output in the lane-group kernels: float, or one of the two 16-bit types
// (DEVIS_MSDA_BF16, DEVIS_MSDA_F16).  A 16-bit element is widened exactly to fp32 on load, every sum is formed in fp32,
// and a 16-bit result is rounded to nearest once, on the store.
enum class Elem { F32, BF16, F16 };

struct Segment {
    const void *loc;   // (outer, Lq, M, n_slots, P, 2)
    const void *aw;    // (outer, Lq, M, n_slots, P)
    void *grad_loc;    // backward only
    void *grad_aw;     // backward only
    int n_slots;
    int P;
};

// Slot source of the per-call op: the reference's device-resident int64 tensors.
struct DeviceLevels {
    const int64_t *shapes;  // (L,2) rows (H,W)
    const int64_t *lsi;     // (L)
};

// Slot source of the whole-clip op: host tables passed by value in the kernel parameters.
struct ClipTable {
    int H[kMaxLevels];
    int W[kMaxLevels];
    int lsi[kMaxLevels];
    int L;
    int Wt;
    uint8_t frame[kMaxFrameTable];  // [t * Wt + j]
};

struct OpDims {
    int outer;  // batch (plain op) or query frames (whole-clip op)
    int S;      // value rows per outer item
    int M, D;
    int Lq;
};

// ---------------------------------------------------------------------------------------------
// slot table in shared memory: int4 {H, W, first value row (absolute, outer offset included), W*M}
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void build_slots(int4 *s_slot, const DeviceLevels &lv, const OpDims &d, int outer,
                                            int n_slots)
{
    for (int s = threadIdx.x; s < n_slots; s += blockDim.x) {
        const int H = (int)lv.shapes[2 * s], W = (int)lv.shapes[2 * s + 1];
        s_slot[s] = make_int4(H, W, outer * d.S + (int)lv.lsi[s], W * d.M);
    }
    __syncthreads();
}

__device__ __forceinline__ void build_slots(int4 *s_slot, const ClipTable &tb, const OpDims &d, int outer,
                                            int n_slots)
{
    for (int s = threadIdx.x; s < n_slots; s += blockDim.x) {
        int frame, l;
        if (s < tb.L) {
            frame = outer;
            l = s;
        } else {
            const int j = (s - tb.L) / tb.L;
            l = (s - tb.L) - j * tb.L;
            frame = tb.frame[outer * tb.Wt + j];
        }
        s_slot[s] = make_int4(tb.H[l], tb.W[l], frame * d.S + tb.lsi[l], tb.W[l] * d.M);
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// k / P and slot % L with RUNTIME P and L: an integer division costs ~20 instructions in kernels that
// are bound by instruction issue (forward: 59 % issue-active with 6 warps per scheduler); points per
// slot and levels are powers of two in every DeVIS configuration (4 and 4), so take shifts and masks
// there and keep the division for the rest.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int pow2_shift(int v) { return (v > 0 && (v & (v - 1)) == 0) ? __ffs(v) - 1 : -1; }
__device__ __forceinline__ int div_p(int k, int P, int pshift) { return pshift >= 0 ? (k >> pshift) : (k / P); }
__device__ __forceinline__ int mod_l(int s, int L, int lshift) { return lshift >= 0 ? (s & (L - 1)) : (s % L); }

// ---------------------------------------------------------------------------------------------
// One tap's geometry, computed by ONE lane and then handed to the lanes that own the channels.
// Mirrors cuda/ms_deform_im2col_cuda.cuh:281-288 (pixel coordinate and range test) and :38-52,80
// (floor cell, bilinear weights); the rounding sequence of the coordinate is the reference's:
// round(round(loc*size) - 0.5), no FMA contraction, so floor() picks the reference's cell.
//
// Corners outside the map get a ZERO weight factor and a clamped (always in-bounds) row, so the
// consumer does four unconditional 16-byte loads per tap with no predicates: the reference's
// "if (h_low >= 0 && w_low >= 0) ..." guards (cuh:56-78) become multiplications by zero.
// ---------------------------------------------------------------------------------------------
struct TapGeom {
    float lh, lw, hh, hw;    // fractional parts and complements (unmasked; the backward needs them)
    int rTL, rTR, rBL, rBR;  // clamped value rows of the 4 corners
    int y0c, x0c;            // clamped (row, column) of the top-left corner inside its map (window placement)
    unsigned ok;             // bit0 top row, bit1 bottom row, bit2 left column, bit3 right column inside the
                             // map; 0 if the whole tap fails the reference's range test
};

__device__ __forceinline__ TapGeom tap_geometry(float x, float y, const int4 slot, bool live)
{
    TapGeom g;
    const int H = slot.x, W = slot.y;
    const float h_im = __fadd_rn(__fmul_rn(y, (float)H), -0.5f);
    const float w_im = __fadd_rn(__fmul_rn(x, (float)W), -0.5f);
    const bool inb = live && h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W;
    const float hf = floorf(h_im), wf = floorf(w_im);
    const int h0 = inb ? (int)hf : 0, w0 = inb ? (int)wf : 0;
    g.lh = h_im - hf;
    g.lw = w_im - wf;
    g.hh = 1.f - g.lh;
    g.hw = 1.f - g.lw;
    g.ok = inb ? ((unsigned)(h0 >= 0) | ((unsigned)(h0 + 1 <= H - 1) << 1) | ((unsigned)(w0 >= 0) << 2) |
                  ((unsigned)(w0 + 1 <= W - 1) << 3))
               : 0u;
    const int h0c = max(h0, 0), h1c = min(h0 + 1, H - 1), w0c = max(w0, 0), w1c = min(w0 + 1, W - 1);
    const int top = slot.z + h0c * W, bot = slot.z + h1c * W;
    g.y0c = h0c;
    g.x0c = w0c;
    g.rTL = top + w0c;
    g.rTR = top + w1c;
    g.rBL = bot + w0c;
    g.rBR = bot + w1c;
    return g;
}

// ---------------------------------------------------------------------------------------------
// Round 2: tap geometry with a VIRTUAL top-left corner.  In the DeVIS-like workload 28 % of all corners are dead (the
// tap leaves a coarse map, or one row / column of its 2 x 2 footprint does): the reference never loads those
// (cuh:56-78), and neither do the round-2 consumers -- every gathered row is a wavefront of the L1 data pipe, the
// resource the kernels are bound by.  Dead corners are predicated off, so nothing needs clamping: the record carries the
// byte offset of the footprint's top-left cell even when that cell is outside the map (row / column -1), the other
// three addresses are TL + one value row, TL + one map row, TL + both, and four live bits say which of them exist.
// ---------------------------------------------------------------------------------------------
struct TapGeomV {
    float lh, lw, hh, hw;   // fractional parts and complements
    int rowv;               // value row of the (possibly virtual) top-left cell; may be up to W + 1 rows before the map
    unsigned live;          // bit0 TL, bit1 TR, bit2 BL, bit3 BR inside the map; 0 if the tap fails the range test
    unsigned ok;            // as TapGeom::ok
};

__device__ __forceinline__ TapGeomV tap_geometry_v(float x, float y, const int4 slot, bool live)
{
    TapGeomV g;
    const int H = slot.x, W = slot.y;
    const float h_im = __fadd_rn(__fmul_rn(y, (float)H), -0.5f);
    const float w_im = __fadd_rn(__fmul_rn(x, (float)W), -0.5f);
    const bool inb = live && h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W;
    const float hf = floorf(h_im), wf = floorf(w_im);
    const int h0 = inb ? (int)hf : 0, w0 = inb ? (int)wf : 0;
    g.lh = h_im - hf;
    g.lw = w_im - wf;
    g.hh = 1.f - g.lh;
    g.hw = 1.f - g.lw;
    const unsigned top = h0 >= 0, bot = h0 + 1 <= H - 1, left = w0 >= 0, right = w0 + 1 <= W - 1;
    g.ok = inb ? (top | (bot << 1) | (left << 2) | (right << 3)) : 0u;
    g.live = inb ? ((top & left) | ((top & right) << 1) | ((bot & left) << 2) | ((bot & right) << 3)) : 0u;
    g.rowv = slot.z + h0 * W + w0;
    return g;
}

// ---------------------------------------------------------------------------------------------
// Padding mask (MSDeformAttn's input_padding_mask): one byte per value row, nonzero = the row reads as zero, exactly as
// value.masked_fill(mask[..., None], 0) before the op.  A masked corner is DROPPED, never multiplied by zero -- a masked
// row may hold NaN or Inf, and 0 x NaN is NaN: it is not gathered, not scattered to, and its value counts as 0 in the
// location and weight gradients.  Only the bytes of corners inside the map are read (rows frame*S + pixel, L1-resident).
// ---------------------------------------------------------------------------------------------
// tap_geometry_v's live bits without the masked corners
__device__ __forceinline__ unsigned unmasked_live(const uint8_t *mask, int rowv, int W, unsigned live)
{
    const uint8_t *p = mask + (ptrdiff_t)rowv;
    if ((live & 1u) && __ldg(p)) live &= ~1u;
    if ((live & 2u) && __ldg(p + 1)) live &= ~2u;
    if ((live & 4u) && __ldg(p + W)) live &= ~4u;
    if ((live & 8u) && __ldg(p + W + 1)) live &= ~8u;
    return live;
}

// per-corner bits of a TapGeom (bit0 TL, bit1 TR, bit2 BL, bit3 BR): the corner is inside the map and not masked
__device__ __forceinline__ unsigned unmasked_corners(const uint8_t *mask, const TapGeom &t)
{
    const unsigned top = t.ok & 1u, bot = (t.ok >> 1) & 1u, left = (t.ok >> 2) & 1u, right = (t.ok >> 3) & 1u;
    unsigned c = (top & left) | ((top & right) << 1) | ((bot & left) << 2) | ((bot & right) << 3);
    if ((c & 1u) && __ldg(mask + t.rTL)) c &= ~1u;
    if ((c & 2u) && __ldg(mask + t.rTR)) c &= ~2u;
    if ((c & 4u) && __ldg(mask + t.rBL)) c &= ~4u;
    if ((c & 8u) && __ldg(mask + t.rBR)) c &= ~8u;
    return c;
}

// ---------------------------------------------------------------------------------------------
// Tap exchange through shared memory.  A group of LPG lanes owns one (query, head); lane j prepares
// tap k0+j and publishes a 32-byte record; then all lanes of the group walk the LPG records.
// (Round-1 profile: doing this with __shfl_sync cost 6 L1-data-pipe wavefronts per tap -- shuffles
// are counted in l1tex__data_pipe_lsu_wavefronts_mem_shared -- against 16 for the four corner
// gathers; two broadcast LDS.128 cost 2.)
//   record = { u32 byte offset of TL, TR, BL, BR corner rows | w*hh, w*lh, hw, lw }   (masked factors)
// Layout per warp and buffer: [tap j][group slot], slot = g ^ (j & 3): readers (fixed j, 4 groups)
// and writers (fixed g, 8 taps; halves written in swapped order for j >= 4) are bank-conflict free.
// ---------------------------------------------------------------------------------------------
template <int LPG>
struct TapExchange {
    static constexpr int GPW = 32 / LPG;                 // groups per warp
    static constexpr int kWordsPerWarpBuf = LPG * GPW * 8;
    static constexpr int kBytesPerWarp = 2 * kWordsPerWarpBuf * 4;  // double buffered

    __device__ static __forceinline__ int rec_word(int j, int g) { return (j * GPW + (g ^ (j & (GPW - 1)))) * 8; }

    // tag: bit 0 of the TL offset (row pitches are even) -- msda_bwd_sort.cuh marks taps whose grad_value
    // contributions take the sorted path; every other caller leaves it 0
    __device__ static __forceinline__ void publish(float *buf, int j, int g, const TapGeom &t, float w, unsigned rowbytes,
                                                   unsigned tag = 0u)
    {
        const bool live = t.ok != 0u;
        uint4 off;
        off.x = ((unsigned)t.rTL * rowbytes) | tag;
        off.y = (unsigned)t.rTR * rowbytes;
        off.z = (unsigned)t.rBL * rowbytes;
        off.w = (unsigned)t.rBR * rowbytes;
        float4 f;
        f.x = (live && (t.ok & 1u)) ? w * t.hh : 0.f;
        f.y = (live && (t.ok & 2u)) ? w * t.lh : 0.f;
        f.z = (t.ok & 4u) ? t.hw : 0.f;
        f.w = (t.ok & 8u) ? t.lw : 0.f;
        float *r = buf + rec_word(j, g);
        if (j & 4) {
            *reinterpret_cast<float4 *>(r + 4) = f;
            *reinterpret_cast<uint4 *>(r) = off;
        } else {
            *reinterpret_cast<uint4 *>(r) = off;
            *reinterpret_cast<float4 *>(r + 4) = f;
        }
    }

    __device__ static __forceinline__ void fetch(const float *buf, int jj, int g, uint4 &off, float4 &c)
    {
        const float *r = buf + rec_word(jj, g);
        off = *reinterpret_cast<const uint4 *>(r);
        const float4 f = *reinterpret_cast<const float4 *>(r + 4);
        c.x = f.x * f.z;  // TL
        c.y = f.x * f.w;  // TR
        c.z = f.y * f.z;  // BL
        c.w = f.y * f.w;  // BR
    }
};

// Cache hints (compile-time A/B, benchmarks/variant_sweep.py).  The value rows are the only data with reuse in L1
// (72-78 % hit rate); locations, weights and every output are touched exactly once.  DEVIS_HINTS bit 0: streaming
// operand loads do not allocate in L1; bit 1: streaming stores do not allocate in L1; bit 2: value rows are loaded
// with L1::evict_last.  Measured (round 1j, DeVIS layer-clip): fp32 forward 527 -> 520 us with all three, backward and bf16
// forward unchanged -> default 7.
#ifndef DEVIS_HINTS
#define DEVIS_HINTS 7
#endif

__device__ __forceinline__ float2 ld_stream_f2(const float2 *p)
{
#if DEVIS_HINTS & 1
    float2 v;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
#else
    return __ldg(p);
#endif
}

__device__ __forceinline__ float ld_stream_f(const float *p)
{
#if DEVIS_HINTS & 1
    float v;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
#else
    return __ldg(p);
#endif
}

__device__ __forceinline__ void st_stream_f4(float4 *p, float4 v)
{
#if DEVIS_HINTS & 2
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
#else
    *p = v;
#endif
}

__device__ __forceinline__ void st_stream_f2(float2 *p, float2 v)
{
#if DEVIS_HINTS & 2
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
#else
    *p = v;
#endif
}

__device__ __forceinline__ void st_stream_f(float *p, float v)
{
#if DEVIS_HINTS & 2
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
#else
    *p = v;
#endif
}

// ---------------------------------------------------------------------------------------------
// L2 residency hints (VERDICT round 1, weak item 2: the backward moved 1025 MB through DRAM against 622 MB of
// algorithmic bytes because 592 MB of single-use streams pushed value / grad_value, 59 MB together, out of the 126 MB
// L2 and the reduction's read-modify-write lines were fetched again).  createpolicy descriptors, sm_80+:
//   DEVIS_L2_HINTS bit 0: single-use streams (locations, weights, grad_out; outputs, grad_loc, grad_aw) -> L2::evict_first
//   bit 1: value gathers -> L2::evict_last        bit 2: grad_value reductions -> L2::evict_last
// Compile-time A/B like DEVIS_HINTS (benchmarks/build_variants.py).  MEASURED (round 2, profiles/r2a_l2_hints.json): no
// effect -- backward 1429-1430 us and 994-1013 MB of DRAM traffic for every combination (0, 1, 4, 6, 7), forward 516 us
// and 318-325 MB: the descriptors do not keep the reduction targets resident, and DRAM (9 % busy) is not what the kernel
// waits for anyway.  Default 0 (the policies would cost the 80-register backward an 8-byte spill for nothing).
// ---------------------------------------------------------------------------------------------
#ifndef DEVIS_L2_HINTS
#define DEVIS_L2_HINTS 0
#endif

struct L2Policy {
    unsigned long long stream;   // evict_first
    unsigned long long keep;     // evict_last
};

__device__ __forceinline__ L2Policy make_l2_policy()
{
    L2Policy p;
    p.stream = 0ull;
    p.keep = 0ull;
#if DEVIS_L2_HINTS & 1
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p.stream));
#endif
#if DEVIS_L2_HINTS & 6
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p.keep));
#endif
    return p;
}

__device__ __forceinline__ float2 ld_stream_f2(const float2 *p, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    float2 v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(p), "l"(pol.stream));
    return v;
#else
    return ld_stream_f2(p);
#endif
}

__device__ __forceinline__ float ld_stream_f(const float *p, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    float v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol.stream));
    return v;
#else
    return ld_stream_f(p);
#endif
}

__device__ __forceinline__ float4 ld_stream_f4(const float4 *p, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    float4 v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
        : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol.stream));
    return v;
#else
    return __ldg(p);
#endif
}

__device__ __forceinline__ void st_stream_f4(float4 *p, float4 v, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w), "l"(pol.stream) : "memory");
#else
    st_stream_f4(p, v);
#endif
}

__device__ __forceinline__ void st_stream_f2(float2 *p, float2 v, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.f32 [%0], {%1,%2}, %3;" ::"l"(p), "f"(v.x), "f"(v.y),
                 "l"(pol.stream) : "memory");
#else
    st_stream_f2(p, v);
#endif
}

__device__ __forceinline__ void st_stream_f(float *p, float v, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 1
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol.stream) : "memory");
#else
    st_stream_f(p, v);
#endif
}

// 16-byte read-only loads / vector reductions --------------------------------------------------
__device__ __forceinline__ float4 ldg_f4(const float4 *p)
{
#if DEVIS_HINTS & 4
    float4 v;
    asm("ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
#else
    return __ldg(p);
#endif
}

__device__ __forceinline__ float4 ldg_f4(const float4 *p, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 2
    float4 v;
    asm("ld.global.nc.L1::evict_last.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
        : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol.keep));
    return v;
#else
    return ldg_f4(p);
#endif
}

__device__ __forceinline__ float4 ldg_bf16x4(const uint2 *p)
{
    const uint2 r = __ldg(p);
    float4 o;
    o.x = __uint_as_float(r.x << 16);
    o.y = __uint_as_float(r.x & 0xffff0000u);
    o.z = __uint_as_float(r.y << 16);
    o.w = __uint_as_float(r.y & 0xffff0000u);
    return o;
}

// four consecutive fp16 channels, widened exactly (cvt.f32.f16)
__device__ __forceinline__ float4 ldg_f16x4(const uint2 *p)
{
    const uint2 r = __ldg(p);
    const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&r.x));
    const float2 hi = __half22float2(*reinterpret_cast<const __half2 *>(&r.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// four consecutive channels of a 16-bit element type E
template <Elem E>
__device__ __forceinline__ float4 ldg_16x4(const uint2 *p)
{
    static_assert(E != Elem::F32, "16-bit element types only");
    return E == Elem::F16 ? ldg_f16x4(p) : ldg_bf16x4(p);
}

__device__ __forceinline__ void red_add_f4(float *p, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// four consecutive bf16 channels as one 8-byte packed reduction (each addend is rounded to bf16, and so is every
// partial sum at the L2 -- the precision of PyTorch's own bf16 atomicAdd scatter, e.g. grid_sample's backward)
__device__ __forceinline__ void red_add_bf16x4(void *p, float a, float b, float c, float d)
{
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    asm volatile("red.global.add.noftz.v2.bf16x2 [%0], {%1,%2};" ::"l"(p),
                 "r"(*reinterpret_cast<const unsigned *>(&lo)), "r"(*reinterpret_cast<const unsigned *>(&hi))
                 : "memory");
}

__device__ __forceinline__ void red_add_f4(float *p, float a, float b, float c, float d, const L2Policy &pol)
{
#if DEVIS_L2_HINTS & 4
    asm volatile("red.global.add.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d),
                 "l"(pol.keep) : "memory");
#else
    red_add_f4(p, a, b, c, d);
#endif
}

template <bool HALF>
__device__ __forceinline__ void red_add_quad(char *p, float a, float b, float c, float d)
{
    if (HALF) red_add_bf16x4(p, a, b, c, d);
    else red_add_f4(reinterpret_cast<float *>(p), a, b, c, d);
}

template <bool HALF>
__device__ __forceinline__ void red_add_quad(char *p, float a, float b, float c, float d, const L2Policy &pol)
{
    if (HALF) red_add_bf16x4(p, a, b, c, d);
    else red_add_f4(reinterpret_cast<float *>(p), a, b, c, d, pol);
}

// ---------------------------------------------------------------------------------------------
// Deterministic grad_value (DEVIS_MSDA_FLAG_DETERMINISTIC).  Floating-point atomics make the
// reference's grad_value run-to-run different (SURVEY.md section 5).  Here every contribution
// (a float product) is converted EXACTLY to a 64-bit fixed-point integer and accumulated with integer
// reductions, which are associative: the sum does not depend on arrival order.  Scale: 2^(36 - e) with
// 2^e > max|grad_out| * max|attn| >= every contribution (weights are <= 1), so |q| < 2^36 and 2^27
// contributions per element fit in int64; resolution is 2^-36 of the largest possible contribution
// (fp32 accumulation has 2^-24 of the running sum).  A finalize pass converts back to float.
// ---------------------------------------------------------------------------------------------
struct DetScale {
    const unsigned *max_bits;  // [0] = bits of max|grad_out|, [1] = bits of max|attn weight| (non-negative floats)
    long long *acc;            // (outer, S, M, D) fixed-point accumulators, zero-filled
};

constexpr int kDetFracBits = 36;

// the bound is the product of n_factors non-negative floats max_bits[0 .. n_factors) (the attention: 2; the deformable
// convolution, deform_conv.cuh: 4)
__device__ __forceinline__ int det_exponent(const unsigned *max_bits, int n_factors = 2)
{
    float bound = __uint_as_float(max_bits[0]);
    for (int i = 1; i < n_factors; ++i) bound *= __uint_as_float(max_bits[i]);
    int e = 0;
    if (bound > 0.f && bound < 3.0e38f) (void)frexpf(bound, &e);   // bound = f * 2^e, f in [0.5, 1)
    return e + 1;
}

// The grouped-lane kernels keep the accumulators of one (row, head) in a PERMUTED channel order: channel 4*j + c
// (lane j's c-th channel) lives at element c*LPG + j, so that the LPG lanes of a group hit LPG consecutive 8-byte
// words with each of their four reductions (64 contiguous bytes for LPG = 8; in channel order a lane's four words
// are 32 bytes apart from its neighbour's and every 32-byte sector left the SM a quarter full: 9.7 ms per DeVIS
// layer-clip backward).  det_finalize_kernel undoes the permutation.
template <int LPG>
__device__ __forceinline__ void det_add4(long long *p, float sh, float a, float b, float c, float d)
{
    // sh is a power of two: the products below are exact; llrint of a float is exact as well
    atomicAdd(reinterpret_cast<unsigned long long *>(p) + 0 * LPG, (unsigned long long)__float2ll_rn(a * sh));
    atomicAdd(reinterpret_cast<unsigned long long *>(p) + 1 * LPG, (unsigned long long)__float2ll_rn(b * sh));
    atomicAdd(reinterpret_cast<unsigned long long *>(p) + 2 * LPG, (unsigned long long)__float2ll_rn(c * sh));
    atomicAdd(reinterpret_cast<unsigned long long *>(p) + 3 * LPG, (unsigned long long)__float2ll_rn(d * sh));
}

// max|x| over n elements (float, bf16 or fp16) into *slot, as the bits of a non-negative float (atomicMax on the
// bit pattern is exact and order independent)
template <Elem E>
__global__ void __launch_bounds__(256) absmax_kernel(const void *x, size_t n, unsigned *slot)
{
    float m = 0.f;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = E == Elem::BF16  ? __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(x)[i])
                        : E == Elem::F16 ? __half2float(reinterpret_cast<const __half *>(x)[i])
                                         : reinterpret_cast<const float *>(x)[i];
        m = fmaxf(m, fabsf(v));
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(slot, __float_as_uint(m));
}

// set_word_kernel and det_finalize_kernel are static: each translation unit that includes this header (the attention's
// and the deformable convolution's) keeps its own copy
static __global__ void set_word_kernel(unsigned *slot, unsigned bits) { *slot = bits; }

// lpg > 0: the accumulators of every D = 4*lpg channels are in the permuted order of det_add4; lpg == 0: channel order.
// n_factors: as det_exponent
static __global__ void __launch_bounds__(256) det_finalize_kernel(const long long *acc, float *out, size_t n,
                                                           const unsigned *max_bits, int lpg, int n_factors = 2)
{
    const double back = ldexp(1.0, det_exponent(max_bits, n_factors) - kDetFracBits);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        size_t src = i;
        if (lpg) {
            const int ch = (int)(i % (size_t)(4 * lpg));
            src = i - ch + (size_t)((ch & 3) * lpg + (ch >> 2));
        }
        out[i] = (float)((double)acc[src] * back);
    }
}

__device__ __forceinline__ uint2 pack_bf16x4(float4 v)
{
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<const unsigned *>(&lo);
    r.y = *reinterpret_cast<const unsigned *>(&hi);
    return r;
}

// round to nearest, once (cvt.rn.f16x2.f32); fp32 values beyond the fp16 range become +-inf, as in a torch cast
__device__ __forceinline__ uint2 pack_f16x4(float4 v)
{
    const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<const unsigned *>(&lo);
    r.y = *reinterpret_cast<const unsigned *>(&hi);
    return r;
}

template <Elem E>
__device__ __forceinline__ uint2 pack_16x4(float4 v)
{
    static_assert(E != Elem::F32, "16-bit element types only");
    return E == Elem::F16 ? pack_f16x4(v) : pack_bf16x4(v);
}

// eight raw 16-bit channels (one 16-byte gather) widened exactly to fp32; bf16 -> fp32 is a shift / mask
template <Elem E>
__device__ __forceinline__ void unpack_16x8(const uint4 &raw, float (&v)[8])
{
    static_assert(E != Elem::F32, "16-bit element types only");
    const unsigned w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (E == Elem::F16) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));
            v[2 * i] = f.x;
            v[2 * i + 1] = f.y;
        } else {
            v[2 * i] = __uint_as_float(w[i] << 16);
            v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
}

}  // namespace devis
