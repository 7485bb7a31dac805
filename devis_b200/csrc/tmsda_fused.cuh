// tmsda_fused.cuh -- whole-clip temporal attention with the PROLOGUE fused in (SURVEY.md section 8f, rank 1).
//
// The reference turns the Linear outputs into op operands with a chain of elementwise kernels
// (modules/ms_deform_attn.py:232-264 and :437-452): view/flatten, cat of the current and temporal logits, one
// softmax over all K = L*Pc + Wt*L*Pt taps, two slices made contiguous, `ref + off / (W, H)` for the current and
// for the temporal taps -- and autograd runs all of it backwards again.  At the DeVIS encoder shape that is
// 178 MB of locations + 89 MB of weights written and re-read per layer-clip and direction.
// Here the kernels read the RAW Linear outputs:
//     off_curr (T,Lq,M,L,Pc,2), logit_curr (T,Lq,M,L*Pc), off_temporal (T,Lq,M,Wt*L,Pt,2), logit_temporal (T,Lq,M,Wt*L*Pt)
// plus the reference points ref (T,Lq,L,2), and the lane that prepares a tap does
//     loc = ref[level] + off / (W_level, H_level)        (current taps; __fdiv_rn/__fadd_rn == torch's div, add)
//     loc = ref[level 0] + off / (W_level, H_level)      (temporal taps start from the level-0 point, :447)
//     w   = exp(logit - rowmax) / rowsum                 (rowmax, rowsum over all K taps of the (query, head))
// The backward returns d/d(off) = grad_loc / (W, H) and d/d(logit) = w * (grad_w - sum_k w_k grad_w_k) directly.
// Template GEN = false is that encoder form and nothing else (its hot loop pays for no generality).  GEN = true adds what
// the DECODER's prologue needs (ms_deform_attn.py:320-404), where the taps are 1000x fewer and the point is to replace
// ~100 small elementwise launches per layer, not bytes:
//     box reference points (ref_dim 4):  loc = ref.xy + ((off / P) * ref.wh) * 0.5                        (:369-371, :390-394)
//     temporal taps start from the level's own point of the query's frame (tref_mode 1, :346-347) or, instance aware,
//     from the SAME query's point in the sampled frame (tref_mode 2, :342-344)
//     the sampling locations and softmax weights are written out as by-products (the module's 5-tuple, :414)
//     d/d(ref) is accumulated (float atomics on a (T, Lq, L, ref_dim) tensor; decoder layer 0 learns its reference points)
// Work split, tap exchange, reductions: identical to msda_fwd.cuh / msda_bwd.cuh (LPG = 8, D = 32).
#pragma once
#include "msda_bwd.cuh"
#include "msda_common.cuh"
#include "msda_fwd.cuh"

namespace devis {

struct FusedArgs {
    const void *value;
    const float *ref;          // (T, Lq, L, ref_dim)
    int ref_dim;               // 2: points (x, y); 4: boxes (x, y, w, h)                                  [GEN]
    int tref_mode;             // reference point of a temporal tap: 0 level 0 of the query's frame (encoder),
                               // 1 the tap's level, query's frame; 2 the tap's level, sampled frame      [GEN]
    float inv_p[2];            // box form: 1 / points per slot (torch divides by a scalar as x * (1/s))   [GEN]
    float *loc_out[2];         // optional by-products of the forward, laid out like the unfused operands  [GEN]
    float *aw_out[2];
    float *grad_ref;           // backward, optional: (T, Lq, L, ref_dim), zero-filled by the caller       [GEN]
    const float *off[2];       // raw sampling offsets, current / temporal
    const float *logit[2];     // raw attention logits, current / temporal
    int n_slots[2];
    int P[2];
    int n_seg;
    ClipTable src;
    OpDims d;
    const int *q_perm;
    // forward
    void *out;
    // backward
    const void *grad_out;
    void *grad_value;          // fp32 (bf16 under HALF_ACC)
    DetScale det;              // deterministic mode (DET kernels): 64-bit fixed-point accumulators replace grad_value
    float *grad_off[2];
    float *grad_logit[2];
    int park_iters;            // > 0: shared memory holds (weight, d/d weight) of that many exchanges per thread
    const uint8_t *mask;       // padding mask (T, S), nonzero = the value row reads as zero (unmasked_live) [MASK]
};

// softmax statistics of one (query, head) row over both segments, computed by the LPG lanes of its group
template <int LPG = 8>
__device__ __forceinline__ void row_softmax_stats(const FusedArgs &a, size_t row, int j, bool live, float &rmax,
                                                  float &rinv)
{
    // Rows of up to 96 logits (DeVIS: 16 current + 80 temporal) are loaded ONCE, all loads in flight together, and kept
    // in registers for both passes; same order of operations as the general loops below, hence the same bits.
    constexpr int R = 96 / LPG;
    const int K0 = a.n_slots[0] * a.P[0], K1 = a.n_seg > 1 ? a.n_slots[1] * a.P[1] : 0;
    // (8-lane groups only: with 4 lanes the 24 registers cost the bf16 forward more than the loads save, 530 -> 545 us)
    if (LPG == 8 && K0 % LPG == 0 && K0 + K1 <= R * LPG) {
        float v[R];
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const int e = j + i * LPG;
            v[i] = -INFINITY;
            if (live && e < K0 + K1) v[i] = __ldg(e < K0 ? a.logit[0] + row * K0 + e : a.logit[1] + row * K1 + (e - K0));
        }
        float mx = v[0];
#pragma unroll
        for (int i = 1; i < R; ++i) mx = fmaxf(mx, v[i]);
#pragma unroll
        for (int o = LPG / 2; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o, LPG));
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < R; ++i)
            if (live && j + i * LPG < K0 + K1) sum += expf(v[i] - mx);
#pragma unroll
        for (int o = LPG / 2; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o, LPG);
        rmax = live ? mx : 0.f;
        rinv = live ? 1.f / sum : 0.f;
        return;
    }
    float mx = -INFINITY;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int K = a.n_slots[sg] * a.P[sg];
        const float *lg = a.logit[sg] + row * K;
        for (int k = j; k < K; k += LPG)
            if (live) mx = fmaxf(mx, __ldg(lg + k));
    }
#pragma unroll
    for (int o = LPG / 2; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o, LPG));
    float sum = 0.f;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int K = a.n_slots[sg] * a.P[sg];
        const float *lg = a.logit[sg] + row * K;
        for (int k = j; k < K; k += LPG)
            if (live) sum += expf(__ldg(lg + k) - mx);
    }
#pragma unroll
    for (int o = LPG / 2; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o, LPG);
    rmax = live ? mx : 0.f;
    rinv = live ? 1.f / sum : 0.f;
}

// raw operands of one tap as the Linear layers wrote them; loaded one exchange AHEAD of their use (like
// msda_fwdv_kernel's load_taps) so that their DRAM latency hides under the 32 corner gathers of the exchange before
struct RawTap {
    float2 off;   // sampling offset (pixels of the tap's level; box form: in units of box size / (2 P))
    float4 rf;    // reference point (x, y) or box (x, y, w, h) the tap starts from
    float lg;     // attention logit
    int ref_row;  // GEN: row of `ref` / `grad_ref` this tap reads (in units of ref_dim floats)
};

template <bool GEN = false>
__device__ __forceinline__ RawTap load_raw_tap(const FusedArgs &a, int sg, size_t row, size_t qrow, int k, bool live)
{
    RawTap r;
    r.off = make_float2(0.f, 0.f);
    r.rf = make_float4(0.f, 0.f, 0.f, 0.f);
    r.lg = 0.f;
    r.ref_row = 0;
    const int P = a.P[sg], K = a.n_slots[sg] * P;
    if (live && k < K) {
        const int slot = div_p(k, P, pow2_shift(P));
        const int level = mod_l(slot, a.src.L, pow2_shift(a.src.L));
        r.off = ld_stream_f2(reinterpret_cast<const float2 *>(a.off[sg] + row * K * 2) + k);
        if (!GEN) {
            const float2 p = __ldg(reinterpret_cast<const float2 *>(a.ref + (qrow * a.src.L + (sg == 0 ? level : 0)) * 2));
            r.rf.x = p.x;
            r.rf.y = p.y;
        } else {
            size_t rrow = qrow;
            int lvl = level;
            if (sg == 1) {
                if (a.tref_mode == 0) {
                    lvl = 0;
                } else if (a.tref_mode == 2) {
                    const int outer = (int)(qrow / (size_t)a.d.Lq);
                    const int frame = a.src.frame[outer * a.src.Wt + slot / a.src.L];
                    rrow = (size_t)((long long)qrow + (long long)(frame - outer) * a.d.Lq);
                }
            }
            r.ref_row = (int)(rrow * a.src.L + lvl);
            const float *rp = a.ref + (size_t)r.ref_row * a.ref_dim;
            const float2 p = __ldg(reinterpret_cast<const float2 *>(rp));
            r.rf.x = p.x;
            r.rf.y = p.y;
            if (a.ref_dim == 4) {
                const float2 wh = __ldg(reinterpret_cast<const float2 *>(rp + 2));
                r.rf.z = wh.x;
                r.rf.w = wh.y;
            }
        }
        r.lg = __ldg(a.logit[sg] + row * K + k);      // in L1 since row_softmax_stats
    }
    return r;
}

// the fused prologue on prefetched operands:  loc = ref + off / (W, H)  with torch's own rounding (IEEE division, then
// addition),  w = exp(logit - rowmax) / rowsum;  box form (GEN, ref_dim 4): loc = ref.xy + ((off * (1/P)) * ref.wh) * 0.5,
// every product rounded separately, in torch's left-to-right order (ms_deform_attn.py:369-371)
template <bool GEN = false>
__device__ __forceinline__ void raw_to_operands(const FusedArgs &a, int sg, const RawTap &r, const int4 sl, float rmax,
                                                float rinv, float &x, float &y, float &w)
{
    if (GEN && a.ref_dim == 4) {
        x = __fadd_rn(r.rf.x, __fmul_rn(__fmul_rn(__fmul_rn(r.off.x, a.inv_p[sg]), r.rf.z), 0.5f));
        y = __fadd_rn(r.rf.y, __fmul_rn(__fmul_rn(__fmul_rn(r.off.y, a.inv_p[sg]), r.rf.w), 0.5f));
    } else {
        x = __fadd_rn(r.rf.x, __fdiv_rn(r.off.x, (float)sl.y));
        y = __fadd_rn(r.rf.y, __fdiv_rn(r.off.y, (float)sl.x));
    }
    w = expf(r.lg - rmax) * rinv;
}

// Dead corners skipped, virtual top-left addressing (consume_tap16v, msda_fwd.cuh); ROWB: bytes of one value row as a
// compile-time constant, 0 = known at run time only.  Signed offsets: value < 2 GiB (the launcher refuses larger ones).
// measured (round 2, fused-prologue forward at the DeVIS layer-clip): 2 taps in flight at 2 blocks per SM 580 us, 1 tap
// at 2 / 3 blocks 605 / 595 us -- the opposite of msda_fwdv_kernel (1 tap, 3 blocks: 480 us against 489 us)
#ifndef DEVIS_FUSED_FWD_MIN_BLOCKS
#define DEVIS_FUSED_FWD_MIN_BLOCKS 2
#endif
#ifndef DEVIS_FUSED_FWD_TB
#define DEVIS_FUSED_FWD_TB 2
#endif
// MASK: a.mask is given; a masked corner's live bit is cleared, so its gather is never issued
template <Elem E, int QPG, bool GEN = false, int ROWB = 0, bool MASK = false>
__global__ void __launch_bounds__(256, DEVIS_FUSED_FWD_MIN_BLOCKS) tmsda_fused_fwd_kernel(const FusedArgs a)
{
    constexpr int LPG = 8;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y, n_slots_total = a.n_slots[0] + (a.n_seg > 1 ? a.n_slots[1] : 0);
    build_slots(s_slot, a.src, a.d, outer, n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + n_slots_total) + (threadIdx.x >> 5) * (2 * Tap16x8::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x % LPG, g = (threadIdx.x & 31) / LPG, grp = threadIdx.x / LPG, QC = blockDim.x / LPG;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;
    const L2Policy pol = make_l2_policy();
    bool qlive[QPG];
    size_t qrow[QPG], row[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        const int qi = (qchunk * QPG + i) * QC + grp;
        qlive[i] = qi < Lq;
        const int q = qlive[i] ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
        qrow[i] = (size_t)outer * Lq + q;
        row[i] = qrow[i] * M + m;
    }

    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kQuadBytes;
    asm volatile("" : "+l"(vbase));

    float rmax[QPG], rinv[QPG];
    float4 acc[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        row_softmax_stats(a, row[i], j, qlive[i], rmax[i], rinv[i]);
        acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    float4 v[DEVIS_FUSED_FWD_TB][4];        // gather destinations of consume_tap16v (see ldg_f4_if)
#pragma unroll
    for (int u = 0; u < DEVIS_FUSED_FWD_TB; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) v[u][e] = make_float4(0.f, 0.f, 0.f, 0.f);

    RawTap nxt[QPG];
#pragma unroll
    for (int i = 0; i < QPG; ++i) nxt[i] = load_raw_tap<GEN>(a, 0, row[i], qrow[i], j, qlive[i]);
    int slot_base = 0, parity = 0;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.P[sg], K = a.n_slots[sg] * P, pshift = pow2_shift(P);   // P % 4 == 0 (checked by the launcher)
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;
            const bool klive = k < K;
            const int ls = klive ? div_p(k, P, pshift) : 0;        // slot within the segment
            const int4 sl = s_slot[slot_base + ls];
            const unsigned my_pitch = (unsigned)sl.y * rowbytes;
            const unsigned pitch_lo = __shfl_sync(0xffffffffu, my_pitch, 0, 8);
            const unsigned pitch_hi = __shfl_sync(0xffffffffu, my_pitch, 4, 8);
            RawTap cur[QPG];
#pragma unroll
            for (int i = 0; i < QPG; ++i) cur[i] = nxt[i];
            if (k0 + LPG < K) {
#pragma unroll
                for (int i = 0; i < QPG; ++i) nxt[i] = load_raw_tap<GEN>(a, sg, row[i], qrow[i], k + LPG, qlive[i]);
            } else if (sg + 1 < a.n_seg) {
#pragma unroll
                for (int i = 0; i < QPG; ++i) nxt[i] = load_raw_tap<GEN>(a, sg + 1, row[i], qrow[i], j, qlive[i]);
            }
#pragma unroll
            for (int i = 0; i < QPG; ++i) {
                const bool live = klive && qlive[i];
                float x = 0.f, y = 0.f, w = 0.f;
                if (live) raw_to_operands<GEN>(a, sg, cur[i], sl, rmax[i], rinv[i], x, y, w);
                if (GEN && live) {      // the decoder module's 5-tuple: locations and weights as the unfused path lays them out
                    if (a.loc_out[sg]) reinterpret_cast<float2 *>(a.loc_out[sg] + row[i] * K * 2)[k] = make_float2(x, y);
                    if (a.aw_out[sg]) a.aw_out[sg][row[i] * K + k] = w;
                }
                float *buf = xbuf + parity * Tap16x8::kWordsPerWarpBuf;
                parity ^= 1;
                TapGeomV t = tap_geometry_v(x, y, sl, live);
                if (MASK) t.live = unmasked_live(a.mask, t.rowv, sl.y, t.live);
                *reinterpret_cast<uint4 *>(buf + Tap16x8::word(j, g)) = make_tap16v(t, w, rowbytes);
                __syncwarp();
                consume_tap16v<E, ROWB, DEVIS_FUSED_FWD_TB>(buf, g, rowbytes, pitch_lo, pitch_hi, vbase, acc[i], v);
            }
        }
        slot_base += a.n_slots[sg];
    }
#pragma unroll
    for (int i = 0; i < QPG; ++i) {
        if (!qlive[i]) continue;
        if constexpr (E != Elem::F32)
            reinterpret_cast<uint2 *>(a.out)[row[i] * LPG + j] = pack_16x4<E>(acc[i]);
        else
            st_stream_f4(reinterpret_cast<float4 *>(a.out) + row[i] * LPG + j, acc[i]);
    }
}

// Four lanes per (query, head), 8 channels per lane (msda_fwd8v_kernel's shape): the forward of choice for 16-bit value
// (bf16 or fp16), whose 64-byte rows cost 0.75 instead of 1.0 data-pipe cycles when 4 lanes fetch 16 bytes each.
// 16-bit value only (the fp32 form of this shape loses to the eight-lane kernel); dead corners skipped, consume_tap16x4v
template <Elem E, int ROWB, bool MASK = false>
__global__ void __launch_bounds__(256) tmsda_fused_fwd8_kernel(const FusedArgs a)
{
    static_assert(E != Elem::F32, "16-bit value only");
    constexpr int LPG = 4;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y, n_slots_total = a.n_slots[0] + (a.n_seg > 1 ? a.n_slots[1] : 0);
    build_slots(s_slot, a.src, a.d, outer, n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + n_slots_total) + (threadIdx.x >> 5) * (2 * Tap16::kWordsPerWarpBuf);

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x & 3, g = (threadIdx.x & 31) >> 2, grp = threadIdx.x >> 2, QC = blockDim.x >> 2;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;
    const int qi = qchunk * QC + grp;
    const bool qlive = qi < Lq;
    const int q = qlive ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
    const size_t qrow = (size_t)outer * Lq + q, row = qrow * M + m;

    constexpr unsigned kLaneBytes = 16u;                   // 8 channels
    const unsigned rowbytes = (unsigned)(M * LPG) * kLaneBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kLaneBytes;
    asm volatile("" : "+l"(vbase));

    float rmax, rinv;
    row_softmax_stats<LPG>(a, row, j, qlive, rmax, rinv);

    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    uint4 v[4];                             // gather destinations of consume_tap16x4v
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = make_uint4(0u, 0u, 0u, 0u);

    int slot_base = 0, parity = 0;
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.P[sg], K = a.n_slots[sg] * P, pshift = pow2_shift(P);   // P % 4 == 0: one slot per exchange, k < K always
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;
            const int4 sl = s_slot[slot_base + div_p(k0, P, pshift)];
            const unsigned pitch = (unsigned)sl.y * rowbytes;
            // loaded at use: with 8 groups per warp a prefetch one exchange ahead does not pay here (531 vs 524 us; the
            // same held for the unfused four-lane kernel, 431 vs 403 us)
            const RawTap cur = load_raw_tap<false>(a, sg, row, qrow, k, qlive);
            float x = 0.f, y = 0.f, w = 0.f;
            if (qlive) raw_to_operands<false>(a, sg, cur, sl, rmax, rinv, x, y, w);
            float *buf = xbuf + parity * Tap16::kWordsPerWarpBuf;
            parity ^= 1;
            TapGeomV t = tap_geometry_v(x, y, sl, qlive);
            if (MASK) t.live = unmasked_live(a.mask, t.rowv, sl.y, t.live);
            *reinterpret_cast<uint4 *>(buf + Tap16::word(j, g)) = make_tap16v(t, w, rowbytes);
            __syncwarp();
            consume_tap16x4v<E, ROWB>(buf, g, rowbytes, pitch, vbase, acc, v);
        }
        slot_base += a.n_slots[sg];
    }
    if (qlive) {
        const uint2 lo = pack_16x4<E>(make_float4(acc[0], acc[1], acc[2], acc[3]));
        const uint2 hi = pack_16x4<E>(make_float4(acc[4], acc[5], acc[6], acc[7]));
        reinterpret_cast<uint4 *>(a.out)[row * LPG + j] = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
}

// HALF_ACC: bf16 grad_value with packed bf16 reductions (see msda_bwd_kernel)
// DET (round 2): DEVIS_MSDA_FLAG_DETERMINISTIC inside the fused path -- the grad_value contributions go to 64-bit
// fixed-point accumulators with integer reductions (det_add4, msda_common.cuh) exactly as in msda_bwd_kernel, with the
// bound max|attn| = 1 (the weights are softmax outputs here); every other gradient of this kernel is written once, in a
// fixed order, so the whole backward is bit-identical run to run.
// MASK: a.mask is given.  TapGeom's row / column bits cannot describe one masked corner, so the record carries four
// per-corner bits (unmasked_corners) in bits 1-4 of the TL byte offset (value rows are >= 64 B; bit 0 is the sort tag of
// msda_bwd_sort.cuh, unused here); a dropped corner reads as zero and scatters nothing -- by selection, not by a product.
template <Elem E, bool HALF_ACC = false, bool GEN = false, bool DET = false, bool MASK = false>
__global__ void __launch_bounds__(256, DEVIS_BWD_MIN_BLOCKS) tmsda_fused_bwd_kernel(const FusedArgs a)
{
    static_assert(!(DET && HALF_ACC), "deterministic mode accumulates in fixed point");
    constexpr int LPG = 8;
    using X = TapExchange<LPG>;
    extern __shared__ int4 s_slot[];
    const int outer = blockIdx.y, n_slots_total = a.n_slots[0] + (a.n_seg > 1 ? a.n_slots[1] : 0);
    build_slots(s_slot, a.src, a.d, outer, n_slots_total);
    float *xbuf = reinterpret_cast<float *>(s_slot + n_slots_total) + (threadIdx.x >> 5) * (2 * X::kWordsPerWarpBuf);
    // softmax backward needs sum_k w_k val_k of the whole row before any d/d(logit) can be written: each thread parks the
    // (w, val) of the taps it prepared -- in shared memory when the row is short enough ([exchange][thread], conflict-free,
    // read back by the same thread: no barrier), else in grad_logit itself (re-read through L2: 13 % of the kernel's
    // stall samples sat in that epilogue, profiles/r1j_fused_bwd_stalls.json)
    float2 *s_park = reinterpret_cast<float2 *>(reinterpret_cast<float *>(s_slot + n_slots_total) +
                                                (blockDim.x >> 5) * (2 * X::kWordsPerWarpBuf)) + threadIdx.x;
    const bool park = a.park_iters > 0;

    const int M = a.d.M, Lq = a.d.Lq;
    const int j = threadIdx.x % LPG, g = (threadIdx.x & 31) / LPG, grp = threadIdx.x / LPG, QC = blockDim.x / LPG;
    const int qchunk = blockIdx.x / M, m = blockIdx.x - qchunk * M;
    const int qi = qchunk * QC + grp;
    const bool qlive = qi < Lq;
    const int q = qlive ? (a.q_perm ? a.q_perm[qi] : qi) : 0;
    const size_t qrow = (size_t)outer * Lq + q, row = qrow * M + m;

    float4 gg = make_float4(0.f, 0.f, 0.f, 0.f);
    if (qlive) {
        if constexpr (E != Elem::F32) gg = ldg_16x4<E>(reinterpret_cast<const uint2 *>(a.grad_out) + row * LPG + j);
        else gg = ldg_f4(reinterpret_cast<const float4 *>(a.grad_out) + row * LPG + j);
    }

    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(a.value) + (size_t)(m * LPG + j) * kQuadBytes;
    asm volatile("" : "+l"(vbase));
    static_assert(!HALF_ACC || E == Elem::BF16, "bf16 accumulation needs bf16 value");
    char *gvb = a.grad_value ? reinterpret_cast<char *>(a.grad_value) + (size_t)(m * LPG + j) * (HALF_ACC ? 8u : 16u) : nullptr;
    constexpr unsigned kGvShift = (E != Elem::F32 && !HALF_ACC) ? 1u : 0u;
    // deterministic mode: 8-byte accumulators, channels of a (row, head) permuted as in det_add4 (lane j starts at word j)
    char *detb = DET ? reinterpret_cast<char *>(a.det.acc) + (size_t)(m * LPG) * 32u + (size_t)j * 8u : nullptr;
    const float det_sh = DET ? ldexpf(1.f, kDetFracBits - det_exponent(a.det.max_bits)) : 0.f;

    float rmax, rinv;
    row_softmax_stats(a, row, j, qlive, rmax, rinv);

    float dotp = 0.f;   // this lane's share of sum_k w_k * d(out.grad_out)/d(w_k)
    int slot_base = 0, parity = 0, it = 0;
    RawTap nxt = load_raw_tap<GEN>(a, 0, row, qrow, j, qlive);
    for (int sg = 0; sg < a.n_seg; ++sg) {
        const int P = a.P[sg], K = a.n_slots[sg] * P, pshift = pow2_shift(P);
        float *goff = a.grad_off[sg] + row * K * 2;
        float *glog = a.grad_logit[sg] + row * K;
        for (int k0 = 0; k0 < K; k0 += LPG) {
            const int k = k0 + j;
            const bool live = k < K && qlive;
            const int ls = live ? div_p(k, P, pshift) : 0;
            const int4 sl = s_slot[slot_base + ls];
            const RawTap cur = nxt;
            if (k0 + LPG < K) nxt = load_raw_tap<GEN>(a, sg, row, qrow, k + LPG, qlive);
            else if (sg + 1 < a.n_seg) nxt = load_raw_tap<GEN>(a, sg + 1, row, qrow, j, qlive);
            float x = 0.f, y = 0.f, w = 0.f;
            if (live) raw_to_operands<GEN>(a, sg, cur, sl, rmax, rinv, x, y, w);
            const TapGeom t = tap_geometry(x, y, sl, live);
            float *buf = xbuf + parity * X::kWordsPerWarpBuf;
            parity ^= 1;
            X::publish(buf, j, g, t, w, rowbytes, MASK ? unmasked_corners(a.mask, t) << 1 : 0u);
            __syncwarp();

            float dsum[LPG][4];
#pragma unroll
            for (int jj = 0; jj < LPG; ++jj) {
                uint4 off;
                float4 c;
                X::fetch(buf, jj, g, off, c);
                unsigned corners = 15u;
                if (MASK) {
                    corners = (off.x >> 1) & 15u;
                    off.x &= ~30u;
                }
                float4 v00, v01, v10, v11;
                if constexpr (E != Elem::F32) {
                    v00 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.x));
                    v01 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.y));
                    v10 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.z));
                    v11 = ldg_16x4<E>(reinterpret_cast<const uint2 *>(vbase + off.w));
                } else {
                    v00 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.x));
                    v01 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.y));
                    v10 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.z));
                    v11 = ldg_f4(reinterpret_cast<const float4 *>(vbase + off.w));
                }
                if (MASK) {
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!(corners & 1u)) v00 = z, c.x = 0.f;
                    if (!(corners & 2u)) v01 = z, c.y = 0.f;
                    if (!(corners & 4u)) v10 = z, c.z = 0.f;
                    if (!(corners & 8u)) v11 = z, c.w = 0.f;
                }
                dsum[jj][0] = fmaf(v00.w, gg.w, fmaf(v00.z, gg.z, fmaf(v00.y, gg.y, v00.x * gg.x)));
                dsum[jj][1] = fmaf(v01.w, gg.w, fmaf(v01.z, gg.z, fmaf(v01.y, gg.y, v01.x * gg.x)));
                dsum[jj][2] = fmaf(v10.w, gg.w, fmaf(v10.z, gg.z, fmaf(v10.y, gg.y, v10.x * gg.x)));
                dsum[jj][3] = fmaf(v11.w, gg.w, fmaf(v11.z, gg.z, fmaf(v11.y, gg.y, v11.x * gg.x)));
                if (DET) {
                    if (c.x != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.x << (kGvShift + 1))), det_sh, c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w);
                    if (c.y != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.y << (kGvShift + 1))), det_sh, c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w);
                    if (c.z != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.z << (kGvShift + 1))), det_sh, c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w);
                    if (c.w != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(detb + ((size_t)off.w << (kGvShift + 1))), det_sh, c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w);
                } else if (gvb) {
                    if (c.x != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.x << kGvShift), c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w);
                    if (c.y != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.y << kGvShift), c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w);
                    if (c.z != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.z << kGvShift), c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w);
                    if (c.w != 0.f) red_add_quad<HALF_ACC>(gvb + ((size_t)off.w << kGvShift), c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w);
                }
            }
            float A[4];
            reduce_scatter_taps<LPG>(dsum, j, A);
            float gr[4] = {0.f, 0.f, 0.f, 0.f};   // GEN: this tap's d/d(ref x, y, w, h)
            if (live) {
                const bool hit = t.ok != 0u;
                const float hh = (t.ok & 1u) ? t.hh : 0.f, lh = (t.ok & 2u) ? t.lh : 0.f;
                const float hw = (t.ok & 4u) ? t.hw : 0.f, lw = (t.ok & 8u) ? t.lw : 0.f;
                const float l_in = (t.ok & 4u) ? 1.f : 0.f, r_in = (t.ok & 8u) ? 1.f : 0.f;
                const float t_in = (t.ok & 1u) ? 1.f : 0.f, b_in = (t.ok & 2u) ? 1.f : 0.f;
                const float val = hit ? hh * (hw * A[0] + lw * A[1]) + lh * (hw * A[2] + lw * A[3]) : 0.f;
                const float gx = hh * (r_in * A[1] - l_in * A[0]) + lh * (r_in * A[3] - l_in * A[2]);
                const float gy = hw * (b_in * A[2] - t_in * A[0]) + lw * (b_in * A[3] - t_in * A[1]);
                // d/d(loc) = (W gx w, H gy w) as in msda_bwd.cuh, then the chain rule of loc = ref + off / (W, H): the two
                // factors cancel (the reference's multiply-then-divide sequence differs from this by <= 1 ulp)
                if (!GEN) {
                    st_stream_f2(reinterpret_cast<float2 *>(goff) + k, hit ? make_float2(gx * w, gy * w) : make_float2(0.f, 0.f));
                } else {
                    // d/d(loc) in normalised coordinates, as msda_bwd.cuh writes it; then the chain rule of the prologue
                    const float glx = hit ? (float)sl.y * gx * w : 0.f, gly = hit ? (float)sl.x * gy * w : 0.f;
                    float2 go2;
                    if (a.ref_dim == 4) {
                        const float sx = a.inv_p[sg] * 0.5f;
                        go2 = make_float2(glx * (sx * cur.rf.z), gly * (sx * cur.rf.w));
                        gr[2] = glx * (cur.off.x * sx);
                        gr[3] = gly * (cur.off.y * sx);
                    } else {
                        go2 = hit ? make_float2(gx * w, gy * w) : make_float2(0.f, 0.f);
                    }
                    gr[0] = glx;
                    gr[1] = gly;
                    st_stream_f2(reinterpret_cast<float2 *>(goff) + k, go2);
                }
                if (park) s_park[it * blockDim.x] = make_float2(w, val);
                else glog[k] = val;       // parked; finished below once the row's  sum_k w_k val_k  is known
                dotp = fmaf(w, val, dotp);
            }
            if (GEN && a.grad_ref) {
                // the 4 taps an aligned lane quad prepared belong to one slot (P % 4 == 0), hence to one reference point:
                // sum them in the quad, one atomic per component
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    gr[c] += __shfl_xor_sync(0xffffffffu, gr[c], 1, 4);
                    gr[c] += __shfl_xor_sync(0xffffffffu, gr[c], 2, 4);
                }
                if (live && (j & 3) == 0) {
                    float *gp = a.grad_ref + (size_t)cur.ref_row * a.ref_dim;
                    atomicAdd(gp, gr[0]);
                    atomicAdd(gp + 1, gr[1]);
                    if (a.ref_dim == 4) {
                        atomicAdd(gp + 2, gr[2]);
                        atomicAdd(gp + 3, gr[3]);
                    }
                }
            }
            ++it;
        }
        slot_base += a.n_slots[sg];
    }
    // softmax backward:  d/d(logit_k) = w_k * (val_k - sum_j w_j val_j)
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) dotp += __shfl_xor_sync(0xffffffffu, dotp, o, 8);
    if (qlive) {
        it = 0;
        for (int sg = 0; sg < a.n_seg; ++sg) {
            const int K = a.n_slots[sg] * a.P[sg];
            float *glog = a.grad_logit[sg] + row * K;
            const float *lg = a.logit[sg] + row * K;
            if (park) {
                for (int k = j; k < K; k += 8, ++it) {
                    const float2 wv = s_park[it * blockDim.x];
                    st_stream_f(glog + k, wv.x * (wv.y - dotp));
                }
                it += (j >= K % 8 && K % 8 != 0) ? 1 : 0;     // exchanges are counted per group, not per lane
            } else {
                for (int k = j; k < K; k += 8) {
                    const float w = expf(__ldg(lg + k) - rmax) * rinv;
                    glog[k] = w * (glog[k] - dotp);
                }
            }
        }
    }
}

}  // namespace devis
