// msda_bwd_sort.cuh -- whole-clip backward with per-block SORTED pre-aggregation of grad_value (encoder form).
//
// msda_bwd_kernel is co-limited by the rate at which reductions can LEAVE an SM (5.2 cycles per 128-byte row for
// red.global.add.v4.f32, benchmarks/micro/smem_accumulate.cu; 79 % busy) and the L1 data pipe, and in the encoder most of
// those rows are duplicates: the
// 64 pixel-queries of an 8 x 8 tile sample the same few hundred rows of every (frame, level) map.  Shared-memory float
// atomics are CAS loops on sm_100a and fixed-point integer windows cost 16 ATOMS per lane and tap (msda_bwd_win.cuh,
// slower than the direct scatter), so the duplicates are merged by SORTING instead:
//
//   * a thread block owns one head and one 8 x 8 pixel tile of one pyramid level (query i == pixel i: encoder
//     self-attention, deformable_transformer.py:184-198; the same reduction for the plain per-call op is
//     ms_deform_attn_col2im_bilinear's atomicAdd scatter, ms_deform_im2col_cuda.cuh:87-159) and walks the taps in
//     BATCHES of 8 taps per query = 2 slots (two levels of one sampled frame) x 4 points: 512 taps, 2048 corner
//     contributions {coefficient, query, target row};
//   * around the tile's footprint in every level lies a WINDOW of rows (tile rectangle scaled to the level, grown by
//     `margin` pixels, clipped to the map); a contribution's key is its row's index in the window.  The lane that
//     prepares a tap takes a rank inside each target row with ONE native integer ATOMS.ADD on that row's counter;
//   * an exclusive scan of the counters turns (key, rank) into a position: a counting sort by target row, 8-byte
//     records, no float atomics;
//   * every 8-lane group then walks an equal share of the sorted records, accumulates  coef x grad_out[query]  (the
//     tile's 64 grad_out rows sit in shared memory) for its 4 channels in registers while the row stays the same, and
//     sends ONE vector reduction per run to grad_value;
//   * taps outside their window, and levels without a window, take msda_bwd_kernel's direct scatter.  Window placement
//     is a performance heuristic only: every contribution is added exactly once either way, with the same products
//     (only the order of the float sums differs).
//
// grad_sampling_loc and grad_attn_weight do not depend on any of this and are bit-identical to msda_bwd_kernel's.
//
// Where it is used (DESIGN.md 3.5, 7.1): the DETERMINISTIC mode of the encoder form (template DET: 64-bit fixed-point
// sums, bit-identical to the direct deterministic scatter, 3.24 -> 2.68 ms).  In the default float mode the sort removes
// 82 % of the reductions but its shared-memory traffic makes the kernel slower than the direct scatter (1.93 vs 1.43 ms:
// the L1/shared data pipe is at 71 % for the whole run), so there it stays opt-in (tuning key 6 = 3).
#pragma once
#include "msda_bwd.cuh"

#ifndef DEVIS_BWDS_MIN_BLOCKS
#define DEVIS_BWDS_MIN_BLOCKS 3
#endif

namespace devis {

constexpr int kSortTile = 8;                                       // queries form kSortTile x kSortTile pixel tiles
constexpr int kSortThreads = 256;                                  // 32 lane groups x 2 queries each
constexpr int kSortQueries = kSortTile * kSortTile;
constexpr int kSortMaxKeys = 1024;                                 // window rows of one level pair (scan width)
constexpr int kSortRecords = kSortQueries * 8 * 4;                 // 64 queries x 8 taps x 4 corners per batch

struct SortArgs {
    BwdArgs<ClipTable> b;
    int tiles_x[kMaxLevels];     // tiles per row of level l
    int tile_start[kMaxLevels];  // first tile index of level l
    int n_tiles;
    int margin;                  // window margin around the tile footprint, in pixels of the sampled level
    int min_level;               // levels below this one keep the direct scatter (they have the fewest duplicates)
    int lut_entries;             // capacity of the key -> row table (host: (L / 2) * kSortMaxKeys)
};

// dynamic shared memory of msda_bwds_kernel (bytes)
__host__ __device__ inline size_t sort_smem_bytes(int n_slots_total, int lut_entries)
{
    return (size_t)n_slots_total * 16 + 5 * kMaxLevels * 4 + 16 * 4 +
           (size_t)(kSortThreads / 32) * TapExchange<8>::kBytesPerWarp + (size_t)kSortQueries * 32 * 4 +
           2 * (size_t)kSortMaxKeys * 4 + 2 * (size_t)kSortRecords * 8 + (((size_t)lut_entries * 2 + 15) & ~(size_t)15);
}

// DET (DEVIS_MSDA_FLAG_DETERMINISTIC): every contribution is converted exactly to 64-bit fixed point (the integers
// msda_bwd_kernel's det_add4 adds, same scale) and both the in-register run sums and the global reductions are integer
// additions: associative, so the result does not depend on the arrival order of the ranks -- and is bit-identical to
// the direct deterministic scatter, with 5x fewer 64-bit reductions leaving the SM.
template <Elem E, bool DET = false>
__global__ void __launch_bounds__(kSortThreads, DEVIS_BWDS_MIN_BLOCKS) msda_bwds_kernel(const SortArgs a)
{
    constexpr int LPG = 8;
    constexpr int P = 4;                                            // points per slot (host-checked)
    using X = TapExchange<LPG>;
    extern __shared__ int4 s_slot[];
    const BwdArgs<ClipTable> &b = a.b;
    const int outer = blockIdx.y;
    const int L = b.src.L;
    build_slots(s_slot, b.src, b.d, outer, b.n_slots_total);
    int *s_lw = reinterpret_cast<int *>(s_slot + b.n_slots_total);           // per level: x_lo, y_lo, ww, wh, first key
    int *s_misc = s_lw + 5 * kMaxLevels;                                     // [0..7] warp sums, [8] records, [9] keys
    float *xbuf_all = reinterpret_cast<float *>(s_misc + 16);
    const int warp = threadIdx.x >> 5;
    float *xbuf = xbuf_all + warp * (2 * X::kWordsPerWarpBuf);
    float *s_go = xbuf_all + (kSortThreads / 32) * 2 * X::kWordsPerWarpBuf;  // [64 tile pixels][32 channels]
    int *s_cnt = reinterpret_cast<int *>(s_go + kSortQueries * 32);          // [2][kSortMaxKeys]
    uint2 *s_stage = reinterpret_cast<uint2 *>(s_cnt + 2 * kSortMaxKeys);    // [kSortRecords] {coef, key|rank|query|valid}
    uint2 *s_sorted = s_stage + kSortRecords;                                // [kSortRecords] {coef, query | key << 6}
    unsigned short *s_lut = reinterpret_cast<unsigned short *>(s_sorted + kSortRecords);  // key -> row inside its level

    const int M = b.d.M, Lq = b.d.Lq;
    const int j = threadIdx.x % LPG;
    const int g = (threadIdx.x & 31) / LPG;
    const int grp = threadIdx.x / LPG;
    constexpr int NG = kSortThreads / LPG;
    constexpr int QPC = kSortQueries / NG;
    const int tile = blockIdx.x / M, m = blockIdx.x - tile * M;

    // which level and which tile of it
    int lq = 0;
    while (lq + 1 < L && tile >= a.tile_start[lq + 1]) ++lq;
    const int tl = tile - a.tile_start[lq];
    const int ty0 = (tl / a.tiles_x[lq]) * kSortTile, tx0 = (tl - (tl / a.tiles_x[lq]) * a.tiles_x[lq]) * kSortTile;
    const int Hq = b.src.H[lq], Wq = b.src.W[lq];
    const int th = min(kSortTile, Hq - ty0), tw = min(kSortTile, Wq - tx0);
    const int n_pix = th * tw;

    // windows: the tile rectangle mapped into every level; a level pair shares one key space of kSortMaxKeys rows
    if (threadIdx.x == 0) {
        for (int l = 0; l < L; ++l) {
            const int H = b.src.H[l], W = b.src.W[l];
            // pixel centres of the tile's first / last column and row, in level-l pixel coordinates
            const float fx0 = ((float)tx0 + 0.5f) / (float)Wq * (float)W - 0.5f;
            const float fx1 = ((float)(tx0 + tw - 1) + 0.5f) / (float)Wq * (float)W - 0.5f;
            const float fy0 = ((float)ty0 + 0.5f) / (float)Hq * (float)H - 0.5f;
            const float fy1 = ((float)(ty0 + th - 1) + 0.5f) / (float)Hq * (float)H - 0.5f;
            const int x_lo = max((int)floorf(fx0) - a.margin, 0), x_hi = min((int)floorf(fx1) + 1 + a.margin, W - 1);
            const int y_lo = max((int)floorf(fy0) - a.margin, 0), y_hi = min((int)floorf(fy1) + 1 + a.margin, H - 1);
            int ww = x_hi - x_lo + 1, wh = y_hi - y_lo + 1;
            if (l < a.min_level || ww < 1 || wh < 1 || ww * wh > kSortMaxKeys) ww = wh = 0;
            s_lw[5 * l + 0] = x_lo;
            s_lw[5 * l + 1] = y_lo;
            s_lw[5 * l + 2] = ww;
            s_lw[5 * l + 3] = wh;
        }
        int used = 0;
        for (int l = 0; l < L; l += 2) {
            // the finer level of a pair gives way first
            if (s_lw[5 * l + 2] * s_lw[5 * l + 3] + s_lw[5 * l + 7] * s_lw[5 * l + 8] > kSortMaxKeys)
                s_lw[5 * l + 2] = s_lw[5 * l + 3] = 0;
            s_lw[5 * l + 4] = used;
            used += s_lw[5 * l + 2] * s_lw[5 * l + 3];
            s_lw[5 * l + 9] = used;
            used += s_lw[5 * l + 7] * s_lw[5 * l + 8];
        }
        if (used > a.lut_entries) {   // cannot happen with the host's sizing; keep the kernel safe anyway
            for (int l = 0; l < L; ++l) s_lw[5 * l + 2] = s_lw[5 * l + 3] = 0, s_lw[5 * l + 4] = 0;
            used = 0;
        }
        s_misc[9] = used;
    }
    for (int i = threadIdx.x; i < 2 * kSortMaxKeys; i += kSortThreads) s_cnt[i] = 0;
    __syncthreads();
    {   // key -> row offset inside the level's map
        const int n_keys_all = s_misc[9];
        for (int key = threadIdx.x; key < n_keys_all; key += kSortThreads) {
            int l = 0;
            while (l + 1 < L && key >= s_lw[5 * (l + 1) + 4]) ++l;
            // skip levels without a window that share their first key with the next level
            while (s_lw[5 * l + 2] == 0 && l + 1 < L) ++l;
            const int rel = key - s_lw[5 * l + 4], ww = s_lw[5 * l + 2];
            const int wy = rel / ww, wx = rel - wy * ww;
            s_lut[key] = (unsigned short)((s_lw[5 * l + 1] + wy) * b.src.W[l] + s_lw[5 * l] + wx);
        }
    }

    // grad_out rows of the tile: registers for the corner dot products, shared memory for the sorted accumulation
    float4 go[QPC];
#pragma unroll
    for (int i = 0; i < QPC; ++i) {
        const int p = grp + i * NG;
        go[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p < n_pix) {
            const int q = b.src.lsi[lq] + (ty0 + p / tw) * Wq + tx0 + (p - (p / tw) * tw);
            const size_t row = ((size_t)outer * Lq + q) * M + m;
            if constexpr (E != Elem::F32) go[i] = ldg_16x4<E>(reinterpret_cast<const uint2 *>(b.grad_out) + row * LPG + j);
            else go[i] = ldg_f4(reinterpret_cast<const float4 *>(b.grad_out) + row * LPG + j);
        }
        reinterpret_cast<float4 *>(s_go)[p * LPG + j] = go[i];
    }
    __syncthreads();

    constexpr unsigned kQuadBytes = E != Elem::F32 ? 8u : 16u;
    const unsigned rowbytes = (unsigned)(M * LPG) * kQuadBytes;
    const char *vbase = reinterpret_cast<const char *>(b.value) + (size_t)(m * LPG + j) * kQuadBytes;
    asm volatile("" : "+l"(vbase));
    // fp32 grad_value (host-checked), or the deterministic mode's 8-byte accumulators in det_add4's permuted order
    char *gvb = DET ? reinterpret_cast<char *>(b.det.acc) + (size_t)(m * LPG) * 32u + (size_t)j * 8u
                    : reinterpret_cast<char *>(b.grad_value) + (size_t)(m * LPG + j) * 16u;
    constexpr unsigned kGvShift = (E != Elem::F32 ? 1u : 0u) + (DET ? 1u : 0u);
    const size_t gv_rowbytes = (size_t)(M * LPG) * (DET ? 32u : 16u);
    const float det_sh = DET ? ldexpf(1.f, kDetFracBits - det_exponent(b.det.max_bits)) : 0.f;

    int slot_base = 0, parity = 0, cp = 0;
    for (int sg = 0; sg < b.n_seg; ++sg) {
        const int K = b.seg[sg].n_slots * P;
        const float *loc = reinterpret_cast<const float *>(b.seg[sg].loc);
        const float *aw = reinterpret_cast<const float *>(b.seg[sg].aw);
        float *gloc = reinterpret_cast<float *>(b.seg[sg].grad_loc);
        float *gaw = reinterpret_cast<float *>(b.seg[sg].grad_aw);
        for (int k0 = 0; k0 < K; k0 += LPG) {
            // ---- B: taps of this batch: geometry, ranks, gathers, grad_loc / grad_aw ---------------------------
            const int k = k0 + j;
            const int slot0 = slot_base + k0 / P;                    // the batch's two slots: slot0, slot0 + 1
            const int slot = slot0 + (j >> 2);
            const int la = (k0 / P) % L;                             // their levels: la, la + 1
            const int lvl = la + (j >> 2);
            const int4 sl = s_slot[slot];
            const int kb0 = s_lw[5 * la + 4];                        // first key of the pair
            const int w_xlo = s_lw[5 * lvl], w_ylo = s_lw[5 * lvl + 1], w_ww = s_lw[5 * lvl + 2], w_wh = s_lw[5 * lvl + 3];
            const int w_kb = s_lw[5 * lvl + 4] - kb0;
            int *cnt = s_cnt + cp * kSortMaxKeys;
#pragma unroll
            for (int qi = 0; qi < QPC; ++qi) {
                const int p = grp + qi * NG;
                const bool live = p < n_pix;
                const int q = live ? b.src.lsi[lq] + (ty0 + p / tw) * Wq + tx0 + (p - (p / tw) * tw) : 0;
                const size_t row = ((size_t)outer * Lq + q) * M + m;
                float2 xy = make_float2(0.f, 0.f);
                float w = 0.f;
                if (live) {
                    xy = __ldg(reinterpret_cast<const float2 *>(loc + row * K * 2) + k);
                    w = __ldg(aw + row * K + k);
                }
                const TapGeom t = tap_geometry(xy.x, xy.y, sl, live);
                // window position of the tap: all four (clamped) corner rows must lie inside
                bool sorted = false;
                int kTL = 0, kdx = 0, kdy = 0;
                if (t.ok != 0u && w_ww > 0) {
                    const int dx = t.rTR - t.rTL;                    // 0 / 1 column
                    const int dy = (t.rBL != t.rTL) ? 1 : 0;         // 0 / 1 row
                    const int wx = t.x0c - w_xlo, wy = t.y0c - w_ylo;
                    if (wx >= 0 && wx + dx < w_ww && wy >= 0 && wy + dy < w_wh) {
                        sorted = true;
                        kTL = w_kb + wy * w_ww + wx;
                        kdx = dx;
                        kdy = dy * w_ww;
                    }
                }
                float *buf = xbuf + parity * X::kWordsPerWarpBuf;
                parity ^= 1;
                X::publish(buf, j, g, t, w, rowbytes, sorted ? 1u : 0u);
                // the four contributions' coefficients: the products X::fetch hands to the direct path
                const float fT = (t.ok & 1u) ? w * t.hh : 0.f, fB = (t.ok & 2u) ? w * t.lh : 0.f;
                const float fL = (t.ok & 4u) ? t.hw : 0.f, fR = (t.ok & 8u) ? t.lw : 0.f;
                const float cf[4] = {fT * fL, fT * fR, fB * fL, fB * fR};
                const int ky[4] = {kTL, kTL + kdx, kTL + kdy, kTL + kdy + kdx};
                int rk[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    rk[c] = -1;
                    if (sorted && cf[c] != 0.f) rk[c] = atomicAdd(cnt + ky[c], 1);
                }
                __syncwarp();

                const float4 gg = go[qi];
                float dsum[LPG][4];
#pragma unroll
                for (int jj = 0; jj < LPG; ++jj) {
                    uint4 off;
                    float4 c;
                    X::fetch(buf, jj, g, off, c);
                    const bool direct = (off.x & 1u) == 0u;
                    off.x &= ~1u;
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
                    dsum[jj][0] = fmaf(v00.w, gg.w, fmaf(v00.z, gg.z, fmaf(v00.y, gg.y, v00.x * gg.x)));
                    dsum[jj][1] = fmaf(v01.w, gg.w, fmaf(v01.z, gg.z, fmaf(v01.y, gg.y, v01.x * gg.x)));
                    dsum[jj][2] = fmaf(v10.w, gg.w, fmaf(v10.z, gg.z, fmaf(v10.y, gg.y, v10.x * gg.x)));
                    dsum[jj][3] = fmaf(v11.w, gg.w, fmaf(v11.z, gg.z, fmaf(v11.y, gg.y, v11.x * gg.x)));
                    if (direct) {
                        if (DET) {
                            if (c.x != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(gvb + ((size_t)off.x << kGvShift)), det_sh, c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w);
                            if (c.y != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(gvb + ((size_t)off.y << kGvShift)), det_sh, c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w);
                            if (c.z != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(gvb + ((size_t)off.z << kGvShift)), det_sh, c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w);
                            if (c.w != 0.f) det_add4<LPG>(reinterpret_cast<long long *>(gvb + ((size_t)off.w << kGvShift)), det_sh, c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w);
                        } else {
                            if (c.x != 0.f) red_add_f4(reinterpret_cast<float *>(gvb + ((size_t)off.x << kGvShift)), c.x * gg.x, c.x * gg.y, c.x * gg.z, c.x * gg.w);
                            if (c.y != 0.f) red_add_f4(reinterpret_cast<float *>(gvb + ((size_t)off.y << kGvShift)), c.y * gg.x, c.y * gg.y, c.y * gg.z, c.y * gg.w);
                            if (c.z != 0.f) red_add_f4(reinterpret_cast<float *>(gvb + ((size_t)off.z << kGvShift)), c.z * gg.x, c.z * gg.y, c.z * gg.z, c.z * gg.w);
                            if (c.w != 0.f) red_add_f4(reinterpret_cast<float *>(gvb + ((size_t)off.w << kGvShift)), c.w * gg.x, c.w * gg.y, c.w * gg.z, c.w * gg.w);
                        }
                    }
                }

                float Ac[4];
                reduce_scatter_taps<LPG>(dsum, j, Ac);
                if (live) {
                    const bool hit = t.ok != 0u;
                    const float hh = (t.ok & 1u) ? t.hh : 0.f, lh = (t.ok & 2u) ? t.lh : 0.f;
                    const float hw = (t.ok & 4u) ? t.hw : 0.f, lw = (t.ok & 8u) ? t.lw : 0.f;
                    const float l_in = (t.ok & 4u) ? 1.f : 0.f, r_in = (t.ok & 8u) ? 1.f : 0.f;
                    const float t_in = (t.ok & 1u) ? 1.f : 0.f, b_in = (t.ok & 2u) ? 1.f : 0.f;
                    const float val = hh * (hw * Ac[0] + lw * Ac[1]) + lh * (hw * Ac[2] + lw * Ac[3]);
                    const float gx = hh * (r_in * Ac[1] - l_in * Ac[0]) + lh * (r_in * Ac[3] - l_in * Ac[2]);
                    const float gy = hw * (b_in * Ac[2] - t_in * Ac[0]) + lw * (b_in * Ac[3] - t_in * Ac[1]);
                    gaw[row * K + k] = hit ? val : 0.f;
                    reinterpret_cast<float2 *>(gloc + row * K * 2)[k] =
                        hit ? make_float2((float)sl.y * gx * w, (float)sl.x * gy * w) : make_float2(0.f, 0.f);
                }
                // unsorted records of this tap (all four written every batch: stale ones must not survive)
                {
                    unsigned meta[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        meta[c] = rk[c] >= 0 ? (0x80000000u | (unsigned)ky[c] | ((unsigned)rk[c] << 11) | ((unsigned)p << 22)) : 0u;
                    uint4 *dst = reinterpret_cast<uint4 *>(s_stage + (qi * kSortThreads + threadIdx.x) * 4);
                    dst[0] = make_uint4(__float_as_uint(cf[0]), meta[0], __float_as_uint(cf[1]), meta[1]);
                    dst[1] = make_uint4(__float_as_uint(cf[2]), meta[2], __float_as_uint(cf[3]), meta[3]);
                }
            }
            __syncthreads();

            // ---- C: exclusive scan of the row counters -> first position of every row ------------------------
            {
                int4 v = reinterpret_cast<int4 *>(cnt)[threadIdx.x];
                const int s0 = v.x, s1 = s0 + v.y, s2 = s1 + v.z, s3 = s2 + v.w;
                int incl = s3;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int n = __shfl_up_sync(0xffffffffu, incl, o);
                    if ((threadIdx.x & 31) >= o) incl += n;
                }
                if ((threadIdx.x & 31) == 31) s_misc[warp] = incl;
                __syncthreads();
                int before = 0;
                for (int wv = 0; wv < warp; ++wv) before += s_misc[wv];
                const int excl = before + incl - s3;
                reinterpret_cast<int4 *>(cnt)[threadIdx.x] = make_int4(excl, excl + s0, excl + s1, excl + s2);
                if (threadIdx.x == kSortThreads - 1) s_misc[8] = excl + s3;
                __syncthreads();
            }

            // ---- D: scatter the records to their sorted positions; clear the other counter buffer -------------
#pragma unroll 4
            for (int i = threadIdx.x; i < kSortRecords; i += kSortThreads) {
                const uint2 r = s_stage[i];
                if (r.y & 0x80000000u) {
                    const unsigned key = r.y & 0x7ffu, rank = (r.y >> 11) & 0x7ffu, qq = (r.y >> 22) & 0x3fu;
                    s_sorted[cnt[key] + rank] = make_uint2(r.x, qq | (key << 6));
                }
            }
            reinterpret_cast<int4 *>(s_cnt + (cp ^ 1) * kSortMaxKeys)[threadIdx.x] = make_int4(0, 0, 0, 0);
            __syncthreads();

            // ---- E: every lane group reduces an equal share of the sorted records, one reduction per row run --
            {
                const int n_rec = s_misc[8];
                const int chunk = ((n_rec + NG - 1) / NG) | 1;       // odd: the 4 groups of a warp read different banks
                const int beg = grp * chunk, end = min(beg + chunk, n_rec);
                const int n_a = s_lw[5 * (la + 1) + 4] - kb0;        // keys below belong to slot0, the rest to slot0 + 1
                const int za = s_slot[slot0].z, zb = s_slot[slot0 + 1].z;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                long long ai[4] = {0, 0, 0, 0};
                int cur = -1;
                auto flush = [&](int key) {
                    const size_t vrow = (size_t)((key < n_a ? za : zb) + (int)s_lut[kb0 + key]);
                    if (DET) {
                        unsigned long long *p = reinterpret_cast<unsigned long long *>(gvb + vrow * gv_rowbytes);
#pragma unroll
                        for (int c = 0; c < 4; ++c) atomicAdd(p + c * LPG, (unsigned long long)ai[c]);
                    } else {
                        red_add_f4(reinterpret_cast<float *>(gvb + vrow * gv_rowbytes), acc.x, acc.y, acc.z, acc.w);
                    }
                };
                uint2 r = make_uint2(0u, 0u);
                if (beg < end) r = s_sorted[beg];
                for (int i = beg; i < end; ++i) {
                    const uint2 rn = s_sorted[min(i + 1, end - 1)];
                    const int key = (int)(r.y >> 6), qq = (int)(r.y & 63u);
                    const float4 gq = reinterpret_cast<const float4 *>(s_go)[qq * LPG + j];
                    if (key != cur) {
                        if (cur >= 0) flush(cur);
                        acc = make_float4(0.f, 0.f, 0.f, 0.f);
                        ai[0] = ai[1] = ai[2] = ai[3] = 0;
                        cur = key;
                    }
                    const float c = __uint_as_float(r.x);
                    if (DET) {
                        // the same integers det_add4 adds for the direct path: round(c * g) to float, exact scaling
                        ai[0] += __float2ll_rn(__fmul_rn(c, gq.x) * det_sh);
                        ai[1] += __float2ll_rn(__fmul_rn(c, gq.y) * det_sh);
                        ai[2] += __float2ll_rn(__fmul_rn(c, gq.z) * det_sh);
                        ai[3] += __float2ll_rn(__fmul_rn(c, gq.w) * det_sh);
                    } else {
                        acc.x = fmaf(c, gq.x, acc.x);
                        acc.y = fmaf(c, gq.y, acc.y);
                        acc.z = fmaf(c, gq.z, acc.z);
                        acc.w = fmaf(c, gq.w, acc.w);
                    }
                    r = rn;
                }
                if (cur >= 0) flush(cur);
            }
            cp ^= 1;
        }
        slot_base += b.seg[sg].n_slots;
    }
}

}  // namespace devis
