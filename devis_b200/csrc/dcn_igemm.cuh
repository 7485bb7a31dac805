// dcn_igemm.cuh -- modulated deformable convolution forward as an IMPLICIT GEMM on the 5th-generation tensor cores
// (tcgen05.mma, accumulator in TMEM) for the WIDE layers of DeVIS's mask head (SURVEY.md section 8 f-3).
//
// The reference evaluates every 3x3 layer of MaskHeadConv (src/models/deformable_segmentation.py:323-380) with
// torchvision.ops.deform_conv2d (:262-267): deformable_im2col writes a (N*Ho*Wo, 9*C) column matrix and at::addmm
// contracts it with the weights.  For the wide layers (264 -> 264, 264 -> 128 at 12 x 20, 136 -> 64 at 23 x 40) round 1
// kept that shape -- a channels-last im2col kernel plus a cuBLAS fp32 GEMM -- because the contraction dominates and the
// CUDA cores cannot do better than SGEMM.  Here the column matrix is never written: a CTA owns 128 output pixels (the MMA
// M dimension) and ALL output channels (N <= 512 TMEM columns) and walks K = 9 kernel positions x C channels in stages
// of 32 channels:
//   * 8 producer warps gather + interpolate + modulate the stage's 128 x 32 column block straight into shared memory in
//     the tensor core's canonical K-major SWIZZLE_128B layout (a pixel's 32 channels = one 128-byte row, written by an
//     8-lane group as 8 x 16 bytes, conflict-free), using the same per-tap arithmetic as dcn_im2col_kernel;
//   * one thread streams the matching 32-channel slab of the pre-packed weights (already in the swizzled image) with
//     ONE cp.async.bulk per stage, completing on the stage's mbarrier;
//   * one thread issues tcgen05.mma.kind::tf32 (M = 128, N = Cout padded to 16, K = 8 per instruction), D in TMEM;
//     tcgen05.commit releases the stage back to the producers;
//   * the 4 epilogue warps read the accumulator with tcgen05.ld, add the bias and store channels-last.
// Precision.  TF32 keeps 10 mantissa bits, which the fp32 parity bar (1e-5) does not allow.  Default = 3xTF32: both
// operands are split x = hi + lo (hi = x rounded to TF32, lo = x - hi, exact in fp32) and D accumulates
// hi*hi + lo*hi + hi*lo in fp32 -- the error drops to ~2^-21 relative per product, the level of an fp32 SGEMM.  With
// `precision = 1` (torch.backends.cuda.matmul.allow_tf32, which torchvision's addmm honours too) a single TF32 pass runs.
#pragma once
#include "deform_conv.cuh"

namespace devis {

constexpr int kIgBM = 128;          // output pixels per CTA (MMA M)
constexpr int kIgBK = 32;           // channels per pipeline stage = one 128-byte swizzle row of tf32
constexpr int kIgProducers = 256;   // 8 warps gather; warps 0-3 also run the epilogue
constexpr int kIgThreads = kIgProducers + 64;   // + weight-loader warp + MMA warp
constexpr int kIgATile = kIgBM * 128;           // bytes of one A tile (128 rows x 128 B)
constexpr int kIgGeomBytes = 2 * kIgBM * 32;    // two generations of per-pixel tap geometry
constexpr int kIgMaxStages = 4;

struct IgArgs {
    const float *input;     // (N, H, W, C) channels-last
    const float *offset;    // (N, 2K, Ho, Wo)
    const float *mask;      // (N, K, Ho, Wo) or nullptr
    const float *wpacked;   // [k][chunk][hi|lo][Npad rows][32 floats, 16-byte chunks XOR-swizzled with row % 8]
    const float *bias;      // (Cout) or nullptr
    float *out;             // (N*Ho*Wo, Cout)
    DcnDims d;
    int Cout, Npad, nchunks, stages, split;
    int n0, n1;             // the N dimension is issued as one or two MMAs (n1 = 0: one)
    int tmem_cols;
    long long P;            // N * Ho * Wo
};

// ---- PTX wrappers -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ig_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ig_mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void ig_mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void ig_mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ig_mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    }
}
// generic-proxy shared-memory writes (the producers' st.shared) -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void ig_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void ig_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void ig_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void ig_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void ig_tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] x B[smem desc], tf32 inputs, fp32 accumulation; accumulate = 0 overwrites D
__device__ __forceinline__ void ig_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void ig_tmem_ld16(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ float ig_tf32_rna(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// shared-memory matrix descriptor of a K-major SWIZZLE_128B operand tile (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
// start address >> 4 | leading byte offset (16 B, unused inside a 128-byte swizzle row) >> 4 at bit 16 | stride byte
// offset (8 rows x 128 B = 1024 B) >> 4 at bit 32 | descriptor version 1 at bit 46 | layout type 2 at bit 61
__device__ __forceinline__ uint64_t ig_smem_desc(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (bit 4), A = B = TF32 (2 at bits 7, 10), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ inline uint32_t ig_instr_desc(int n)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kIgBM >> 4) << 24);
}

// ---- weight packing ---------------------------------------------------------------------------------------------------
// torchvision weight (Cout, C, kh, kw) -> [k][chunk][hi|lo][Npad][32]: the exact shared-memory image of a stage's B tile
__global__ void __launch_bounds__(256) dcn_igemm_pack_kernel(const float *__restrict__ w, float *__restrict__ packed, int Cout,
                                                             int C, int K, int Npad, int nchunks)
{
    const long long total = (long long)K * nchunks * Npad * kIgBK;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int col = (int)(i % kIgBK);
        const int n = (int)((i / kIgBK) % Npad);
        const int chunk = (int)((i / ((long long)kIgBK * Npad)) % nchunks);
        const int k = (int)(i / ((long long)kIgBK * Npad * nchunks));
        const int c = chunk * kIgBK + col;
        const float v = (n < Cout && c < C) ? w[((long long)n * C + c) * K + k] : 0.f;
        const float hi = ig_tf32_rna(v), lo = ig_tf32_rna(v - hi);     // lo rounded here (the tensor core would truncate it)
        const long long block = ((long long)k * nchunks + chunk) * 2 * Npad * kIgBK;
        const int phys = n * kIgBK + ((((col >> 2) ^ (n & 7)) << 2) | (col & 3));
        packed[block + phys] = hi;
        packed[block + (long long)Npad * kIgBK + phys] = lo;
    }
}

// ---- the kernel ---------------------------------------------------------------------------------------------------------
// MINB: thread blocks per SM the register budget is sized for.  The wide layers are bound by shared memory to one block
// per SM; the narrow ones (few 32-channel stages per kernel position) are latency chains inside a block and want a
// second / third block on the SM to overlap them.
template <int MINB>
__global__ void __launch_bounds__(kIgThreads, MINB) dcn_igemm_fwd_kernel(const IgArgs a)
{
    extern __shared__ unsigned char ig_smem_raw[];
    // 1024-byte alignment: the swizzle pattern is a function of the address bits
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(ig_smem_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_a = a.split ? 2 : 1;
    const int b_bytes = a.Npad * 128;                               // one B tile (hi or lo)
    const int stage_bytes = n_a * kIgATile + n_a * b_bytes;
    unsigned char *geom = smem + (size_t)a.stages * stage_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(geom + kIgGeomBytes);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kIgMaxStages + 1);
    const uint32_t bar_full = ig_smem_u32(bars), bar_empty = ig_smem_u32(bars + kIgMaxStages),
                   bar_accum = ig_smem_u32(bars + 2 * kIgMaxStages);
    const uint32_t smem_base = ig_smem_u32(smem);

    if (tid == 0) {
        for (int s = 0; s < a.stages; ++s) {
            ig_mbar_init(bar_full + 8 * s, kIgProducers + 1);       // every producer thread + the loader's expect_tx
            ig_mbar_init(bar_empty + 8 * s, 1);                     // one tcgen05.commit
        }
        ig_mbar_init(bar_accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kIgProducers / 32 + 1) {                            // the MMA warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(ig_smem_u32(tmem_slot)),
                     "r"((uint32_t)a.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    ig_tc_fence_before();
    __syncthreads();
    ig_tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const DcnDims &d = a.d;
    const int K = d.kh * d.kw, n_iter = K * a.nchunks;
    const long long pix0 = (long long)blockIdx.x * kIgBM;

    if (tid < kIgProducers) {
        // ================= producers: column block of (128 pixels x 32 channels) per stage =================
        const int j = tid & 7, g = tid >> 3;                        // 32 groups of 8 lanes; group g owns pixels g, g+32, g+64, g+96
        const int plane = d.Ho * d.Wo;
        for (int k = 0; k < K; ++k) {
            int4 *grow = reinterpret_cast<int4 *>(geom + (k & 1) * (kIgBM * 32));
            float4 *gfac = reinterpret_cast<float4 *>(grow + kIgBM);
            if (tid < kIgBM) {                                      // geometry of (pixel tid, kernel position k), once
                const long long pix = pix0 + tid;
                int4 rows = make_int4(-1, -1, -1, -1);                  // -1: corner outside the map, never read
                float4 fac = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pix < a.P) {
                    const int n = (int)(pix / plane), pp = (int)(pix - (long long)n * plane);
                    const DcnTapId id = dcn_tap_id(pp, n, k, d);
                    float h, w, m;
                    dcn_sample_point(a.offset, a.mask, id, d, h, w, m);
                    const DcnTap<float> t = dcn_tap(h, w, d.H, d.W);
                    const int img = n * d.H * d.W;
                    rows = make_int4(t.ok[0] ? (img + t.row[0]) * d.C : -1, t.ok[1] ? (img + t.row[1]) * d.C : -1,
                                     t.ok[2] ? (img + t.row[2]) * d.C : -1, t.ok[3] ? (img + t.row[3]) * d.C : -1);
                    fac = make_float4(m * t.w[0], m * t.w[1], m * t.w[2], m * t.w[3]);
                }
                grow[tid] = rows;
                gfac[tid] = fac;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kIgProducers) : "memory");
            for (int chunk = 0; chunk < a.nchunks; ++chunk) {
                const int it = k * a.nchunks + chunk, s = it % a.stages;
                const uint32_t phase = (uint32_t)(it / a.stages) & 1u;
                unsigned char *a_hi = smem + (size_t)s * stage_bytes;
                unsigned char *a_lo = a_hi + kIgATile;
                const int c0 = chunk * kIgBK + 4 * j;
                const bool live = c0 < d.C;
                // gather and interpolate into registers FIRST: none of it needs the stage's shared memory, so the 16
                // corner loads of this thread are in flight while the tensor core still reads the slot's previous tiles
                float4 v[4][4];
                float4 f[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int p = g + 32 * i;
                    const int4 r = grow[p];
                    f[i] = gfac[p];
                    v[i][0] = dcn_corner4(reinterpret_cast<const float4 *>(a.input + max(r.x, 0) + c0), live && r.x >= 0);
                    v[i][1] = dcn_corner4(reinterpret_cast<const float4 *>(a.input + max(r.y, 0) + c0), live && r.y >= 0);
                    v[i][2] = dcn_corner4(reinterpret_cast<const float4 *>(a.input + max(r.z, 0) + c0), live && r.z >= 0);
                    v[i][3] = dcn_corner4(reinterpret_cast<const float4 *>(a.input + max(r.w, 0) + c0), live && r.w >= 0);
                }
                float4 col[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {                       // dcn_im2col_kernel's arithmetic, term for term
                    col[i].x = f[i].x * v[i][0].x + f[i].y * v[i][1].x + f[i].z * v[i][2].x + f[i].w * v[i][3].x;
                    col[i].y = f[i].x * v[i][0].y + f[i].y * v[i][1].y + f[i].z * v[i][2].y + f[i].w * v[i][3].y;
                    col[i].z = f[i].x * v[i][0].z + f[i].y * v[i][1].z + f[i].z * v[i][2].z + f[i].w * v[i][3].z;
                    col[i].w = f[i].x * v[i][0].w + f[i].y * v[i][1].w + f[i].z * v[i][2].w + f[i].w * v[i][3].w;
                }
                ig_mbar_wait(bar_empty + 8 * s, phase ^ 1u);        // the MMAs that read this slot last have completed
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int p = g + 32 * i;
                    const float4 c = col[i];
                    const float4 hi = make_float4(ig_tf32_rna(c.x), ig_tf32_rna(c.y), ig_tf32_rna(c.z), ig_tf32_rna(c.w));
                    const int at = p * 128 + ((j ^ (p & 7)) << 4);
                    *reinterpret_cast<float4 *>(a_hi + at) = hi;
                    if (a.split)     // lo rounded to TF32 here (the tensor core would truncate it)
                        *reinterpret_cast<float4 *>(a_lo + at) = make_float4(ig_tf32_rna(c.x - hi.x), ig_tf32_rna(c.y - hi.y),
                                                                             ig_tf32_rna(c.z - hi.z), ig_tf32_rna(c.w - hi.w));
                }
                ig_fence_async_smem();
                ig_mbar_arrive(bar_full + 8 * s);
            }
        }
        // ================= epilogue (warps 0-3): TMEM -> registers -> (+ bias) -> global, channels-last =================
        if (warp < 4) {
            ig_mbar_wait(bar_accum, 0u);
            ig_tc_fence_after();
            const long long pix = pix0 + warp * 32 + lane;
            float *orow = a.out + pix * a.Cout;
            for (int col0 = 0; col0 < a.Npad; col0 += 16) {
                float acc[16];
                ig_tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)col0, acc);
                if (pix < a.P) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int c = col0 + 4 * q;
                        if (c < a.Cout) {
                            float4 o = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
                            if (a.bias) {
                                const float4 b = __ldg(reinterpret_cast<const float4 *>(a.bias + c));
                                o.x += b.x;
                                o.y += b.y;
                                o.z += b.z;
                                o.w += b.w;
                            }
                            *reinterpret_cast<float4 *>(orow + c) = o;
                        }
                    }
                }
            }
        }
    } else if (warp == kIgProducers / 32) {
        // ================= weight loader: one bulk copy per stage =================
        if (lane == 0) {
            const uint32_t bytes = (uint32_t)(n_a * b_bytes);
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % a.stages;
                const uint32_t phase = (uint32_t)(it / a.stages) & 1u;
                ig_mbar_wait(bar_empty + 8 * s, phase ^ 1u);
                ig_mbar_expect_tx(bar_full + 8 * s, bytes);
                ig_bulk_g2s(smem_base + (uint32_t)(s * stage_bytes + n_a * kIgATile),
                            a.wpacked + (size_t)it * 2 * a.Npad * kIgBK, bytes, bar_full + 8 * s);
            }
        }
    } else {
        // ================= MMA issuer: one thread =================
        if (lane == 0) {
            const uint32_t idesc0 = ig_instr_desc(a.n0), idesc1 = ig_instr_desc(a.n1 > 0 ? a.n1 : 16);
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % a.stages, chunk = it % a.nchunks;
                const uint32_t phase = (uint32_t)(it / a.stages) & 1u;
                ig_mbar_wait(bar_full + 8 * s, phase);
                ig_tc_fence_after();
                const uint32_t a_hi = smem_base + (uint32_t)(s * stage_bytes), a_lo = a_hi + kIgATile;
                const uint32_t b_hi = a_hi + (uint32_t)(n_a * kIgATile), b_lo = b_hi + (uint32_t)b_bytes;
                const int rem = d.C - chunk * kIgBK;
                const int ksteps = rem >= kIgBK ? kIgBK / 8 : (rem + 7) / 8;
                for (int ks = 0; ks < ksteps; ++ks) {
                    const uint32_t koff = (uint32_t)ks * 32u;        // 8 tf32 = 32 bytes along the swizzled row
                    const uint32_t acc = (it > 0 || ks > 0) ? 1u : 0u;
                    for (int half = 0; half < (a.n1 > 0 ? 2 : 1); ++half) {
                        const uint32_t dcol = tmem_base + (half ? (uint32_t)a.n0 : 0u);
                        const uint32_t brow = half ? (uint32_t)a.n0 * 128u : 0u;
                        const uint32_t idesc = half ? idesc1 : idesc0;
                        const uint64_t da_hi = ig_smem_desc(a_hi + koff), db_hi = ig_smem_desc(b_hi + brow + koff);
                        ig_mma_tf32(dcol, da_hi, db_hi, idesc, acc);
                        if (a.split) {
                            ig_mma_tf32(dcol, ig_smem_desc(a_lo + koff), db_hi, idesc, 1u);
                            ig_mma_tf32(dcol, da_hi, ig_smem_desc(b_lo + brow + koff), idesc, 1u);
                        }
                    }
                }
                ig_tc_commit(bar_empty + 8 * s);                    // stage free once these MMAs have read it
            }
            ig_tc_commit(bar_accum);                                // accumulator complete
        }
    }
    ig_tc_fence_before();
    __syncthreads();
    if (warp == kIgProducers / 32 + 1) {
        ig_tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)a.tmem_cols) : "memory");
    }
}

}  // namespace devis
