// msda_capi.cu -- C ABI (include/devis_msda.h) of the sm_100a multi-scale deformable attention library.
//
// Host side of the drop-in boundary: validates the operands the way the reference's C++ host does
// (cuda/ms_deform_attn_cuda.cu:28-52,93-119), picks a kernel, launches on the caller's stream and
// reports launch failures as error codes.  No torch types, no allocation, no synchronisation.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "../../include/devis_msda.h"
#include "msda_bwd.cuh"
#include "msda_bwd_sort.cuh"
#include "msda_common.cuh"
#include "msda_fwd.cuh"
#include "msda_generic.cuh"
#include "tmsda_fused.cuh"

#include "capi_common.h"

using namespace devis;

namespace {

std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_family_launches[DEVIS_MSDA_KERNEL_FAMILIES];
thread_local int t_last_cuda_error = 0;

// Keys of devis_msda_set_tuning; include/devis_msda.h documents them, and the numbers are part of the ABI.
enum TuningKey {
    kKeyFwdThreads = 0,    // forward threads per block
    kKeyFwdQpg = 1,        // forward queries per lane group
    kKeyBwdThreads = 2,    // backward threads per block
    kKeyBwdQpg = 3,        // backward queries per lane group
    kKeyDirectScatter = 6, // 1: the deterministic mode uses the direct 64-bit scatter instead of the sorted kernel
    kKeySortMargin = 7,    // sorted kernel: window margin in pixels (0 = 6)
    kKeySortMinLevel = 9,  // sorted kernel: first level with a window + 1 (0 = all levels)
};

// Launch-shape knobs of the developer benchmarks (benchmarks/sweep.py, variant A/B runs).  They only exist when the
// process was started with DEVIS_MSDA_TUNING=1: a product process cannot have its kernel selection changed behind its
// back (devis_msda_set_tuning returns DEVIS_MSDA_ERR_UNSUPPORTED), and every key then reads 0 = built-in heuristic.
std::atomic<int> g_tuning_store[16];
bool tuning_enabled()
{
    static const bool on = [] {
        const char *e = std::getenv("DEVIS_MSDA_TUNING");
        return e && e[0] == '1';
    }();
    return on;
}
struct TuningView {
    struct Key {
        int k;
        int load() const { return tuning_enabled() ? g_tuning_store[k].load() : 0; }
    };
    Key operator[](TuningKey k) const { return Key{k}; }
} g_tuning;

}  // namespace

// grid of the grid-stride helper kernels: 8 blocks per SM of the CURRENT device (queried once per device)
int devis_capi_helper_blocks()
{
    static std::atomic<int> cached[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148 * 8;
    int v = cached[dev].load(std::memory_order_relaxed);
    if (v == 0) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        v = sms * 8;
        cached[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

// shared with the other translation units of the library (capi_common.h)
int devis_capi_cuda_fail(cudaError_t e)
{
    t_last_cuda_error = (int)e;
    return DEVIS_MSDA_ERR_CUDA;
}

int devis_capi_check_launch(int family)
{
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (family >= 0 && family < DEVIS_MSDA_KERNEL_FAMILIES) g_family_launches[family].fetch_add(1, std::memory_order_relaxed);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? DEVIS_MSDA_OK : devis_capi_cuda_fail(e);
}

namespace {

int cuda_fail(cudaError_t e) { return devis_capi_cuda_fail(e); }

// DEVIS_MSDA_BF16 and DEVIS_MSDA_F16 take the same kernels, launch shapes and byte thresholds (2-byte elements); only
// the widening on load and the rounding on store differ (Elem)
bool is_16bit(int dtype) { return dtype == DEVIS_MSDA_BF16 || dtype == DEVIS_MSDA_F16; }
int check_launch(int family) { return devis_capi_check_launch(family); }

size_t elem_size(int dtype) { return dtype == DEVIS_MSDA_F64 ? 8 : is_16bit(dtype) ? 2 : 4; }

// ---- compile-time dispatch ---------------------------------------------------------------------------------------
// Each helper calls a generic lambda with a std::integral_constant (or a type tag) for a run-time value.  The lambdas
// guard the combinations no kernel is built for with `if constexpr`, so a dispatch instantiates only what can run.

// value / output / grad_output type of the lane-group, fused, sorted and helper kernels: DEVIS_MSDA_BF16, DEVIS_MSDA_F16,
// anything else Elem::F32 (fp64 never reaches a lane-group kernel)
template <class F>
auto with_elem(int dtype, F &&f)
{
    if (dtype == DEVIS_MSDA_BF16) return f(std::integral_constant<Elem, Elem::BF16>{});
    if (dtype == DEVIS_MSDA_F16) return f(std::integral_constant<Elem, Elem::F16>{});
    return f(std::integral_constant<Elem, Elem::F32>{});
}

// element type of the generic kernels: all four codes
template <class T>
struct TypeTag {
    using type = T;
};
template <class F>
void with_scalar(int dtype, F &&f)
{
    if (dtype == DEVIS_MSDA_F32) f(TypeTag<float>{});
    else if (dtype == DEVIS_MSDA_F64) f(TypeTag<double>{});
    else if (dtype == DEVIS_MSDA_F16) f(TypeTag<__half>{});
    else f(TypeTag<__nv_bfloat16>{});
}

// v as the first of Vs it equals, or as the last of Vs
template <int V, int... Rest, class F>
void with_int(int v, F &&f)
{
    if constexpr (sizeof...(Rest) == 0) f(std::integral_constant<int, V>{});
    else if (v == V) f(std::integral_constant<int, V>{});
    else with_int<Rest...>(v, f);
}

// ROWB of the D = 32 kernels: with 8 heads the size of a value row is a compile-time immediate of the gathers, else 0
template <Elem E, class F>
void with_row_bytes(int M, F &&f)
{
    constexpr int kRow8 = 8 * 32 * (E == Elem::F32 ? 4 : 2);
    with_int<kRow8, 0>(M == 8 ? kRow8 : 0, f);
}

// channel counts served by the grouped-lane kernels: D = 4 * LPG.  They address value with 32-bit byte
// offsets, so tensors of 4 GiB and more go to the generic kernels.
int lanes_per_group(int dtype, const OpDims &d)
{
    if (dtype == DEVIS_MSDA_F64) return 0;
    const unsigned long long bytes = (unsigned long long)d.outer * d.S * d.M * d.D * elem_size(dtype);
    if (bytes >= (1ull << 32)) return 0;
    return d.D == 32 ? 8 : d.D == 16 ? 4 : 0;
}

size_t exchange_bytes(int lpg, int threads)
{
    return (size_t)(threads / 32) * (lpg == 8 ? TapExchange<8>::kBytesPerWarp : TapExchange<4>::kBytesPerWarp);
}

struct LaunchShape {
    int threads, qpg;
};

// Launch shape of the grouped-lane and fused kernels.  Defaults from benchmarks/sweep.py at the DeVIS layer-clip shape
// (profiles/r1f_sweep_*.json): the backward wants 128-thread blocks (84 registers -> 5 blocks = 20 warps per SM
// against 2 x 8 warps with 256 threads: 1428 vs 1536 us), the fp32 forward 256 threads x 2 queries per group
// (527 vs 549 us), the bf16 forward 128 threads, the fused bf16 / fp16 forward 64 threads below 1024 queries.  Tuning
// keys 0, 1 (forward) or 2, 3 (backward) override (developer tools only); max_qpg is the largest QPG the chosen kernel
// is instantiated with -- anything else would launch a grid that does not cover the queries.  A key QPG the kernel has
// no instantiation for is brought to one it has, or with clamp_key_qpg = false (the fused forward) left to the default.
enum ShapeKind { kShapeFwdF32, kShapeFwdBf16, kShapeFusedFwd16, kShapeBwd };

LaunchShape pick_shape(int Lq, ShapeKind kind, int max_qpg, bool clamp_key_qpg = true)
{
    const bool bwd = kind == kShapeBwd;
    LaunchShape s;
    s.threads = g_tuning[bwd ? kKeyBwdThreads : kKeyFwdThreads].load();
    s.qpg = g_tuning[bwd ? kKeyBwdQpg : kKeyFwdQpg].load();
    if (!clamp_key_qpg && (s.qpg < 1 || s.qpg > max_qpg)) s.qpg = 0;
    if (s.threads == 0) {
        const int big = kind == kShapeFwdF32 ? 256 : 128;
        s.threads = Lq >= 1024 ? big : (Lq >= 128 && kind != kShapeFusedFwd16) ? 128 : 64;
    }
    if (s.qpg == 0) s.qpg = (kind == kShapeFwdF32 && Lq >= 2048) ? 2 : 1;
    if (s.threads < 32) s.threads = 32;
    if (s.threads > 256) s.threads = 256;
    s.threads = (s.threads / 32) * 32;
    if (s.qpg != 1 && s.qpg != 2 && s.qpg != 4) s.qpg = 1;
    if (s.qpg > max_qpg) s.qpg = max_qpg;
    return s;
}

// grid of the lane-group kernels: blocks of queries_per_block lane groups with qpg queries each, one head per block
int lane_group_grid(const OpDims &d, int queries_per_block, int qpg, dim3 &grid)
{
    const long long per_block = (long long)queries_per_block * qpg;
    const long long chunks = ((long long)d.Lq + per_block - 1) / per_block;
    if (chunks * d.M > 0x7fffffffLL) return DEVIS_MSDA_ERR_TOO_LARGE;
    grid = dim3((unsigned)(chunks * d.M), (unsigned)d.outer);
    return DEVIS_MSDA_OK;
}

// grid of the generic kernels: one warp per (query, head)
constexpr int kGenericThreads = 128;
int generic_grid(const OpDims &d, dim3 &grid)
{
    constexpr int wpc = kGenericThreads / 32;
    const long long blocks = ((long long)d.Lq * d.M + wpc - 1) / wpc;
    if (blocks > 0x7fffffffLL) return DEVIS_MSDA_ERR_TOO_LARGE;
    grid = dim3((unsigned)blocks, (unsigned)d.outer);
    return DEVIS_MSDA_OK;
}

template <class SlotSrc>
int launch_forward(const FwdArgs<SlotSrc> &a, int dtype, cudaStream_t st)
{
    const OpDims &d = a.d;
    if (d.outer == 0 || d.Lq == 0) return DEVIS_MSDA_OK;
    size_t smem = (size_t)a.n_slots_total * sizeof(int4);
    const int lpg = lanes_per_group(dtype, d);
    dim3 grid;
    int rc;
    // D = 32 with P % 4 == 0 in every segment and value below 2 GiB (signed 32-bit tap offsets): the round-2 kernels with
    // 16-byte tap records and the dead corners skipped.  fp32 value: eight lanes x 4 channels (msda_fwdv_kernel); bf16 / fp16
    // value: four lanes x 8 channels (msda_fwd8v_kernel: 64-byte rows cost 0.75 instead of 1.0 data-pipe cycles that way;
    // for fp32 the four-lane shape needs LDG.E.256 and loses, profiles/r2s_fwd_wide_f32_variants.json).  Everything else
    // takes msda_fwd_kernel below.
    bool compact = lpg == 8 && (unsigned long long)d.outer * d.S * d.M * d.D * elem_size(dtype) < (1ull << 31);
    for (int sg = 0; sg < a.n_seg; ++sg) compact = compact && (a.seg[sg].P % 4 == 0);
    if (compact && is_16bit(dtype)) {
        const LaunchShape s = pick_shape(d.Lq, kShapeFwdBf16, 2);
        smem += (size_t)(s.threads / 32) * Tap16::kBytesPerWarp;
        if ((rc = lane_group_grid(d, s.threads / 4, s.qpg, grid))) return rc;
        with_elem(dtype, [&](auto e) {
            constexpr Elem E = decltype(e)::value;
            if constexpr (E != Elem::F32)
                with_row_bytes<E>(d.M, [&](auto rowb) {
                    with_int<2, 1>(s.qpg, [&](auto q) { msda_fwd8v_kernel<E, q, SlotSrc, rowb><<<grid, s.threads, smem, st>>>(a); });
                });
        });
        return check_launch(DEVIS_MSDA_KERNEL_FWD_GROUPED);
    }
    if (compact) {
        LaunchShape s = pick_shape(d.Lq, kShapeFwdF32, 4);
        if (s.threads > DEVIS_FWDV_MAXT) s.threads = DEVIS_FWDV_MAXT;
        smem += (size_t)(s.threads / 32) * Tap16x8::kBytesPerWarp;
        if ((rc = lane_group_grid(d, s.threads / 8, s.qpg, grid))) return rc;
        with_row_bytes<Elem::F32>(d.M, [&](auto rowb) {
            with_int<4, 2, 1>(s.qpg, [&](auto q) { msda_fwdv_kernel<Elem::F32, q, SlotSrc, rowb><<<grid, s.threads, smem, st>>>(a); });
        });
        return check_launch(DEVIS_MSDA_KERNEL_FWD_GROUPED);
    }
    if (lpg) {
        const LaunchShape s = pick_shape(d.Lq, is_16bit(dtype) ? kShapeFwdBf16 : kShapeFwdF32, 4);
        smem += exchange_bytes(lpg, s.threads);
        if ((rc = lane_group_grid(d, s.threads / lpg, s.qpg, grid))) return rc;
        with_elem(dtype, [&](auto e) {
            with_int<8, 4>(lpg, [&](auto l) {
                with_int<4, 2, 1>(s.qpg, [&](auto q) {
                    msda_fwd_kernel<decltype(e)::value, l, q, SlotSrc><<<grid, s.threads, smem, st>>>(a);
                });
            });
        });
        return check_launch(DEVIS_MSDA_KERNEL_FWD_GROUPED);
    }
    if ((rc = generic_grid(d, grid))) return rc;
    with_scalar(dtype, [&](auto t) {
        msda_fwd_generic_kernel<typename decltype(t)::type, SlotSrc><<<grid, kGenericThreads, smem, st>>>(a);
    });
    return check_launch(DEVIS_MSDA_KERNEL_FWD_GENERIC);
}

// ---- backward set-up shared by the unfused and fused ops ---------------------------------------------------------

// deterministic-mode workspace: [int64 accumulators: outer*S*M*D][2 x u32 max slots, padded to 16 B]
size_t det_workspace_bytes(long long outer, long long S, long long M, long long D)
{
    return (size_t)(outer * S * M * D) * sizeof(long long) + 16;
}

// bytes per grad_value element: float (also for 16-bit value), double for fp64, bf16 when accumulated in bf16
size_t grad_value_elem_size(int dtype, bool half_acc) { return dtype == DEVIS_MSDA_F64 ? 8 : half_acc ? 2 : 4; }

// the reference's at::zeros_like(value), ms_deform_attn_cuda.cu:121
int zero_fill(void *p, size_t bytes, cudaStream_t st)
{
    if (!bytes) return DEVIS_MSDA_OK;
    const cudaError_t e = cudaMemsetAsync(p, 0, bytes, st);
    return e == cudaSuccess ? DEVIS_MSDA_OK : cuda_fail(e);
}

// Deterministic mode, before the backward kernel: zero-fills the workspace, points det at its accumulators and slots,
// and stores the two factors of the fixed-point bound: max|grad_out| in slot 0, max|attention weight| in slot 1 -- over
// the n_seg segments' weights, or 1 when seg is null (the fused kernels' weights are softmax outputs).
int det_begin(DetScale &det, void *workspace, size_t workspace_bytes, int dtype, const OpDims &d, const void *grad_out,
              const Segment *seg, int n_seg, cudaStream_t st)
{
    const size_t need = det_workspace_bytes(d.outer, d.S, d.M, d.D);
    if (!workspace || workspace_bytes < need) return DEVIS_MSDA_ERR_WORKSPACE;
    const cudaError_t e = cudaMemsetAsync(workspace, 0, need, st);
    if (e != cudaSuccess) return cuda_fail(e);
    const size_t n_value = (size_t)d.outer * d.S * d.M * d.D;
    unsigned *slots = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(workspace) + n_value * sizeof(long long));
    det.acc = reinterpret_cast<long long *>(workspace);
    det.max_bits = slots;
    if (d.outer == 0 || d.Lq == 0) return DEVIS_MSDA_OK;
    const size_t n_go = (size_t)d.outer * d.Lq * d.M * d.D;
    const int blocks = devis_capi_helper_blocks();
    with_elem(dtype, [&](auto el) { absmax_kernel<decltype(el)::value><<<blocks, 256, 0, st>>>(grad_out, n_go, slots); });
    int rc = check_launch(DEVIS_MSDA_KERNEL_AUX);
    if (rc) return rc;
    if (!seg) {
        set_word_kernel<<<1, 1, 0, st>>>(slots + 1, 0x3f800000u);
        return check_launch(DEVIS_MSDA_KERNEL_AUX);
    }
    for (int sg = 0; sg < n_seg; ++sg) {
        const size_t n_aw = (size_t)d.outer * d.Lq * d.M * seg[sg].n_slots * seg[sg].P;
        absmax_kernel<Elem::F32><<<blocks, 256, 0, st>>>(seg[sg].aw, n_aw, slots + 1);
        if ((rc = check_launch(DEVIS_MSDA_KERNEL_AUX))) return rc;
    }
    return DEVIS_MSDA_OK;
}

// Deterministic mode, after the backward kernel: the fixed-point accumulators, in the channel order of lane groups of
// lpg lanes (0: channel order), into the float grad_value
int det_finish(const DetScale &det, void *grad_value, size_t n_value, int lpg, cudaStream_t st)
{
    if (n_value == 0) return DEVIS_MSDA_OK;
    det_finalize_kernel<<<devis_capi_helper_blocks(), 256, 0, st>>>(det.acc, reinterpret_cast<float *>(grad_value),
                                                                   n_value, det.max_bits, lpg);
    return check_launch(DEVIS_MSDA_KERNEL_AUX);
}

// sorted deterministic whole-clip backward (msda_bwd_sort.cuh), defined below
bool sort_applicable(const BwdArgs<ClipTable> &a, int dtype, unsigned flags);
int launch_backward_sort(const BwdArgs<ClipTable> &a, int dtype, cudaStream_t st);
inline bool sort_applicable(const BwdArgs<DeviceLevels> &, int, unsigned) { return false; }
inline int launch_backward_sort(const BwdArgs<DeviceLevels> &, int, cudaStream_t) { return DEVIS_MSDA_ERR_UNSUPPORTED; }

template <class SlotSrc>
int launch_backward(BwdArgs<SlotSrc> a, int dtype, unsigned flags, void *workspace, size_t workspace_bytes,
                    cudaStream_t st)
{
    const OpDims &d = a.d;
    const bool det = (flags & DEVIS_MSDA_FLAG_DETERMINISTIC) && a.grad_value != nullptr;
    // bf16 grad_value accumulated with packed bf16 reductions: bf16 value, grouped-lane kernels, default mode only
    const bool half_acc = (flags & DEVIS_MSDA_FLAG_BF16_GRAD_VALUE) && a.grad_value != nullptr;
    if (half_acc && (dtype != DEVIS_MSDA_BF16 || det || lanes_per_group(dtype, d) == 0)) return DEVIS_MSDA_ERR_UNSUPPORTED;
    const size_t n_value = (size_t)d.outer * d.S * d.M * d.D;
    void *const final_grad_value = a.grad_value;
    int rc;
    if (det) {
        if (dtype == DEVIS_MSDA_F64) return DEVIS_MSDA_ERR_UNSUPPORTED;
        if ((rc = det_begin(a.det, workspace, workspace_bytes, dtype, d, a.grad_out, a.seg, a.n_seg, st))) return rc;
        a.grad_value = nullptr;  // the float reductions are replaced by the fixed-point ones
    }
    if (a.grad_value && (rc = zero_fill(a.grad_value, n_value * grad_value_elem_size(dtype, half_acc), st))) return rc;
    const int lpg = lanes_per_group(dtype, d);
    auto finalize = [&]() { return det ? det_finish(a.det, final_grad_value, n_value, lpg, st) : DEVIS_MSDA_OK; };
    if (d.outer == 0 || d.Lq == 0) return finalize();
    size_t smem = (size_t)a.n_slots_total * sizeof(int4);
    dim3 grid;
    if (lpg && det && sort_applicable(a, dtype, flags)) {
        // deterministic mode, encoder form: sorted pre-aggregation in 64-bit fixed point (bit-identical to the direct
        // deterministic scatter, ~4x faster: 5x fewer 64-bit reductions leave the SM)
        rc = launch_backward_sort(a, dtype, st);
        return rc ? rc : finalize();
    }
    if (lpg) {
        const LaunchShape s = pick_shape(d.Lq, kShapeBwd, half_acc ? 1 : 2);
        smem += exchange_bytes(lpg, s.threads);
        if ((rc = lane_group_grid(d, s.threads / lpg, s.qpg, grid))) return rc;
        with_elem(dtype, [&](auto e) {
            constexpr Elem E = decltype(e)::value;
            with_int<8, 4>(lpg, [&](auto l) {
                if (half_acc) {
                    if constexpr (E == Elem::BF16) msda_bwd_kernel<E, l, 1, SlotSrc, true><<<grid, s.threads, smem, st>>>(a);
                } else {
                    with_int<2, 1>(s.qpg, [&](auto q) { msda_bwd_kernel<E, l, q, SlotSrc><<<grid, s.threads, smem, st>>>(a); });
                }
            });
        });
        rc = check_launch(DEVIS_MSDA_KERNEL_BWD_GROUPED);
        return rc ? rc : finalize();
    }
    if ((rc = generic_grid(d, grid))) return rc;
    with_scalar(dtype, [&](auto t) {
        msda_bwd_generic_kernel<typename decltype(t)::type, SlotSrc><<<grid, kGenericThreads, smem, st>>>(a);
    });
    rc = check_launch(DEVIS_MSDA_KERNEL_BWD_GENERIC);
    return rc ? rc : finalize();
}

// ---- sorted deterministic whole-clip backward (msda_bwd_sort.cuh) ------------------------------------------------
// Serves the deterministic mode of the encoder form: one query per pyramid pixel (the caller says so by passing a
// query_order), D = 32, fp32 / bf16 / fp16 value, levels stored back to back, an even number of levels, 4 points per slot.
// ~4x faster than the direct 64-bit scatter and bit-identical to it.  (The float variant of the same scheme lost to the
// direct float scatter -- data-pipe bound, DESIGN.md section 7 -- and is no longer built; benchmarks/experimental keeps
// the round-1 windowed kernel for the record.)  Developer keys: kKeyDirectScatter, kKeySortMargin, kKeySortMinLevel.
bool sort_applicable(const BwdArgs<ClipTable> &a, int dtype, unsigned flags)
{
    if (g_tuning[kKeyDirectScatter].load() == 1) return false;
    if (!a.det.acc || !a.q_perm || (flags & DEVIS_MSDA_FLAG_BF16_GRAD_VALUE)) return false;
    if (lanes_per_group(dtype, a.d) != 8 || a.d.Lq != a.d.S || a.d.outer == 0) return false;
    const ClipTable &tb = a.src;
    if (tb.L % 2 != 0) return false;
    int next = 0;
    for (int l = 0; l < tb.L; ++l) {
        if (tb.lsi[l] != next || tb.H[l] * (long long)tb.W[l] > 65536) return false;
        next += tb.H[l] * tb.W[l];
    }
    if (next != a.d.S) return false;
    for (int sg = 0; sg < a.n_seg; ++sg)
        if (a.seg[sg].P != 4 || a.seg[sg].n_slots % tb.L != 0) return false;
    if (sort_smem_bytes(a.n_slots_total, (tb.L / 2) * kSortMaxKeys) > 200 * 1024) return false;
    return true;
}

// the caller (launch_backward) has set up a.det and zero-filled the accumulators, and runs the finalize pass
int launch_backward_sort(const BwdArgs<ClipTable> &a, int dtype, cudaStream_t st)
{
    const OpDims &d = a.d;
    SortArgs w{};
    w.b = a;
    int tiles = 0;
    for (int l = 0; l < a.src.L; ++l) {
        w.tiles_x[l] = (a.src.W[l] + kSortTile - 1) / kSortTile;
        w.tile_start[l] = tiles;
        tiles += w.tiles_x[l] * ((a.src.H[l] + kSortTile - 1) / kSortTile);
    }
    w.n_tiles = tiles;
    const int margin = g_tuning[kKeySortMargin].load(), min_level = g_tuning[kKeySortMinLevel].load();
    w.margin = margin > 0 ? margin : 6;
    w.min_level = min_level > 0 ? min_level - 1 : 0;
    w.lut_entries = (a.src.L / 2) * kSortMaxKeys;
    const size_t smem = sort_smem_bytes(a.n_slots_total, w.lut_entries);
    if ((long long)tiles * d.M > 0x7fffffffLL) return DEVIS_MSDA_ERR_TOO_LARGE;
    const dim3 grid((unsigned)(tiles * d.M), (unsigned)d.outer);
    return with_elem(dtype, [&](auto e) {
        constexpr Elem E = decltype(e)::value;
        const cudaError_t err = cudaFuncSetAttribute(msda_bwds_kernel<E, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return cuda_fail(err);
        msda_bwds_kernel<E, true><<<grid, kSortThreads, smem, st>>>(w);
        return check_launch(DEVIS_MSDA_KERNEL_BWD_SORTED);
    });
}

int check_common(int outer, int S, int M, int D, int L, int Lq, int dtype)
{
    if (dtype != DEVIS_MSDA_F32 && dtype != DEVIS_MSDA_F64 && !is_16bit(dtype)) return DEVIS_MSDA_ERR_BAD_DTYPE;
    if (outer < 0 || S < 0 || M <= 0 || D <= 0 || L <= 0 || Lq < 0) return DEVIS_MSDA_ERR_BAD_SHAPE;
    if (outer > 65535) return DEVIS_MSDA_ERR_TOO_LARGE;
    // value rows are indexed with 31-bit integers in every kernel
    if ((long long)outer * S >= (1LL << 31)) return DEVIS_MSDA_ERR_TOO_LARGE;
    return DEVIS_MSDA_OK;
}

int fill_clip_table(ClipTable &tb, const int64_t *shapes, const int64_t *lsi, const int32_t *frames, int T, int S,
                    int L, int Wt)
{
    if (L > kMaxLevels || (long long)T * Wt > kMaxFrameTable || T > 255) return DEVIS_MSDA_ERR_TOO_LARGE;
    std::memset(&tb, 0, sizeof(tb));
    tb.L = L;
    tb.Wt = Wt;
    for (int l = 0; l < L; ++l) {
        const int64_t H = shapes[2 * l], W = shapes[2 * l + 1], st = lsi[l];
        if (H <= 0 || W <= 0 || st < 0 || st + H * W > S) return DEVIS_MSDA_ERR_BAD_SHAPE;
        tb.H[l] = (int)H;
        tb.W[l] = (int)W;
        tb.lsi[l] = (int)st;
    }
    for (int i = 0; i < T * Wt; ++i) {
        if (frames[i] < 0 || frames[i] >= T) return DEVIS_MSDA_ERR_BAD_FRAME_TABLE;
        tb.frame[i] = (uint8_t)frames[i];
    }
    return DEVIS_MSDA_OK;
}

// every device tensor of a non-empty call is given: value, output or grad_output, and the first n_seg segments'
// locations and weights (and their gradients in the backward)
bool seg_given(const Segment &s, bool grads) { return s.loc && s.aw && (!grads || (s.grad_loc && s.grad_aw)); }
template <class SlotSrc>
bool tensors_given(const FwdArgs<SlotSrc> &a, int n_seg)
{
    return a.value && a.out && seg_given(a.seg[0], false) && (n_seg < 2 || seg_given(a.seg[1], false));
}
template <class SlotSrc>
bool tensors_given(const BwdArgs<SlotSrc> &a, int n_seg)
{
    return a.value && a.grad_out && seg_given(a.seg[0], true) && (n_seg < 2 || seg_given(a.seg[1], true));
}

// Drop-in op (devis_msda_forward / backward): the caller has put the device pointers and P into a (seg[0]);
// grad_value_missing: the backward wants grad_value and got none.  Validates in the reference's order and fills the rest.
template <class Args>
int fill_level_args(Args &a, bool grad_value_missing, const int64_t *shapes, const int64_t *lsi, int batch, int S,
                    int M, int D, int L, int Lq, int im2col_step, int dtype)
{
    const int rc = check_common(batch, S, M, D, L, Lq, dtype);
    if (rc) return rc;
    if (a.seg[0].P <= 0 || im2col_step <= 0 || L > kMaxSlots) return DEVIS_MSDA_ERR_BAD_SHAPE;
    if (batch > 0 && batch % (batch < im2col_step ? batch : im2col_step) != 0) return DEVIS_MSDA_ERR_BATCH_STEP;
    const bool empty = batch == 0 || Lq == 0;
    if ((!empty && (!shapes || !lsi || !tensors_given(a, 1))) || grad_value_missing) return DEVIS_MSDA_ERR_NULL_POINTER;
    a.seg[0].n_slots = L;
    a.n_seg = 1;
    a.n_slots_total = L;
    a.src = DeviceLevels{shapes, lsi};
    a.d = OpDims{batch, S, M, D, Lq};
    a.q_perm = nullptr;
    return DEVIS_MSDA_OK;
}

// Whole-clip op (devis_tmsda_forward / backward): the caller has put the device pointers and the points per slot of
// the current (seg[0]) and temporal (seg[1]) segments into a; as fill_level_args otherwise.
template <class Args>
int fill_clip_args(Args &a, bool grad_value_missing, const int64_t *shapes, const int64_t *lsi, const int32_t *frames,
                   const int32_t *order, int T, int S, int M, int D, int L, int Lq, int Wt, int dtype)
{
    int rc = check_common(T, S, M, D, L, Lq, dtype);
    if (rc) return rc;
    if (a.seg[0].P <= 0 || a.seg[1].P < 0 || Wt < 0) return DEVIS_MSDA_ERR_BAD_SHAPE;
    const bool temporal = Wt > 0 && a.seg[1].P > 0;
    if (!shapes || !lsi || (temporal && !frames)) return DEVIS_MSDA_ERR_NULL_POINTER;
    const bool empty = T == 0 || Lq == 0;
    if ((!empty && !tensors_given(a, temporal ? 2 : 1)) || grad_value_missing) return DEVIS_MSDA_ERR_NULL_POINTER;
    rc = fill_clip_table(a.src, shapes, lsi, frames, T, S, L, temporal ? Wt : 0);
    if (rc) return rc;
    a.seg[0].n_slots = L;
    if (temporal) a.seg[1].n_slots = Wt * L;
    else a.seg[1] = Segment{};
    a.n_seg = temporal ? 2 : 1;
    a.n_slots_total = L + a.seg[1].n_slots;
    if (a.n_slots_total > kMaxSlots) return DEVIS_MSDA_ERR_TOO_LARGE;
    a.d = OpDims{T, S, M, D, Lq};
    a.q_perm = order;
    return DEVIS_MSDA_OK;
}

}  // namespace

extern "C" {

int devis_msda_abi_version(void) { return DEVIS_MSDA_ABI_VERSION; }

const char *devis_msda_error_string(int code)
{
    switch (code) {
        case DEVIS_MSDA_OK: return "ok";
        case DEVIS_MSDA_ERR_NULL_POINTER: return "null pointer for a non-empty tensor";
        case DEVIS_MSDA_ERR_BAD_SHAPE: return "invalid dimension";
        case DEVIS_MSDA_ERR_BAD_DTYPE: return "unsupported dtype code";
        case DEVIS_MSDA_ERR_BATCH_STEP: return "batch must be divisible by min(batch, im2col_step)";
        case DEVIS_MSDA_ERR_TOO_LARGE: return "tensor too large for the kernels' indexing";
        case DEVIS_MSDA_ERR_WORKSPACE: return "workspace missing or too small";
        case DEVIS_MSDA_ERR_CUDA: return "CUDA runtime error (see devis_msda_last_cuda_error)";
        case DEVIS_MSDA_ERR_UNSUPPORTED: return "no kernel for this request in this build";
        case DEVIS_MSDA_ERR_BAD_FRAME_TABLE: return "frame table entry outside [0, num_frames)";
        default: return "unknown error code";
    }
}

int devis_msda_last_cuda_error(void) { return t_last_cuda_error; }
uint64_t devis_msda_launch_count(void) { return g_launches.load(); }

uint64_t devis_msda_kernel_launches(int family)
{
    return (family >= 0 && family < DEVIS_MSDA_KERNEL_FAMILIES) ? g_family_launches[family].load() : 0;
}

int devis_msda_set_tuning(int key, int value)
{
    if (key < 0 || key >= 16) return DEVIS_MSDA_ERR_BAD_SHAPE;
    if (!tuning_enabled()) return DEVIS_MSDA_ERR_UNSUPPORTED;
    g_tuning_store[key].store(value);
    return DEVIS_MSDA_OK;
}

int devis_msda_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                       const void *sampling_loc, const void *attn_weight, void *output, int batch,
                       int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                       int num_point, int im2col_step, int dtype, void *stream)
{
    FwdArgs<DeviceLevels> a{};
    a.value = value;
    a.out = output;
    a.seg[0] = Segment{sampling_loc, attn_weight, nullptr, nullptr, 0, num_point};
    const int rc = fill_level_args(a, false, spatial_shapes, level_start_index, batch, spatial_size, num_heads, channels,
                                   num_levels, num_query, im2col_step, dtype);
    return rc ? rc : launch_forward(a, dtype, (cudaStream_t)stream);
}

size_t devis_msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels, int, int, int,
                                           int dtype, unsigned flags)
{
    if (!(flags & DEVIS_MSDA_FLAG_DETERMINISTIC) || (flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE) || dtype == DEVIS_MSDA_F64)
        return 0;
    return det_workspace_bytes(batch, spatial_size, num_heads, channels);
}

int devis_msda_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                        const void *sampling_loc, const void *attn_weight, const void *grad_output,
                        void *grad_value, void *grad_sampling_loc, void *grad_attn_weight, int batch,
                        int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                        int num_point, int im2col_step, int dtype, unsigned flags, void *workspace,
                        size_t workspace_bytes, void *stream)
{
    const bool want_gv = !(flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE);
    BwdArgs<DeviceLevels> a{};
    a.value = value;
    a.grad_out = grad_output;
    a.grad_value = want_gv ? grad_value : nullptr;
    a.seg[0] = Segment{sampling_loc, attn_weight, grad_sampling_loc, grad_attn_weight, 0, num_point};
    const int rc = fill_level_args(a, want_gv && !grad_value && (size_t)batch * spatial_size > 0, spatial_shapes,
                                   level_start_index, batch, spatial_size, num_heads, channels, num_levels, num_query,
                                   im2col_step, dtype);
    return rc ? rc : launch_backward(a, dtype, flags, workspace, workspace_bytes, (cudaStream_t)stream);
}

int devis_tmsda_forward(const void *value, const int64_t *spatial_shapes_host,
                        const int64_t *level_start_index_host, const int32_t *frame_table_host,
                        const void *loc_curr, const void *aw_curr, const void *loc_temporal,
                        const void *aw_temporal, void *output, const int32_t *query_order, int num_frames,
                        int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                        int n_curr_points, int n_temporal_points, int t_window, int dtype, void *stream)
{
    FwdArgs<ClipTable> a{};
    a.value = value;
    a.out = output;
    a.seg[0] = Segment{loc_curr, aw_curr, nullptr, nullptr, 0, n_curr_points};
    a.seg[1] = Segment{loc_temporal, aw_temporal, nullptr, nullptr, 0, n_temporal_points};
    const int rc = fill_clip_args(a, false, spatial_shapes_host, level_start_index_host, frame_table_host, query_order,
                                  num_frames, spatial_size, num_heads, channels, num_levels, num_query, t_window, dtype);
    return rc ? rc : launch_forward(a, dtype, (cudaStream_t)stream);
}

size_t devis_tmsda_backward_workspace_bytes(int num_frames, int spatial_size, int num_heads, int channels, int, int,
                                            int, int, int, int dtype, unsigned flags)
{
    if ((flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE) || dtype == DEVIS_MSDA_F64) return 0;
    if (!(flags & DEVIS_MSDA_FLAG_DETERMINISTIC)) return 0;
    return det_workspace_bytes(num_frames, spatial_size, num_heads, channels);
}

int devis_tmsda_backward(const void *value, const int64_t *spatial_shapes_host,
                         const int64_t *level_start_index_host, const int32_t *frame_table_host,
                         const void *loc_curr, const void *aw_curr, const void *loc_temporal,
                         const void *aw_temporal, const void *grad_output, void *grad_value,
                         void *grad_loc_curr, void *grad_aw_curr, void *grad_loc_temporal,
                         void *grad_aw_temporal, const int32_t *query_order, int num_frames, int spatial_size,
                         int num_heads, int channels, int num_levels, int num_query, int n_curr_points,
                         int n_temporal_points, int t_window, int dtype, unsigned flags, void *workspace,
                         size_t workspace_bytes, void *stream)
{
    const bool want_gv = !(flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE);
    BwdArgs<ClipTable> a{};
    a.value = value;
    a.grad_out = grad_output;
    a.grad_value = want_gv ? grad_value : nullptr;
    a.seg[0] = Segment{loc_curr, aw_curr, grad_loc_curr, grad_aw_curr, 0, n_curr_points};
    a.seg[1] = Segment{loc_temporal, aw_temporal, grad_loc_temporal, grad_aw_temporal, 0, n_temporal_points};
    const int rc = fill_clip_args(a, want_gv && !grad_value && (size_t)num_frames * spatial_size > 0,
                                  spatial_shapes_host, level_start_index_host, frame_table_host, query_order,
                                  num_frames, spatial_size, num_heads, channels, num_levels, num_query, t_window, dtype);
    return rc ? rc : launch_backward(a, dtype, flags, workspace, workspace_bytes, (cudaStream_t)stream);
}

static int fill_fused(FusedArgs &a, const void *value, const int64_t *shapes, const int64_t *lsi, const int32_t *frames,
                      const void *ref, const void *off_c, const void *logit_c, const void *off_t, const void *logit_t,
                      const int32_t *order, int T, int S, int M, int D, int L, int Lq, int Pc, int Pt, int Wt, int ref_dim,
                      int tref_mode, int dtype)
{
    int rc = check_common(T, S, M, D, L, Lq, dtype);
    if (rc) return rc;
    if (Pc <= 0 || Pt < 0 || Wt < 0 || (ref_dim != 2 && ref_dim != 4) || tref_mode < 0 || tref_mode > 2)
        return DEVIS_MSDA_ERR_BAD_SHAPE;
    if (dtype == DEVIS_MSDA_F64 || D != 32 || Pc % 4 != 0 || (Wt > 0 && Pt > 0 && Pt % 4 != 0))
        return DEVIS_MSDA_ERR_UNSUPPORTED;
    if ((unsigned long long)T * S * M * D * elem_size(dtype) >= (1ull << 32)) return DEVIS_MSDA_ERR_UNSUPPORTED;
    if ((unsigned long long)T * Lq * L >= (1ull << 31)) return DEVIS_MSDA_ERR_TOO_LARGE;   // ref rows are 31-bit
    const bool temporal = Wt > 0 && Pt > 0;
    if (!shapes || !lsi || (temporal && !frames)) return DEVIS_MSDA_ERR_NULL_POINTER;
    const bool empty = T == 0 || Lq == 0;
    if (!empty && (!value || !ref || !off_c || !logit_c || (temporal && (!off_t || !logit_t))))
        return DEVIS_MSDA_ERR_NULL_POINTER;
    rc = fill_clip_table(a.src, shapes, lsi, frames, T, S, L, temporal ? Wt : 0);
    if (rc) return rc;
    a.value = value;
    a.ref = reinterpret_cast<const float *>(ref);
    a.ref_dim = ref_dim;
    a.tref_mode = tref_mode;
    a.off[0] = reinterpret_cast<const float *>(off_c);
    a.logit[0] = reinterpret_cast<const float *>(logit_c);
    a.off[1] = reinterpret_cast<const float *>(off_t);
    a.logit[1] = reinterpret_cast<const float *>(logit_t);
    a.n_slots[0] = L;
    a.P[0] = Pc;
    a.n_slots[1] = temporal ? Wt * L : 0;
    a.P[1] = temporal ? Pt : 1;
    a.inv_p[0] = 1.f / (float)Pc;
    a.inv_p[1] = temporal ? 1.f / (float)Pt : 1.f;
    a.n_seg = temporal ? 2 : 1;
    if (a.n_slots[0] + a.n_slots[1] > kMaxSlots) return DEVIS_MSDA_ERR_TOO_LARGE;
    a.d = OpDims{T, S, M, D, Lq};
    a.q_perm = order;
    return DEVIS_MSDA_OK;
}

int devis_tmsda_fused_forward(const void *value, const int64_t *spatial_shapes_host,
                              const int64_t *level_start_index_host, const int32_t *frame_table_host,
                              const void *ref, const void *off_curr, const void *logit_curr,
                              const void *off_temporal, const void *logit_temporal, void *output,
                              void *loc_curr_out, void *aw_curr_out, void *loc_temporal_out, void *aw_temporal_out,
                              const int32_t *query_order, int num_frames, int spatial_size, int num_heads,
                              int channels, int num_levels, int num_query, int n_curr_points,
                              int n_temporal_points, int t_window, int ref_dim, int temporal_ref_mode, int dtype,
                              void *stream)
{
    FusedArgs a{};
    int rc = fill_fused(a, value, spatial_shapes_host, level_start_index_host, frame_table_host, ref, off_curr,
                        logit_curr, off_temporal, logit_temporal, query_order, num_frames, spatial_size, num_heads,
                        channels, num_levels, num_query, n_curr_points, n_temporal_points, t_window, ref_dim,
                        temporal_ref_mode, dtype);
    if (rc) return rc;
    if (num_frames == 0 || num_query == 0) return DEVIS_MSDA_OK;
    if (!output) return DEVIS_MSDA_ERR_NULL_POINTER;
    a.out = output;
    a.loc_out[0] = reinterpret_cast<float *>(loc_curr_out);
    a.aw_out[0] = reinterpret_cast<float *>(aw_curr_out);
    a.loc_out[1] = a.n_seg > 1 ? reinterpret_cast<float *>(loc_temporal_out) : nullptr;
    a.aw_out[1] = a.n_seg > 1 ? reinterpret_cast<float *>(aw_temporal_out) : nullptr;
    // dead corners skipped, virtual top-left addressing: signed 32-bit offsets, so value must stay below 2 GiB (the Python
    // side then uses the unfused op)
    if ((unsigned long long)num_frames * spatial_size * num_heads * channels * elem_size(dtype) >= (1ull << 31))
        return DEVIS_MSDA_ERR_UNSUPPORTED;
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t slot_smem = (size_t)(a.n_slots[0] + a.n_slots[1]) * sizeof(int4);
    dim3 grid;
    // the general (decoder) form: boxes, per-level / instance-aware temporal reference points, by-products
    const bool general = ref_dim == 4 || (a.n_seg > 1 && temporal_ref_mode != 0) || loc_curr_out || aw_curr_out ||
                         a.loc_out[1] || a.aw_out[1];
    if (!general && is_16bit(dtype)) {
        // bf16 / fp16 value: four lanes x 8 channels per (query, head) like msda_fwd8v_kernel
        const LaunchShape s = pick_shape(num_query, kShapeFusedFwd16, 1);
        if ((rc = lane_group_grid(a.d, s.threads / 4, s.qpg, grid))) return rc;
        const size_t smem = slot_smem + (size_t)(s.threads / 32) * Tap16::kBytesPerWarp;
        with_elem(dtype, [&](auto e) {
            constexpr Elem E = decltype(e)::value;
            if constexpr (E != Elem::F32)
                with_row_bytes<E>(num_heads, [&](auto rowb) { tmsda_fused_fwd8_kernel<E, rowb><<<grid, s.threads, smem, st>>>(a); });
        });
        return check_launch(DEVIS_MSDA_KERNEL_FUSED_FWD);
    }
    // eight lanes x 4 channels; the fp32 encoder form takes two queries per lane group at encoder sizes, like
    // msda_fwdv_kernel (a key-1 value other than 1 or 2 leaves that choice to the heuristic)
    const LaunchShape s = general ? pick_shape(num_query, kShapeFwdF32, 1) : pick_shape(num_query, kShapeFwdF32, 2, false);
    if ((rc = lane_group_grid(a.d, s.threads / 8, s.qpg, grid))) return rc;
    const size_t smem = slot_smem + exchange_bytes(8, s.threads);
    with_elem(dtype, [&](auto e) {
        constexpr Elem E = decltype(e)::value;
        with_row_bytes<E>(num_heads, [&](auto rowb) {
            if (general) {
                tmsda_fused_fwd_kernel<E, 1, true, rowb><<<grid, s.threads, smem, st>>>(a);
            } else if constexpr (E == Elem::F32) {
                with_int<2, 1>(s.qpg, [&](auto q) { tmsda_fused_fwd_kernel<E, q, false, rowb><<<grid, s.threads, smem, st>>>(a); });
            }
        });
    });
    return check_launch(DEVIS_MSDA_KERNEL_FUSED_FWD);
}

size_t devis_tmsda_fused_backward_workspace_bytes(int num_frames, int spatial_size, int num_heads, int channels, unsigned flags)
{
    if (!(flags & DEVIS_MSDA_FLAG_DETERMINISTIC) || (flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE)) return 0;
    if (num_frames < 0 || spatial_size < 0 || num_heads < 0 || channels < 0) return 0;
    return det_workspace_bytes(num_frames, spatial_size, num_heads, channels);
}

int devis_tmsda_fused_backward(const void *value, const int64_t *spatial_shapes_host,
                               const int64_t *level_start_index_host, const int32_t *frame_table_host,
                               const void *ref, const void *off_curr, const void *logit_curr,
                               const void *off_temporal, const void *logit_temporal, const void *grad_output,
                               void *grad_value, void *grad_off_curr, void *grad_logit_curr,
                               void *grad_off_temporal, void *grad_logit_temporal, void *grad_ref,
                               const int32_t *query_order, int num_frames, int spatial_size, int num_heads,
                               int channels, int num_levels, int num_query, int n_curr_points,
                               int n_temporal_points, int t_window, int ref_dim, int temporal_ref_mode, int dtype,
                               unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    FusedArgs a{};
    int rc = fill_fused(a, value, spatial_shapes_host, level_start_index_host, frame_table_host, ref, off_curr,
                        logit_curr, off_temporal, logit_temporal, query_order, num_frames, spatial_size, num_heads,
                        channels, num_levels, num_query, n_curr_points, n_temporal_points, t_window, ref_dim,
                        temporal_ref_mode, dtype);
    if (rc) return rc;
    const bool want_gv = !(flags & DEVIS_MSDA_FLAG_NO_GRAD_VALUE);
    const bool half_acc = want_gv && (flags & DEVIS_MSDA_FLAG_BF16_GRAD_VALUE);
    if (half_acc && dtype != DEVIS_MSDA_BF16) return DEVIS_MSDA_ERR_UNSUPPORTED;
    // deterministic mode: grad_value through 64-bit fixed point (workspace); d/d(ref) is a float-atomic sum over
    // queries' heads and taps and has no fixed-point form here
    const bool det = (flags & DEVIS_MSDA_FLAG_DETERMINISTIC) && want_gv;
    if ((flags & DEVIS_MSDA_FLAG_DETERMINISTIC) && (grad_ref || half_acc)) return DEVIS_MSDA_ERR_UNSUPPORTED;
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t n_value = (size_t)num_frames * spatial_size * num_heads * channels;
    if (det && (rc = det_begin(a.det, workspace, workspace_bytes, dtype, a.d, grad_output, nullptr, 0, st))) return rc;
    if (want_gv) {
        const size_t bytes = n_value * grad_value_elem_size(dtype, half_acc);
        if (bytes && !grad_value) return DEVIS_MSDA_ERR_NULL_POINTER;
        if ((rc = zero_fill(grad_value, bytes, st))) return rc;
    }
    if (grad_ref && (rc = zero_fill(grad_ref, (size_t)num_frames * num_query * num_levels * ref_dim * sizeof(float), st)))
        return rc;
    if (num_frames == 0 || num_query == 0) return DEVIS_MSDA_OK;
    if (!grad_output || !grad_off_curr || !grad_logit_curr || (a.n_seg > 1 && (!grad_off_temporal || !grad_logit_temporal)))
        return DEVIS_MSDA_ERR_NULL_POINTER;
    a.grad_out = grad_output;
    a.grad_value = want_gv ? grad_value : nullptr;
    a.grad_off[0] = reinterpret_cast<float *>(grad_off_curr);
    a.grad_logit[0] = reinterpret_cast<float *>(grad_logit_curr);
    a.grad_off[1] = reinterpret_cast<float *>(grad_off_temporal);
    a.grad_logit[1] = reinterpret_cast<float *>(grad_logit_temporal);
    a.grad_ref = reinterpret_cast<float *>(grad_ref);
    const LaunchShape s = pick_shape(num_query, kShapeBwd, 1);
    dim3 grid;
    if ((rc = lane_group_grid(a.d, s.threads / 8, s.qpg, grid))) return rc;
    size_t smem = (size_t)(a.n_slots[0] + a.n_slots[1]) * sizeof(int4) + exchange_bytes(8, s.threads);
    {   // (weight, d/d weight) of every tap parked in shared memory until the row's softmax-backward sum is known
        int iters = 0;
        for (int sg = 0; sg < a.n_seg; ++sg) iters += (a.n_slots[sg] * a.P[sg] + 7) / 8;
        const size_t park = (size_t)iters * s.threads * sizeof(float2);
        if (smem + park <= 48 * 1024) {
            a.park_iters = iters;
            smem += park;
        }
    }
    const bool general = ref_dim == 4 || (a.n_seg > 1 && temporal_ref_mode != 0) || grad_ref;
    with_elem(dtype, [&](auto e) {
        constexpr Elem E = decltype(e)::value;
        auto launch = [&](auto gen) {
            if (det) {
                tmsda_fused_bwd_kernel<E, false, gen, true><<<grid, s.threads, smem, st>>>(a);
            } else if (half_acc) {
                if constexpr (E == Elem::BF16) tmsda_fused_bwd_kernel<E, true, gen><<<grid, s.threads, smem, st>>>(a);
            } else {
                tmsda_fused_bwd_kernel<E, false, gen><<<grid, s.threads, smem, st>>>(a);
            }
        };
        if (general) launch(std::true_type{});
        else launch(std::false_type{});
    });
    rc = check_launch(DEVIS_MSDA_KERNEL_FUSED_BWD);
    if (rc || !det) return rc;
    return det_finish(a.det, grad_value, n_value, 8, st);
}

}  // extern "C"
