"""Case table of the deformable-convolution kernel sweep (test_dcn_kernels_gpu.py), the seeded operands of a case, and
the host-side rules that map a case to the kernel instantiations and launch shapes it reaches (test_dcn_kernels_host.py
checks that the table reaches every instantiation).  Importable without a GPU.

The rules restate the dispatch of devis_b200/csrc/deform_conv_capi.cu (dispatch, fused_plan, the constant-bank chunking,
devis_dcn_weight_grad's run length, igemm_plan) and of devis_b200/deform_conv.py (which autograd Function serves a
call, how the backward is sliced into calls)."""
import math
from dataclasses import dataclass

import torch

SMALL_COUT = (1, 2, 4, 8, 16)
CONST_C = (16, 32, 40, 64, 72)             # dcn_fusedc_fwd_kernel<C, CT> instantiations
MAX_GRID_Z = 65535
CONST_FLOATS = 16384                       # kDcnConstFloats
CHUNK_BYTES = 256 << 20                    # deform_conv._COLS_CHUNK_BYTES == _DET_ACC_CHUNK_BYTES
IG_SMEM, IG_ATILE, IG_GEOM, IG_MAX_STAGES, IG_BK = 227 * 1024, 128 * 128, 2 * 128 * 32, 4, 32
B200_HELPER_BLOCKS = 148 * 8               # devis_capi_helper_blocks on a 148-SM B200


@dataclass(frozen=True)
class Case:
    name: str
    n: int
    cin: int
    cout: int
    h: int
    w: int
    kh: int = 3
    kw: int = 3
    stride: tuple = (1, 1)
    pad: tuple = (1, 1)
    dil: tuple = (1, 1)
    mask: bool = True
    bias: bool = True
    form: str = "auto"          # im2col | fused | igemm | auto (the library's own choice, every form enabled)
    train: bool = True
    dtype: str = "float32"
    og: int = 1
    tf32: bool = False          # igemm: single-pass TF32 forward instead of 3xTF32

    @property
    def ho(self):
        return (self.h + 2 * self.pad[0] - (self.dil[0] * (self.kh - 1) + 1)) // self.stride[0] + 1

    @property
    def wo(self):
        return (self.w + 2 * self.pad[1] - (self.dil[1] * (self.kw - 1) + 1)) // self.stride[1] + 1

    @property
    def k(self):
        return self.kh * self.kw


def _c(name, n, cin, cout, h, w, **kw):
    return Case(name, n, cin, cout, h, w, **kw)


ASYM = dict(kh=2, kw=3, stride=(2, 1), pad=(1, 2), dil=(1, 2))       # every geometry parameter unequal
ASYM2 = dict(kh=3, kw=2, stride=(1, 2), pad=(2, 0), dil=(2, 1))
BIG_N = 65535 + 4

# (name, Cin, Cout, H, W) of the mask head's deformable layers (benchmarks/dcn_bench.py)
LAYERS = [("lay1", 264, 264, 12, 20), ("lay2", 264, 128, 12, 20), ("lay3", 136, 64, 23, 40), ("lay4", 72, 32, 45, 80),
          ("lay5", 32, 16, 90, 160), ("out_lay", 16, 1, 90, 160)]
# instances per layer: lay5 and out_lay with enough to make the weight-gradient kernel take its longest pixel runs
LAYER_N = {"lay1": 6, "lay2": 6, "lay3": 6, "lay4": 6, "lay5": 17, "out_lay": 33}

CASES = [
    # ---- im2col / col2im (cuBLAS GEMMs): float <V, G> by the group's channel count, double <1, G> -------------------
    _c("i2c_f32_v4g4_asym", 3, 16, 5, 11, 13, form="im2col", **ASYM),
    _c("i2c_f32_v4g8_asym2_nomask", 2, 40, 7, 12, 9, form="im2col", mask=False, **ASYM2),
    _c("i2c_f32_v1g8_nobias", 3, 6, 3, 10, 12, form="im2col", bias=False, **ASYM),
    _c("i2c_f32_v1g32", 2, 33, 4, 9, 11, form="im2col", **ASYM2),
    _c("i2c_f64_v1g8_asym", 2, 6, 3, 10, 12, form="im2col", dtype="float64", **ASYM),
    _c("i2c_f64_v1g32_asym2", 2, 33, 4, 9, 11, form="im2col", dtype="float64", **ASYM2),
    _c("i2c_f64_c16", 2, 16, 5, 11, 13, form="im2col", dtype="float64", mask=False, bias=False),
    _c("i2c_f32_og2", 2, 16, 6, 10, 11, form="im2col", og=2, **ASYM),
    _c("i2c_f32_bign", BIG_N, 8, 3, 3, 2, kh=2, kw=1, pad=(0, 0), form="im2col"),
    _c("i2c_f64_bign", BIG_N, 6, 2, 3, 2, kh=2, kw=1, pad=(0, 0), form="im2col", dtype="float64"),
    # ---- lane-group fused forward + backward: COUT x G (G = 4: C/4 <= 4, G = 8 beyond), partial 8 x (32/G)*2 tiles ---
    _c("lane_o1_g4", 2, 12, 1, 11, 19, form="fused"),
    _c("lane_o2_g4_asym", 2, 12, 2, 13, 21, form="fused", **ASYM),
    _c("lane_o4_g4", 2, 12, 4, 9, 17, form="fused", mask=False),
    _c("lane_o8_g4_asym2", 2, 12, 8, 15, 20, form="fused", bias=False, **ASYM2),
    _c("lane_o16_g4", 2, 8, 16, 10, 18, form="fused"),
    _c("lane_o1_g8_asym", 2, 24, 1, 13, 11, form="fused", **ASYM),
    _c("lane_o2_g8", 2, 24, 2, 9, 10, form="fused", bias=False),
    _c("lane_o4_g8_asym2", 2, 24, 4, 17, 12, form="fused", **ASYM2),
    _c("lane_o8_g8", 2, 36, 8, 11, 13, form="fused", mask=False),
    _c("lane_o16_g8", 2, 24, 16, 10, 9, form="fused"),
    _c("lane_og2_o4_g4", 2, 16, 4, 10, 11, form="fused", og=2, **ASYM),
    _c("lane_fwd_infer_o4_g4", 2, 12, 4, 11, 19, form="fused", train=False, **ASYM2),
    # ---- weight-gradient kernel (C in {16, 32} x COUT); the lane-group kernels serve the data gradients ------------
    _c("wg_c16_o1", 2, 16, 1, 10, 12, form="fused", **ASYM2),
    _c("wg_c16_o2", 2, 16, 2, 11, 9, form="fused"),
    _c("wg_c16_o4_asym", 2, 16, 4, 12, 14, form="fused", **ASYM),
    _c("wg_c16_o8", 2, 16, 8, 9, 12, form="fused", bias=False),
    _c("wg_c32_o1", 2, 32, 1, 9, 10, form="fused", mask=False),
    _c("wg_c32_o2_asym2", 2, 32, 2, 11, 12, form="fused", **ASYM2),
    _c("wg_c32_o4", 2, 32, 4, 10, 9, form="fused"),
    _c("wg_c32_o8_asym", 2, 32, 8, 13, 11, form="fused", **ASYM),
    _c("wg_run16", 5, 32, 4, 90, 160, form="fused"),
    _c("wg_run32", 9, 32, 2, 90, 160, form="fused", mask=False),
    _c("wg_bign", BIG_N, 16, 2, 3, 2, kh=2, kw=1, pad=(0, 0), form="fused"),
    # ---- constant-bank forward: C x CT (Cout 16 -> CT 16 with the lane-group backward and the weight-gradient kernel;
    #      wider layers in inference), Cout = 48 (three tiles), 1 / 2 / 3 kernel-position chunks, partial tiles -------
    _c("cb_c16_ct16", 2, 16, 16, 11, 37, form="fused"),
    _c("cb_c32_ct16_asym", 2, 32, 16, 19, 45, form="fused", **ASYM),
    _c("cb_c40_ct16", 2, 40, 16, 9, 33, form="fused", train=False, mask=False),
    _c("cb_c64_ct16_asym2", 2, 64, 16, 17, 35, form="fused", train=False, **ASYM2),
    _c("cb_c72_ct16", 2, 72, 16, 10, 34, form="fused", train=False, bias=False),
    _c("cb_c16_ct32", 2, 16, 32, 9, 33, form="fused", train=False),
    _c("cb_c32_ct32_asym", 2, 32, 32, 11, 36, form="fused", train=False, **ASYM),
    _c("cb_c40_ct32", 2, 40, 64, 10, 34, form="fused", train=False),
    _c("cb_c64_ct32_2chunks", 2, 64, 32, 12, 40, form="fused", train=False),
    _c("cb_c72_ct32_1chunk", 2, 72, 32, 9, 35, kh=1, kw=3, pad=(0, 1), form="fused", train=False),
    _c("cb_c72_ct32_2chunks", 2, 72, 32, 11, 33, form="fused", train=False, mask=False),
    _c("cb_c72_ct32_3chunks", 2, 72, 32, 10, 38, kh=3, kw=5, pad=(1, 2), form="fused", train=False),
    _c("cb_c40_o48", 2, 40, 48, 9, 37, form="fused", train=False, **ASYM2),
    _c("cb_bign", BIG_N, 16, 16, 3, 2, kh=2, kw=1, pad=(0, 0), form="fused"),
    # ---- tcgen05 implicit-GEMM forward: every reachable (precision, blocks per SM, stages), one / two MMAs along N
    #      (Npad up to 304), Cout % 16 = 12, C % 32 in {8, 16, 24, 0}, K = 1, P < 128 and P % 128 != 0, no bias / mask
    _c("ig3_o44_mb2_s2", 2, 40, 44, 11, 13, form="igemm"),
    _c("ig3_o80_mb1_s4_asym", 2, 48, 80, 12, 14, form="igemm", **ASYM),
    _c("ig3_o112_mb1_s3", 2, 24, 112, 9, 10, form="igemm", bias=False),
    _c("ig3_o304_mb1_s2_2mma", 2, 64, 304, 7, 9, form="igemm", mask=False),
    _c("ig3_o264_2mma_asym2", 1, 72, 264, 8, 9, form="igemm", **ASYM2),
    _c("ig3_k1_c8", 1, 8, 20, 5, 7, kh=1, kw=1, pad=(0, 0), form="igemm", mask=False, bias=False),
    _c("igt_o44_mb2_s4", 2, 40, 44, 11, 13, form="igemm", tf32=True),
    _c("igt_o80_mb2_s3_asym", 2, 48, 80, 12, 14, form="igemm", tf32=True, **ASYM),
    _c("igt_o176_mb2_s2", 2, 24, 176, 9, 10, form="igemm", tf32=True, bias=False),
    _c("igt_o300_mb1_s4_2mma", 2, 64, 300, 7, 9, form="igemm", tf32=True, mask=False),
    _c("igt_o264_2mma_asym2", 1, 72, 264, 8, 9, form="igemm", tf32=True, **ASYM2),
    _c("igt_k1_c8", 1, 8, 20, 5, 7, kh=1, kw=1, pad=(0, 0), form="igemm", tf32=True, mask=False, bias=False),
]
# the mask head's layers at one offset group, as the library dispatches them, in training and in inference
CASES += [_c(f"{name}_{'train' if train else 'infer'}", LAYER_N[name], cin, cout, h, w, train=train)
          for name, cin, cout, h, w in LAYERS for train in (True, False)]
# float64 through the im2col form at the real shapes
CASES += [_c(f"{name}_f64", 2, cin, cout, h, w, form="im2col", dtype="float64") for name, cin, cout, h, w in LAYERS]

CASE_IDS = [c.name for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS)


# ---------------------------------------------------------------------------------------------------------------------
# host rules
# ---------------------------------------------------------------------------------------------------------------------
def zslices(n):
    """grid-z launches of a CUDA-core launcher over n batch items"""
    return -(-n // MAX_GRID_Z) if n > 0 else 0


def gather_vg(c, og, dtype):
    """(V, G) of dcn_im2col_kernel / dcn_col2im_kernel (deform_conv_capi.cu dispatch)"""
    cg = c // og
    if dtype == "float32" and cg % 4 == 0:
        return 4, (8 if cg // 4 >= 8 else 4)
    return 1, (32 if cg >= 32 else 8)


def fused_plan(c, cout, kh, kw, og):
    """deform_conv_capi.cu fused_plan for float32"""
    p = dict(G=0, lanes_fwd=False, lanes_bwd=False, constant=False, CT=16, lanes_elems=0, const_elems=0)
    if c % og or (c // og) % 4:
        return p
    cg, k = c // og, kh * kw
    small = cout in SMALL_COUT
    p["G"] = 8 if cg // 4 > 4 else 4
    p["constant"] = og == 1 and c in CONST_C and cout % 16 == 0 and cout <= 64
    p["CT"] = 32 if cout % 32 == 0 else 16
    p["lanes_bwd"] = small
    p["lanes_fwd"] = small and not p["constant"]
    if p["lanes_fwd"] or p["lanes_bwd"]:
        p["lanes_elems"] = k * og * (-(-(cg // 4) // p["G"])) * cout * p["G"] * 4
    if p["constant"]:
        p["const_elems"] = k * c * cout
    return p


def fused_form(c, cout, kh, kw, og, dtype="float32"):
    if dtype != "float32":
        return 0
    p = fused_plan(c, cout, kh, kw, og)
    return (1 if p["lanes_fwd"] or p["constant"] else 0) | (2 if p["lanes_bwd"] else 0)


def const_chunks(c, ct, k):
    """kernel-position chunks of the constant-bank forward (one launch per 16/32-channel tile and chunk)"""
    k_fit = CONST_FLOATS // (c * ct)
    n_chunks = -(-k // k_fit)
    step = -(-k // n_chunks)
    return len(range(0, k, step))


def wgrad_supported(c, cout, kh, kw):
    return c in (16, 32) and cout in SMALL_COUT and kh * kw <= 65535


def wgrad_run(c, n, ho, wo, k, helper_blocks):
    """pixels per lane group of dcn_wgrad_kernel (devis_dcn_weight_grad)"""
    gpb, plane, run = 256 // (c // 4), ho * wo, 64
    while run > 8 and -(-plane // (gpb * run)) * k * n < helper_blocks:
        run //= 2
    return run


def igemm_plan(c, cout, kh, kw):
    """deform_conv_capi.cu igemm_plan: None when unsupported, else Npad, n0, n1 and per precision (MINB, stages)"""
    if c <= 0 or cout <= 0 or c % 8 or cout % 4:
        return None
    npad = -(-cout // 16) * 16
    if npad > 512:
        return None
    n0 = npad if npad <= 256 else -(-(npad // 2) // 16) * 16

    def shape(split):
        stage = (2 if split else 1) * (IG_ATILE + npad * 128)
        blocks = 2 if (2 * stage + IG_GEOM + 2048) * 2 <= IG_SMEM else 1
        return blocks, min(IG_MAX_STAGES, (IG_SMEM // blocks - IG_GEOM - 256 - 1024 - 1024) // stage)

    if shape(True)[1] < 2:
        return None
    return dict(Npad=npad, n0=n0, n1=npad - n0, nchunks=-(-c // IG_BK), split=shape(True), tf32=shape(False))


def route(case):
    """which autograd Function serves the call: im2col | fused | igemm"""
    if case.form == "igemm":
        return "igemm"
    fused_on = case.form in ("fused", "auto")
    form = fused_form(case.cin, case.cout, case.kh, case.kw, case.og, case.dtype) if fused_on else 0
    fn = "fused" if form & 1 and (form & 2 or not case.train) else "im2col"
    if case.form == "auto" and case.og == 1 and case.dtype == "float32" and \
            igemm_plan(case.cin, case.cout, case.kh, case.kw) is not None and \
            (not form & 1 or (case.cin * case.k >= 576 and case.cout >= 32 and not form & 2 and not case.train)):
        fn = "igemm"
    return fn


def _per(n, per):
    return max(1, min(n, per))


def _slices(n, per):
    return [min(n, n0 + per) - n0 for n0 in range(0, n, per)]


def plan(case, det=False, helper_blocks=B200_HELPER_BLOCKS):
    """what one forward (+ backward in training) of the case does:
       calls     C entry points that launch kernels, in call order
       dcn       KERNEL_DCN launches, igemm KERNEL_DCN_IGEMM launches
       inst      kernel instantiations reached, launch shapes included"""
    c, cout, kh, kw, og, n = case.cin, case.cout, case.kh, case.kw, case.og, case.n
    ho, wo, k, dt = case.ho, case.wo, case.k, case.dtype
    calls, inst = [], set()
    dcn = igemm = 0
    fn = route(case)
    v, g = gather_vg(c, og, dt)
    det = det and case.train and dt == "float32"
    col_per = CHUNK_BYTES // max(1, ho * wo * k * c * 4)
    det_per = lambda per: min(per, CHUNK_BYTES // max(1, case.h * case.w * c * 8)) if det else per

    def im2col_calls(name, per):
        nonlocal dcn
        for m in _slices(n, per):
            calls.append(name)
            dcn += zslices(m)
        inst.add(("im2col", dt, v, g))

    def col2im_calls(name, per):
        nonlocal dcn
        for m in _slices(n, _per(n, det_per(per))):
            calls.append(name)
            dcn += zslices(m)
        inst.add(("col2im_det" if det else "col2im", dt, v, g))

    if fn == "im2col":
        im2col_calls("devis_dcn_im2col_og", n)
        if case.train:
            col2im_calls("devis_dcn_col2im_og", n)
    elif fn == "fused":
        p = fused_plan(c, cout, kh, kw, og)
        calls.append("devis_dcn_pack_weight_og")
        dcn += (p["lanes_elems"] > 0) + (p["const_elems"] > 0)
        calls.append("devis_dcn_fused_forward_og")
        if p["constant"]:
            chunks = const_chunks(c, p["CT"], k)
            dcn += (cout // p["CT"]) * chunks * zslices(n)
            inst.add(("const_fwd", c, p["CT"]))
            inst.add(("const_chunks", min(chunks, 3)))
            if cout // p["CT"] > 2:
                inst.add(("const_tiles", 3))
        else:
            dcn += zslices(n)
            inst.add(("lane_fwd", cout, p["G"]))
        if case.train:
            for m in _slices(n, _per(n, det_per(n))):
                calls.append("devis_dcn_fused_backward_og")
                dcn += zslices(m)
            inst.add(("lane_bwd_det" if det else "lane_bwd", cout, p["G"]))
            if og == 1 and not det and wgrad_supported(c, cout, kh, kw):
                calls.append("devis_dcn_weight_grad")
                dcn += zslices(n)
                inst.add(("wgrad", cout, c // 4))
                inst.add(("wgrad_run", wgrad_run(c, n, ho, wo, k, helper_blocks)))
            else:
                im2col_calls("devis_dcn_im2col_og", _per(n, col_per))
    else:
        ip = igemm_plan(c, cout, kh, kw)
        calls += ["devis_dcn_igemm_pack_weight", "devis_dcn_igemm_forward"]
        dcn += 1
        igemm += 1
        minb, stages = ip["tf32"] if case.tf32 else ip["split"]
        inst.add(("igemm", "tf32" if case.tf32 else "3xtf32", minb, stages))
        inst.add(("igemm_mmas", "tf32" if case.tf32 else "3xtf32", 2 if ip["n1"] else 1))
        if case.train:
            im2col_calls("devis_dcn_im2col", _per(n, col_per))
            col2im_calls("devis_dcn_col2im_ex", _per(n, col_per))
    return dict(route=fn, calls=calls, dcn=dcn, igemm=igemm, inst=inst)


def all_instantiations():
    """every kernel instantiation and launch shape of the deformable convolution"""
    inst = set()
    for v, g in ((4, 4), (4, 8), (1, 8), (1, 32)):
        inst |= {("im2col", "float32", v, g), ("col2im", "float32", v, g), ("col2im_det", "float32", v, g)}
    for g in (8, 32):
        inst |= {("im2col", "float64", 1, g), ("col2im", "float64", 1, g)}
    for co in SMALL_COUT:
        for g in (4, 8):
            inst |= {("lane_fwd", co, g), ("lane_bwd", co, g), ("lane_bwd_det", co, g), ("wgrad", co, g)}
    inst |= {("const_fwd", c, ct) for c in CONST_C for ct in (16, 32)}
    inst |= {("const_chunks", m) for m in (1, 2, 3)} | {("const_tiles", 3)}
    inst |= {("wgrad_run", r) for r in (8, 16, 32, 64)}
    for prec, key in (("3xtf32", "split"), ("tf32", "tf32")):
        for npad in range(16, 513, 16):
            ip = igemm_plan(64, npad, 3, 3)
            if ip is not None:
                inst.add(("igemm", prec) + ip[key])
                inst.add(("igemm_mmas", prec, 2 if ip["n1"] else 1))
    return inst


# ---------------------------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------------------------
GRID = 1024.0      # offsets on a 2^-10 grid: every sampling coordinate is exact in float32 and float64 alike


def _base(case):
    """integer sampling position of every (virtual position, output pixel) before the offset: (1, og*K, Ho, Wo) x 2"""
    kk = torch.arange(case.og * case.k) % case.k
    ky = (kk // case.kw).double().view(1, -1, 1, 1) * case.dil[0]
    kx = (kk % case.kw).double().view(1, -1, 1, 1) * case.dil[1]
    by = torch.arange(case.ho).double().view(1, 1, -1, 1) * case.stride[0] - case.pad[0] + ky
    bx = torch.arange(case.wo).double().view(1, 1, 1, -1) * case.stride[1] - case.pad[1] + kx
    return by, bx


def _edge_targets(size, shape, gen):
    """sampling coordinates on the edges of [0, size): an integer inside, size - 1, inside (-1, 0), -1, size"""
    kind = torch.randint(0, 5, shape, generator=gen)
    inner = torch.randint(0, size, shape, generator=gen).double()
    frac = -torch.randint(1, int(GRID), shape, generator=gen).double() / GRID
    return torch.stack([inner, torch.full(shape, size - 1.0, dtype=torch.float64), frac,
                        torch.full(shape, -1.0, dtype=torch.float64),
                        torch.full(shape, float(size), dtype=torch.float64)]).gather(0, kind[None])[0]


def operands(case, seed, edge_share=0.25):
    """seeded float64 operands (x, offset, weight, bias, mask, grad_out) on the CPU; ``edge_share`` of the taps have their
    row and, independently, their column coordinate steered onto an edge coordinate"""
    gen = torch.Generator().manual_seed(seed)
    n, c, cout, k, og = case.n, case.cin, case.cout, case.k, case.og
    shape = (n, og * k, case.ho, case.wo)
    x = torch.randn(n, c, case.h, case.w, generator=gen, dtype=torch.float64)
    by, bx = _base(case)
    py = by + torch.round(torch.randn(shape, generator=gen, dtype=torch.float64) * 2 * GRID) / GRID
    px = bx + torch.round(torch.randn(shape, generator=gen, dtype=torch.float64) * 2 * GRID) / GRID
    py = torch.where(torch.rand(shape, generator=gen) < edge_share, _edge_targets(case.h, shape, gen), py)
    px = torch.where(torch.rand(shape, generator=gen) < edge_share, _edge_targets(case.w, shape, gen), px)
    off = torch.stack([py - by, px - bx], dim=2).reshape(n, 2 * og * k, case.ho, case.wo)
    weight = torch.randn(cout, c, case.kh, case.kw, generator=gen, dtype=torch.float64) / math.sqrt(c * k)
    bias = torch.randn(cout, generator=gen, dtype=torch.float64) if case.bias else None
    mask = 2 * torch.rand(shape, generator=gen, dtype=torch.float64) if case.mask else None
    gout = torch.randn(n, cout, case.ho, case.wo, generator=gen, dtype=torch.float64)
    return x, off, weight, bias, mask, gout


def poison(case, x, off, far=-50.0):
    """pixels (0..1, 0..1) of every channel become non-finite (Inf, -Inf, NaN); every tap one of whose LIVE corners is such
    a pixel is moved entirely outside the map (``far`` rows above it), so the poisoned pixels are reached only as dead
    corners.  Returns (poisoned x, finite x, offsets): the two inputs differ in those pixels only."""
    by, bx = _base(case)
    n, k, og = case.n, case.k, case.og
    o = off.view(n, og * k, 2, case.ho, case.wo)
    py, px = by + o[:, :, 0], bx + o[:, :, 1]
    inside = (py > -1) & (px > -1) & (py < case.h) & (px < case.w)
    y0, x0 = torch.floor(py), torch.floor(px)
    touch = torch.zeros_like(inside)
    for dy in (0, 1):
        for dx in (0, 1):
            yy, xx = y0 + dy, x0 + dx
            live = inside & (yy >= 0) & (yy <= case.h - 1) & (xx >= 0) & (xx <= case.w - 1)
            touch |= live & (yy <= 1) & (xx <= 1)
    # and a fixed share of the other taps too, so taps entirely outside the map occur in every case
    touch |= (torch.arange(touch.numel()).view(touch.shape) % 5) == 0
    py = torch.where(touch, torch.full_like(py, far), py)
    off = torch.stack([py - by, px - bx], dim=2).reshape(off.shape)
    bad = x.clone()
    bad[:, :, 0, 0], bad[:, :, 0, 1], bad[:, :, 1, 0], bad[:, :, 1, 1] = float("inf"), float("-inf"), float("nan"), float("inf")
    return bad, x, off
