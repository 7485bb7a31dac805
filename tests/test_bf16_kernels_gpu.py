"""Every bfloat16 instantiation of the attention kernels, and every launch shape the tuning keys can force, against a
float64 reference evaluated on exactly the values the kernels read.

Inputs are generated in fp32; value and grad_out are rounded to bf16 before both the kernel and the reference see them
(sampling locations, attention weights, offsets and logits stay fp32, as the kernels read them).  The reference is the
float64 PyTorch oracle: oracle/msda_torch.py for the drop-in op, oracle/temporal_torch.temporal_core_per_frame for the
whole-clip op, and the fused op's prologue (encoder_locations / decoder_locations plus the joint softmax) in float64.

Acceptance rule of a bf16 result (the output, and grad_value, which is accumulated in fp32 and rounded once):
  * every element:  |got - ref| <= 2^-8 |ref| + EPS max|ref|.  2^-8 is bf16's unit roundoff, so a correctly rounded
    result meets the bound with EPS = 0; EPS covers the fp32 accumulation and the fp32 location arithmetic before the
    rounding;
  * at most 1 % of the non-zero elements differ from round-to-nearest(ref).  A kernel that truncates instead of
    rounding changes about half of them, while staying within the 1e-2 class bounds of the older bf16 tests.
The fp32 results of a bf16 run (grad_sampling_loc, grad_attn_weight; the fused op's offset, logit and reference-point
gradients) are computed in fp32 from the same operands as the reference and meet the fp32 suite's bound: normalised max
error <= 1e-4.
The bf16 grad_value accumulation mode (every partial sum rounded to bf16) keeps the bounds of
test_temporal_gpu.py::test_bf16_grad_value_accumulation_mode, and every other result must be bit-identical to the
default mode.  The same launch-shape sweep runs for fp32 at the fp32 bounds (output 1e-5, gradients 1e-4).

Every case asserts which kernel family served it (devis_msda_kernel_launches), so a silent change of path cannot pass.
Setting DEVIS_TEST_ERROR_LOG=<file> appends the measured errors of every case to that file as JSON lines.
"""
import contextlib
import functools
import json
import os

import pytest
import torch

from conftest import nmax

pytestmark = pytest.mark.gpu

U_BF16 = 2.0 ** -8          # unit roundoff of bfloat16 (8-bit significand)
# fp32-side error allowed before the final rounding, in units of max|ref|.  Measured on an NVIDIA B200 (1000 W power
# limit) over every case of this file: 2.8e-7 at most (the output of the 20-frame fused clip, 320 taps per query; the
# drop-in op 1.3e-7, the fused op 1.2e-7, the whole-clip op 1.9e-8), so 2e-6 leaves a factor of 7.  The share of
# elements that differ from round-to-nearest(ref) was 0.07 % at most.
EPS = 2e-6
MAX_RN_MISMATCH = 0.01
TOL_F32_OUT, TOL_F32_GRAD = 1e-5, 1e-4
# bounds of the bf16 grad_value accumulation mode (test_temporal_gpu.py::test_bf16_grad_value_accumulation_mode)
TOL_HALF_NMAX, TOL_HALF_RMS = 1e-1, 1e-2


# ---- bookkeeping ------------------------------------------------------------------------------------------------------
def _families():
    from devis_b200 import _lib
    return {k: _lib.kernel_launches(getattr(_lib, k)) for k in
            ("KERNEL_FWD_GROUPED", "KERNEL_FWD_GENERIC", "KERNEL_BWD_GROUPED", "KERNEL_BWD_GENERIC",
             "KERNEL_FUSED_FWD", "KERNEL_FUSED_BWD", "KERNEL_BWD_SORTED")}


@contextlib.contextmanager
def _launches():
    """yields a dict that holds, after the block, how many kernels of each family the block launched"""
    before = _families()
    delta = {}
    yield delta
    torch.cuda.synchronize()
    after = _families()
    delta.update({k: after[k] - before[k] for k in after})


def _expect(delta, **want):
    """`want`: family name without the KERNEL_ prefix -> launches; every family not named must not have run"""
    full = {"KERNEL_" + k: v for k, v in want.items()}
    assert {k: v for k, v in delta.items() if v or k in full} == full, delta


def _record(case, errs):
    path = os.environ.get("DEVIS_TEST_ERROR_LOG")
    if path:
        with open(path, "a") as fh:
            fh.write(json.dumps({"case": case, **errs}) + "\n")


@pytest.fixture
def knobs():
    """sets tuning keys (launch shapes) and the backward modes for one test, and restores the defaults afterwards"""
    from devis_b200 import MultiScaleDeformableAttention as MSDA, _lib

    def set_keys(**keys):
        for k, v in keys.items():
            _lib.set_tuning(int(k.lstrip("k")), v)
    try:
        yield set_keys
    finally:
        for k in range(16):
            _lib.set_tuning(k, 0)
        MSDA.set_deterministic(False)
        MSDA.set_bf16_grad_value_accumulation(False)


@contextlib.contextmanager
def _mode(mode):
    """default | deterministic (64-bit fixed-point grad_value) | half (bf16 grad_value accumulation)"""
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    MSDA.set_deterministic(mode == "deterministic")
    MSDA.set_bf16_grad_value_accumulation(mode == "half")
    try:
        yield
    finally:
        MSDA.set_deterministic(False)
        MSDA.set_bf16_grad_value_accumulation(False)


# ---- acceptance -------------------------------------------------------------------------------------------------------
def _bf16_errors(got, ref):
    """(eps, mismatch) of a bf16 result against its float64 reference: eps is the smallest EPS for which every element
    meets |got - ref| <= 2^-8 |ref| + EPS max|ref|; mismatch is the fraction of non-zero reference elements where got
    differs from round-to-nearest(ref)"""
    assert got.dtype == torch.bfloat16, got.dtype
    g = got.detach().double().cpu()
    r = ref.detach().double().cpu()
    scale = max(r.abs().max().item(), 1e-30)
    eps = ((g - r).abs() - U_BF16 * r.abs()).clamp_min(0).max().item() / scale
    nz = r != 0
    rn = r.to(torch.bfloat16).double()
    mismatch = (g[nz] != rn[nz]).double().mean().item() if nz.any() else 0.0
    return eps, mismatch


def _check(case, got, ref, tol):
    """got / ref: dicts of result name -> tensor.  tol[name] is "bf16" (the rule above) or a normalised max error bound"""
    errs, bad = {}, []
    for name, want in ref.items():
        t = tol[name]
        if t == "bf16":
            eps, mismatch = _bf16_errors(got[name], want)
            errs[name + ".eps"], errs[name + ".rn_mismatch"] = eps, mismatch
            if not (eps <= EPS and mismatch <= MAX_RN_MISMATCH):
                bad.append(name)
        else:
            e = nmax(got[name].detach().double().cpu().numpy(), want.detach().double().cpu().numpy())
            errs[name + ".nmax"] = e
            if not e <= t:
                bad.append(name)
    _record(case, errs)
    assert not bad, (bad, errs)


def _check_half(case, got, base, ref, exact):
    """bf16 grad_value accumulation: grad_value within the bf16-accumulation bounds of the float64 reference, every
    name in `exact` bit-identical to the default-mode run `base`"""
    gv, want = got["grad_value"], ref["grad_value"].detach().double().cpu()
    assert gv.dtype == torch.bfloat16
    g = gv.double().cpu()
    scale = want.abs().max().item()
    errs = {"grad_value.nmax": (g - want).abs().max().item() / scale,
            "grad_value.rms": ((g - want) ** 2).mean().sqrt().item() / scale}
    _record(case, errs)
    assert errs["grad_value.nmax"] < TOL_HALF_NMAX and errs["grad_value.rms"] < TOL_HALF_RMS, errs
    for name in exact:
        assert torch.equal(got[name], base[name]), name


def _tol(dtype, names_bf16, names_f32):
    bf = dtype == torch.bfloat16
    tol = {n: "bf16" if bf else (TOL_F32_OUT if n == "out" else TOL_F32_GRAD) for n in names_bf16}
    tol.update({n: TOL_F32_OUT if n.startswith(("loc_", "aw_")) else TOL_F32_GRAD for n in names_f32})
    return tol


# ---- drop-in op (MSDeformAttnFunction) --------------------------------------------------------------------------------
# What msda_capi.cu (launch_forward / launch_backward) selects for each shape; BF = bf16 value, QPG from pick_shape or
# tuning keys 1 / 3.  fp32 value: the same kernels with BF = false, and msda_fwdv_kernel for the D = 32, P % 4 == 0 forward.
DROPIN = {
    # msda_fwd8v_kernel<QPG, DeviceLevels, 512> (row size an immediate), msda_bwd_kernel<true, 8, QPG>
    "d32p4m8": dict(d=32, m=8, p=4, grouped=True),
    # msda_fwd8v_kernel<QPG, DeviceLevels, 0> (row size at run time), msda_bwd_kernel<true, 8, QPG>
    "d32p4m3": dict(d=32, m=3, p=4, grouped=True),
    # P % 4 != 0: msda_fwd_kernel<true, 8, QPG>, msda_bwd_kernel<true, 8, QPG>
    "d32p3": dict(d=32, m=8, p=3, grouped=True),
    # msda_fwd_kernel<true, 4, QPG>, msda_bwd_kernel<true, 4, QPG> (half accumulation: msda_bwd_kernel<true, 4, 1, ., true>)
    "d16": dict(d=16, m=8, p=4, grouped=True),
    # msda_fwd_generic_kernel<__nv_bfloat16>, msda_bwd_generic_kernel<__nv_bfloat16>
    "d8": dict(d=8, m=4, p=4, grouped=False),
    "d33": dict(d=33, m=2, p=3, grouped=False),
}
DROPIN_SHAPES = ((9, 13), (5, 7), (3, 4))
DROPIN_BATCH = 2
# Lq in each band of pick_shape (< 128, 128..1023, >= 1024); all prime, so the last block of every launch shape is partial
LQ_SMALL, LQ_MID, LQ_LARGE = 97, 331, 1031
FWD_THREADS, QPGS = (32, 64, 128, 256), (1, 2, 4)
# launch: None = the built-in heuristic, else (threads, qpg) forced through keys 0 / 1 (forward) and 2 / 3 (backward);
# a QPG the kernel is not instantiated with is clamped to its largest one by pick_shape (backward: 2; fwd8v: 2)
LAUNCHES = [(None, LQ_SMALL), (None, LQ_MID), (None, LQ_LARGE)] + [((t, q), LQ_MID) for t in FWD_THREADS for q in QPGS]


def _dropin_params():
    for dtype in ("bf16", "fp32"):
        for name, cfg in DROPIN.items():
            modes = ["default", "deterministic"] + (["half"] if dtype == "bf16" and cfg["grouped"] else [])
            for mode in modes:
                for launch, lq in LAUNCHES:
                    if launch is not None and not cfg["grouped"]:
                        continue        # the generic kernels have one launch shape
                    tag = "auto" if launch is None else f"t{launch[0]}q{launch[1]}"
                    yield pytest.param(dtype, name, mode, launch, lq, id=f"{dtype}-{name}-{mode}-{tag}-lq{lq}")


def _dtype(name):
    return {"bf16": torch.bfloat16, "fp32": torch.float32}[name]


@functools.lru_cache(maxsize=None)
def _dropin_case(name, lq, dtype_name):
    """CPU inputs (value / grad_out in `dtype`, locations and weights fp32) and the float64 reference on them"""
    from devis_b200 import synthetic
    from oracle import msda_torch
    cfg = DROPIN[name]
    dtype = _dtype(dtype_name)
    g = torch.Generator().manual_seed(1000 * list(DROPIN).index(name) + lq)
    n, m, d, p, nl = DROPIN_BATCH, cfg["m"], cfg["d"], cfg["p"], len(DROPIN_SHAPES)
    s = sum(h * w for h, w in DROPIN_SHAPES)
    sizes = torch.tensor([[w, h] for h, w in DROPIN_SHAPES], dtype=torch.float32)
    loc = torch.rand(n, lq, m, nl, p, 2, generator=g) * 1.2 - 0.1          # some taps leave the map across an edge
    loc = synthetic.make_boundary_safe(loc, sizes).contiguous()
    aw = torch.softmax(torch.randn(n, lq, m, nl * p, generator=g), -1).view(n, lq, m, nl, p).contiguous()
    value = torch.randn(n, s, m, d, generator=g).to(dtype)
    gout = torch.randn(n, lq, m * d, generator=g).to(dtype)
    out, gv, gl, ga = msda_torch.msda_forward_backward_torch(value.double(), torch.tensor(DROPIN_SHAPES), loc.double(),
                                                             aw.double(), gout.double())
    ref = {"out": out, "grad_value": gv, "grad_loc": gl, "grad_aw": ga}
    return (value, loc, aw, gout), ref


def _dropin_run(inputs):
    from devis_b200 import MSDeformAttnFunction
    value, loc, aw, gout = (t.cuda() for t in inputs)
    shapes = torch.tensor(DROPIN_SHAPES, device="cuda")
    areas = shapes.prod(1)
    lsi = torch.cat([areas.new_zeros(1), areas.cumsum(0)[:-1]])
    v, l_, a = (t.clone().requires_grad_(True) for t in (value, loc, aw))
    out = MSDeformAttnFunction.apply(v, shapes, lsi, l_, a, 64)
    out.backward(gout)
    return {"out": out.detach(), "grad_value": v.grad, "grad_loc": l_.grad, "grad_aw": a.grad}


@pytest.mark.parametrize("dtype_name,name,mode,launch,lq", list(_dropin_params()))
def test_dropin_op_against_float64(knobs, dtype_name, name, mode, launch, lq):
    """Drop-in op at every shape of DROPIN (the comment of each names the instantiation it selects), in the default,
    deterministic and bf16-accumulation modes, at the heuristic's launch shape in each Lq band and at every forced
    (threads, QPG); the forced fp32 shapes run msda_fwdv_kernel / msda_fwd_kernel<false, ...> / msda_bwd_kernel<false,
    ...> the same way."""
    cfg = DROPIN[name]
    dtype = _dtype(dtype_name)
    inputs, ref = _dropin_case(name, lq, dtype_name)
    if launch is not None:
        t, q = launch
        knobs(k0=t, k1=q, k2=t, k3=q)
    with _mode(mode), _launches() as delta:
        got = _dropin_run(inputs)
    if cfg["grouped"]:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    else:
        _expect(delta, FWD_GENERIC=1, BWD_GENERIC=1)
    assert got["out"].dtype == dtype and got["grad_value"].dtype == dtype and got["grad_loc"].dtype == torch.float32
    case = f"dropin-{dtype_name}-{name}-{mode}-{launch}-{lq}"
    if mode == "half":
        with _mode("default"):
            base = _dropin_run(inputs)
        _check_half(case, got, base, ref, exact=("out", "grad_loc", "grad_aw"))
        return
    _check(case, got, ref, _tol(dtype, ("out", "grad_value"), ("grad_loc", "grad_aw")))


# ---- whole-clip op (temporal_ms_deform_attn) ----------------------------------------------------------------------------
# reduced encoder clip: one query per pixel, 4 levels stored back to back (an even count: the sorted deterministic
# backward applies), D = 32, 8 heads, 4 + 4 points -> msda_fwd8v_kernel<1, ClipTable, 512>, msda_bwd_kernel<true, 8, 1>,
# msda_bwds_kernel<true, true>
CLIP_SHAPES = ((12, 16), (6, 8), (3, 4), (2, 2))
CLIP_FRAMES = 3
CLIP_NAMES = ("value", "loc_curr", "aw_curr", "loc_temporal", "aw_temporal")


@functools.lru_cache(maxsize=None)
def _clip_case():
    from devis_b200 import synthetic
    from oracle import temporal_torch
    clip = synthetic.make_clip(n_frames=CLIP_FRAMES, shapes=CLIP_SHAPES, dist="local", seed=31, dtype=torch.bfloat16,
                               device="cpu")
    leaves = [clip[k].double().requires_grad_(True) for k in CLIP_NAMES]
    offs = [torch.tensor([f - t for f in row]) for t, row in enumerate(clip["frame_table"])]
    out = temporal_torch.temporal_core_per_frame(*leaves, torch.tensor(CLIP_SHAPES), offs)
    out.backward(clip["grad_out"].double())
    ref = {"out": out.detach()}
    ref.update({"grad_" + k: x.grad for k, x in zip(CLIP_NAMES, leaves)})
    return clip, ref


@pytest.mark.parametrize("order,mode", [("none", "default"), ("tiles", "default"), ("none", "deterministic"),
                                        ("tiles", "deterministic"), ("tiles", "half")])
def test_whole_clip_op_bf16_against_float64(knobs, order, mode):
    """temporal_ms_deform_attn on a bf16 clip, queries in index order or in geom.tile_order; deterministic mode with a
    query order runs the sorted fixed-point backward (KERNEL_BWD_SORTED), without one the direct fixed-point scatter"""
    from devis_b200 import clip_geometry, temporal_ms_deform_attn
    clip, ref = _clip_case()
    geom = clip_geometry.ClipGeometry(CLIP_SHAPES, CLIP_FRAMES, clip["frame_table"])
    q_order = geom.tile_order("cuda") if order == "tiles" else None
    assert order == "none" or q_order is not None

    def run():
        leaves = [clip[k].cuda().requires_grad_(True) for k in CLIP_NAMES]
        out = temporal_ms_deform_attn(*leaves, geom, q_order)
        out.backward(clip["grad_out"].cuda())
        got = {"out": out.detach()}
        got.update({"grad_" + k: x.grad for k, x in zip(CLIP_NAMES, leaves)})
        return got

    with _mode(mode), _launches() as delta:
        got = run()
    if mode == "deterministic" and q_order is not None:
        _expect(delta, FWD_GROUPED=1, BWD_SORTED=1)
    else:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    case = f"clip-{order}-{mode}"
    if mode == "half":
        with _mode("default"):
            base = run()
        _check_half(case, got, base, ref, exact=["out"] + ["grad_" + k for k in CLIP_NAMES[1:]])
        return
    _check(case, got, ref, _tol(torch.bfloat16, ("out", "grad_value"), ["grad_" + k for k in CLIP_NAMES[1:]]))


# ---- fused op (TemporalMSDeformAttnFusedFunction) -----------------------------------------------------------------------
def _safe_offsets(locate, off_c, off_t, sizes, wt):
    """fp32 offsets whose sampling locations keep 0.02 px from every cell border (synthetic.make_boundary_safe).
    `locate(off_c, off_t) -> (loc_c, loc_t)` is affine in the offsets (float64), so one step along its slope lands on
    the safe location; the fp32 rounding of the offsets then moves a tap by far less than the margin."""
    from devis_b200 import synthetic
    lc, lt = locate(off_c, off_t)
    lc1, lt1 = locate(off_c + 1, off_t + 1)
    sc = synthetic.make_boundary_safe(lc, sizes)
    st = synthetic.make_boundary_safe(lt, sizes.repeat(wt, 1))
    return (off_c + (sc - lc) / (lc1 - lc)).float(), (off_t + (st - lt) / (lt1 - lt)).float()


FUSED_CASES = {
    # encoder form (pixel reference points, one query per pixel): tmsda_fused_fwd8_kernel<512> / <0>,
    # tmsda_fused_bwd_kernel<BF, HALF_ACC, false, DET>
    "enc_m8": dict(m=8, form="enc"),
    "enc_m3": dict(m=3, form="enc"),
    # general form (decoder: box reference points, by-products): tmsda_fused_fwd_kernel<BF, 1, true, 512>,
    # tmsda_fused_bwd_kernel<BF, HALF_ACC, true, DET>
    "box_own": dict(m=8, form="box", tref="own"),
    "box_sampled": dict(m=8, form="box", tref="sampled"),
}
FUSED_SHAPES = ((10, 14), (5, 7), (3, 4), (2, 2))
FUSED_FRAMES, FUSED_PC, FUSED_PT, FUSED_DEC_QUERIES = 3, 4, 4, 37


def _fused_inputs(cfg, dtype, shapes, n_frames, pc, pt, seed):
    """CPU operands of the fused op and a float64 forward/backward of the unfused reference on them"""
    from devis_b200 import clip_geometry, synthetic
    from oracle import temporal_torch
    g = torch.Generator().manual_seed(seed)
    nl, wt, m = len(shapes), n_frames - 1, cfg["m"]
    s = sum(h * w for h, w in shapes)
    sizes = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float64)
    shp = torch.tensor(shapes)
    offs = temporal_torch.all_frames_offsets(n_frames)
    if cfg["form"] == "enc":
        lq = s
        ref = synthetic.pixel_reference_points(shapes, n_frames, "cpu")
        off_c = 2.0 * torch.randn(n_frames, lq, m, nl, pc, 2, generator=g, dtype=torch.float64)
        off_t = 2.0 * torch.randn(n_frames, lq, m, wt * nl, pt, 2, generator=g, dtype=torch.float64)

        def locate(oc, ot, r=None):
            return temporal_torch.encoder_locations((ref if r is None else r).double(), oc, ot, shp, wt)
    else:
        lq = FUSED_DEC_QUERIES
        xy = torch.rand(n_frames, lq, nl, 2, generator=g) * 0.8 + 0.1
        wh = torch.rand(n_frames, lq, nl, 2, generator=g) * 0.3 + 0.1
        ref = torch.cat([xy, wh], -1).contiguous()
        off_c = 0.8 * pc * torch.randn(n_frames, lq, m, nl, pc, 2, generator=g, dtype=torch.float64)
        off_t = 0.8 * pt * torch.randn(n_frames, lq, m, wt * nl, pt, 2, generator=g, dtype=torch.float64)
        ia = cfg["tref"] == "sampled"

        def locate(oc, ot, r=None):
            return temporal_torch.decoder_locations((ref if r is None else r).double(), oc, ot, shp, wt, offs, pc, pt, ia)
    off_c, off_t = _safe_offsets(locate, off_c, off_t, sizes, wt)
    lg_c = torch.randn(n_frames, lq, m, nl * pc, generator=g)
    lg_t = torch.randn(n_frames, lq, m, wt * nl * pt, generator=g)
    value = torch.randn(n_frames, s, m, 32, generator=g).to(dtype)
    gout = torch.randn(n_frames, lq, m * 32, generator=g).to(dtype)

    vv, rr, oc, ot, lc, lt = (x.double().requires_grad_(True) for x in (value, ref, off_c, off_t, lg_c, lg_t))
    joint = torch.softmax(torch.cat([lc, lt], -1), -1)
    aw_c = joint[..., :nl * pc].reshape(n_frames, lq, m, nl, pc)
    aw_t = joint[..., nl * pc:].reshape(n_frames, lq, m, wt * nl, pt)
    loc_c, loc_t = locate(oc, ot, rr)
    out = temporal_torch.temporal_core_per_frame(vv, loc_c, aw_c, loc_t, aw_t, shp, offs)
    out.backward(gout.double())
    ref64 = {"out": out.detach(), "grad_value": vv.grad, "grad_off_c": oc.grad, "grad_off_t": ot.grad,
             "grad_logit_c": lc.grad, "grad_logit_t": lt.grad, "grad_ref": rr.grad,
             "loc_c": loc_c.detach(), "aw_c": aw_c.detach(), "loc_t": loc_t.detach(), "aw_t": aw_t.detach()}
    geom = clip_geometry.ClipGeometry(shapes, n_frames, clip_geometry.all_frames_table(n_frames))
    return dict(value=value, ref=ref, off_c=off_c, off_t=off_t, lg_c=lg_c, lg_t=lg_t, gout=gout, geom=geom), ref64


@functools.lru_cache(maxsize=None)
def _fused_case(name, dtype_name):
    return _fused_inputs(FUSED_CASES[name], _dtype(dtype_name), FUSED_SHAPES, FUSED_FRAMES, FUSED_PC, FUSED_PT,
                         seed=500 + list(FUSED_CASES).index(name))


def _fused_run(x, ref_grad=False, want_sampling=False, tref=0, order=None):
    from devis_b200 import TemporalMSDeformAttnFusedFunction
    v, oc, ot, lc, lt = (x[k].cuda().requires_grad_(True) for k in ("value", "off_c", "off_t", "lg_c", "lg_t"))
    r = x["ref"].cuda().requires_grad_(ref_grad)
    res = TemporalMSDeformAttnFusedFunction.apply(v, r, oc, lc, ot, lt, x["geom"], order, tref, want_sampling)
    out = res[0] if want_sampling else res
    out.backward(x["gout"].cuda())
    got = {"out": out.detach(), "grad_value": v.grad, "grad_off_c": oc.grad, "grad_off_t": ot.grad,
           "grad_logit_c": lc.grad, "grad_logit_t": lt.grad}
    if ref_grad:
        got["grad_ref"] = r.grad
    if want_sampling:
        got.update(dict(zip(FUSED_SAMPLING, res[1:])))
    return got


FUSED_GRADS = ("grad_off_c", "grad_off_t", "grad_logit_c", "grad_logit_t")
FUSED_SAMPLING = ("loc_c", "aw_c", "loc_t", "aw_t")     # the by-products of want_sampling, in the order returned


def _fused_params():
    for name, cfg in FUSED_CASES.items():
        for mode in ("default", "deterministic", "half"):
            threads = (None,) if mode != "default" else (None, 32, 64, 128, 256)
            for t in threads:
                yield pytest.param(name, mode, t, id=f"{name}-{mode}-" + ("auto" if t is None else f"fwd{t}"))


@pytest.mark.parametrize("name,mode,fwd_threads", list(_fused_params()))
def test_fused_op_bf16_against_float64(knobs, name, mode, fwd_threads):
    """fused op on a bf16 clip, forward threads from the heuristic or forced through key 0.  General form: ref_dim 4,
    TREF_OWN / TREF_SAMPLED, sampling locations and weights returned, reference points that require grad -- except in
    deterministic mode, which the library refuses with them, and in the bf16 accumulation mode, whose other results
    must be bit-identical to the default mode (d/d(ref) is a float-atomic sum, not reproducible bit for bit)."""
    from devis_b200 import _lib
    cfg = FUSED_CASES[name]
    x, ref = _fused_case(name, "bf16")
    general = cfg["form"] == "box"
    tref = {"own": _lib.TREF_OWN, "sampled": _lib.TREF_SAMPLED}.get(cfg.get("tref"), _lib.TREF_LEVEL0)
    ref_grad = general and mode == "default"
    order = x["geom"].tile_order("cuda") if not general else None
    if fwd_threads is not None:
        knobs(k0=fwd_threads)
    kw = dict(ref_grad=ref_grad, want_sampling=general, tref=tref, order=order)
    with _mode(mode), _launches() as delta:
        got = _fused_run(x, **kw)
    _expect(delta, FUSED_FWD=1, FUSED_BWD=1)
    case = f"fused-{name}-{mode}-{fwd_threads}"
    sampling = FUSED_SAMPLING if general else ()
    if mode == "half":
        with _mode("default"):
            base = _fused_run(x, **kw)
        _check_half(case, got, base, ref, exact=("out",) + FUSED_GRADS + sampling)
        return
    f32 = FUSED_GRADS + (("grad_ref",) if ref_grad else ()) + sampling
    want = {k: ref[k] for k in ("out", "grad_value") + f32}
    _check(case, got, want, _tol(torch.bfloat16, ("out", "grad_value"), f32))


# ---- fused backward without the shared-memory park ----------------------------------------------------------------------
# devis_tmsda_fused_backward (msda_capi.cu) parks (w, d/dw) of every tap in shared memory only when
#     slot table + tap exchange + exchanges * threads * sizeof(float2) <= 48 KiB;
# otherwise tmsda_fused_bwd_kernel writes d/d(logit) to grad_logit and finishes it in a second loop.  _fused_bwd_smem
# restates that sum; keep the two in step.
def _fused_bwd_smem(n_levels, t_window, pc, pt, threads):
    n_slots = n_levels + t_window * n_levels
    exchanges = (n_levels * pc + 7) // 8 + (t_window * n_levels * pt + 7) // 8
    tap_exchange = (threads // 32) * 2048           # TapExchange<8>::kBytesPerWarp per warp
    return n_slots * 16 + tap_exchange + exchanges * threads * 8


NOPARK_CASES = {
    # the DeVIS clip of 20 frames, all frames sampled: 80 slots, 40 exchanges; 151 pixel queries select 128 threads
    "t20": dict(shapes=((9, 12), (5, 6), (3, 3), (2, 2)), n_frames=20, pc=4, pt=4, threads=None, default_threads=128),
    # a short clip with 8 + 8 points forced to 256 backward threads (key 2): 24 slots, 24 exchanges
    "t6p8": dict(shapes=((6, 8), (3, 4), (2, 2), (1, 1)), n_frames=6, pc=8, pt=8, threads=256, default_threads=64),
}
PARK_THREADS = 64


@functools.lru_cache(maxsize=None)
def _nopark_case(name, dtype_name):
    c = NOPARK_CASES[name]
    return _fused_inputs(dict(m=8, form="enc"), _dtype(dtype_name), c["shapes"], c["n_frames"], c["pc"], c["pt"],
                         seed=700 + list(NOPARK_CASES).index(name))


@pytest.mark.parametrize("dtype_name", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(NOPARK_CASES))
def test_fused_backward_without_park_against_float64_and_parked_run(knobs, name, dtype_name):
    """tmsda_fused_bwd_kernel<BF, false, false, false> with park_iters = 0 (d/d(logit) finished through grad_logit), at
    the default launch shape of a 20-frame clip and at a forced 256-thread launch, against float64 and against the same
    inputs at 64 backward threads, where the taps are parked in shared memory: the per-tap gradients do not depend on
    where the taps wait, so they must be bit-identical; grad_value differs only by the order of its float atomics"""
    c = NOPARK_CASES[name]
    dtype = _dtype(dtype_name)
    nl, wt = len(c["shapes"]), c["n_frames"] - 1
    threads = c["threads"] or c["default_threads"]
    lq = sum(h * w for h, w in c["shapes"])
    assert threads == (c["threads"] or (128 if lq >= 128 else 64))      # pick_shape's heuristic for this Lq
    assert _fused_bwd_smem(nl, wt, c["pc"], c["pt"], threads) > 48 * 1024
    assert _fused_bwd_smem(nl, wt, c["pc"], c["pt"], PARK_THREADS) <= 48 * 1024
    x, ref = _nopark_case(name, dtype_name)
    order = x["geom"].tile_order("cuda")
    if c["threads"]:
        knobs(k2=c["threads"])
    with _launches() as delta:
        got = _fused_run(x, order=order)
    _expect(delta, FUSED_FWD=1, FUSED_BWD=1)
    knobs(k2=PARK_THREADS)
    parked = _fused_run(x, order=order)
    for k in ("out",) + FUSED_GRADS:
        assert torch.equal(got[k], parked[k]), k
    assert nmax(got["grad_value"].float().cpu().numpy(), parked["grad_value"].float().cpu().numpy()) < \
        (1e-2 if dtype == torch.bfloat16 else 1e-5)
    want = {k: ref[k] for k in ("out", "grad_value") + FUSED_GRADS}
    _check(f"nopark-{name}-{dtype_name}", got, want, _tol(dtype, ("out", "grad_value"), FUSED_GRADS))
