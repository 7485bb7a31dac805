"""Every float16 instantiation of the attention kernels, and every launch shape the tuning keys can force, against a
float64 reference evaluated on exactly the values the kernels read; the deterministic mode, the temporal modules under
torch.autocast("cuda") (whose default dtype is float16) with a GradScaler step, and a performance guard.

Inputs are generated in fp32; value and grad_out are rounded to fp16 before both the kernel and the reference see them
(sampling locations, attention weights, offsets and logits stay fp32, as the kernels read them).  References: the
float64 PyTorch oracle (oracle/msda_torch.py for the drop-in op's shapes, oracle/temporal_torch.temporal_core_per_frame
for the whole-clip op, the fused op's prologue in float64 as in test_bf16_kernels_gpu.py).

Acceptance rule of an fp16 result (the output, and grad_value, which is accumulated in fp32 and rounded once):
  * every element:  |got - ref| <= 2^-11 |ref| + EPS max|ref|  (2^-11: fp16's unit roundoff; EPS covers the fp32
    accumulation and location arithmetic before the rounding, as in the bf16 file);
  * at most 1 % of the non-zero elements differ from round-to-nearest(ref).
The float results of an fp16 run meet the fp32 bars (normalised max error <= 1e-4).

The drop-in op keeps the reference's dtype dispatch in Python (MSDeformAttnFunction refuses float16), so its fp16
kernels are driven here through the C ABI directly.  Every case asserts which kernel family served it.
Setting DEVIS_TEST_ERROR_LOG=<file> appends the measured errors of every case to that file as JSON lines.
"""
import ctypes
import functools

import pytest
import torch

from conftest import nmax
from test_bf16_kernels_gpu import (FUSED_CASES, FUSED_FRAMES, FUSED_GRADS, FUSED_PC, FUSED_PT, FUSED_SAMPLING,
                                   FUSED_SHAPES, LAUNCHES, LQ_LARGE, LQ_MID, LQ_SMALL, _expect, _fused_inputs,
                                   _fused_run, _launches, _mode, _record, knobs)  # noqa: F401  (knobs: fixture)

pytestmark = pytest.mark.gpu

U_F16 = 2.0 ** -11          # unit roundoff of float16 (11-bit significand)
# measured on an NVIDIA B200 (1000 W power limit) over every case of this file: EPS 3.3e-7 at most, rn mismatch 0.4 %
EPS = 2e-6
MAX_RN_MISMATCH = 0.01
TOL_F32_OUT, TOL_F32_GRAD = 1e-5, 1e-4
F16 = torch.float16


def _f16_errors(got, ref):
    assert got.dtype == F16, got.dtype
    g = got.detach().double().cpu()
    r = ref.detach().double().cpu()
    assert torch.isfinite(r).all() and torch.isfinite(g).all()
    scale = max(r.abs().max().item(), 1e-30)
    eps = ((g - r).abs() - U_F16 * r.abs()).clamp_min(0).max().item() / scale
    nz = r != 0
    rn = r.to(F16).double()
    mismatch = (g[nz] != rn[nz]).double().mean().item() if nz.any() else 0.0
    return eps, mismatch


def _check(case, got, ref, f16_names):
    """f16_names: results held to the fp16 rule; every other name of `ref` to the fp32 bars"""
    errs, bad = {}, []
    for name, want in ref.items():
        if name in f16_names:
            eps, mismatch = _f16_errors(got[name], want)
            errs[name + ".eps"], errs[name + ".rn_mismatch"] = eps, mismatch
            if not (eps <= EPS and mismatch <= MAX_RN_MISMATCH):
                bad.append(name)
        else:
            t = TOL_F32_OUT if name.startswith(("loc_", "aw_")) else TOL_F32_GRAD
            e = nmax(got[name].detach().double().cpu().numpy(), want.detach().double().cpu().numpy())
            errs[name + ".nmax"] = e
            if not e <= t:
                bad.append(name)
    _record(case, errs)
    assert not bad, (bad, errs)


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


# ---- drop-in op through the C ABI (DeviceLevels kernels) ----------------------------------------------------------------
DROPIN = {
    # msda_fwd8v_kernel<F16, QPG, DeviceLevels, 512>, msda_bwd_kernel<F16, 8, QPG, DeviceLevels>
    "d32p4m8": dict(d=32, m=8, p=4, grouped=True),
    # msda_fwd8v_kernel<F16, QPG, DeviceLevels, 0> (row size at run time)
    "d32p4m3": dict(d=32, m=3, p=4, grouped=True),
    # P % 4 != 0: msda_fwd_kernel<F16, 8, QPG>, msda_bwd_kernel<F16, 8, QPG>
    "d32p3": dict(d=32, m=8, p=3, grouped=True),
    # msda_fwd_kernel<F16, 4, QPG>, msda_bwd_kernel<F16, 4, QPG>
    "d16": dict(d=16, m=8, p=4, grouped=True),
    # msda_fwd_generic_kernel<__half>, msda_bwd_generic_kernel<__half>
    "d30": dict(d=30, m=4, p=4, grouped=False),
}
DROPIN_SHAPES = ((9, 13), (5, 7), (3, 4))
DROPIN_BATCH = 2
# a pixel of batch 0, level 0 that the "nan" variant makes non-finite after moving every tap whose footprint holds it
NAN_PIXEL = (4, 6)


def _dropin_params():
    for name, cfg in DROPIN.items():
        for mode in ("default", "deterministic"):
            for launch, lq in LAUNCHES:
                if launch is not None and not cfg["grouped"]:
                    continue
                tag = "auto" if launch is None else f"t{launch[0]}q{launch[1]}"
                yield pytest.param(name, mode, launch, lq, "", id=f"{name}-{mode}-{tag}-lq{lq}")
    for name in ("d32p4m8", "d16", "d30"):
        for special in ("big", "nan"):
            yield pytest.param(name, "default", None, LQ_MID, special, id=f"{name}-{special}")


@functools.lru_cache(maxsize=None)
def _dropin_case(name, lq, special=""):
    """CPU inputs (value / grad_out fp16, locations and weights fp32) and the float64 reference on them.
    special "big": a checkerboard of +-60000 over level 0 of batch 0, head 0 (within fp16 range, and so is every output);
    "nan": NAN_PIXEL of batch 0 is NaN in every head and no tap's footprint (live or clamped corners) holds it"""
    from devis_b200 import synthetic
    from oracle import msda_torch
    cfg = DROPIN[name]
    g = torch.Generator().manual_seed(3000 + 1000 * list(DROPIN).index(name) + lq)
    n, m, d, p, nl = DROPIN_BATCH, cfg["m"], cfg["d"], cfg["p"], len(DROPIN_SHAPES)
    s = sum(h * w for h, w in DROPIN_SHAPES)
    sizes = torch.tensor([[w, h] for h, w in DROPIN_SHAPES], dtype=torch.float32)
    loc = torch.rand(n, lq, m, nl, p, 2, generator=g) * 1.2 - 0.1
    h0w, w0w = DROPIN_SHAPES[0]
    if special == "nan":
        px = torch.floor(loc[0, :, :, 0, :, 0] * w0w - 0.5)
        py = torch.floor(loc[0, :, :, 0, :, 1] * h0w - 0.5)
        hit = ((py == NAN_PIXEL[0]) | (py == NAN_PIXEL[0] - 1)) & ((px == NAN_PIXEL[1]) | (px == NAN_PIXEL[1] - 1))
        loc[0, :, :, 0, :, 0][hit] = 1.3 / w0w          # cell (1, 1): far from NAN_PIXEL
        loc[0, :, :, 0, :, 1][hit] = 1.3 / h0w
    loc = synthetic.make_boundary_safe(loc, sizes).contiguous()
    aw = torch.softmax(torch.randn(n, lq, m, nl * p, generator=g), -1).view(n, lq, m, nl, p).contiguous()
    value = torch.randn(n, s, m, d, generator=g)
    if special == "big":
        sign = (torch.arange(h0w * w0w) % 2) * 2 - 1
        value[0, :h0w * w0w, 0, :] = 60000.0 * sign[:, None].float()
    value = value.to(F16)
    gout = torch.randn(n, lq, m * d, generator=g).to(F16)
    vref = value.double()
    if special == "nan":
        value[0, NAN_PIXEL[0] * w0w + NAN_PIXEL[1]] = float("nan")
        # the oracle on the finite value is the reference wherever NAN_PIXEL is not read (nowhere, by construction);
        # its grad_value keeps the NaN pixel's entries, which no tap scatters to: zero
    out, gv, gl, ga = msda_torch.msda_forward_backward_torch(vref, torch.tensor(DROPIN_SHAPES), loc.double(), aw.double(),
                                                             gout.double())
    return (value, loc, aw, gout), {"out": out, "grad_value": gv, "grad_loc": gl, "grad_aw": ga}


def _dropin_run(inputs, deterministic):
    from devis_b200 import _lib
    lib = _lib.load()
    value, loc, aw, gout = (t.cuda() for t in inputs)
    n, s, m, d = value.shape
    lq, nl, p = loc.shape[1], loc.shape[3], loc.shape[4]
    shapes = torch.tensor(DROPIN_SHAPES, device="cuda")
    areas = shapes.prod(1)
    lsi = torch.cat([areas.new_zeros(1), areas.cumsum(0)[:-1]])
    out = torch.empty(n, lq, m * d, dtype=F16, device="cuda")
    gv = torch.empty(value.shape, dtype=torch.float32, device="cuda")
    gl, ga = torch.empty_like(loc), torch.empty_like(aw)
    flags = _lib.FLAG_DETERMINISTIC if deterministic else 0
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.devis_msda_forward(_ptr(value), _ptr(shapes), _ptr(lsi), _ptr(loc), _ptr(aw), _ptr(out),
                                      n, s, m, d, nl, lq, p, 64, _lib.F16, stream))
    ws_bytes = lib.devis_msda_backward_workspace_bytes(n, s, m, d, nl, lq, p, _lib.F16, flags)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda") if ws_bytes else None
    _lib.check(lib.devis_msda_backward(_ptr(value), _ptr(shapes), _ptr(lsi), _ptr(loc), _ptr(aw), _ptr(gout), _ptr(gv),
                                       _ptr(gl), _ptr(ga), n, s, m, d, nl, lq, p, 64, _lib.F16, flags, _ptr(ws),
                                       ctypes.c_size_t(ws_bytes), stream))
    return {"out": out, "grad_value": gv.to(F16), "grad_loc": gl, "grad_aw": ga}


@pytest.mark.parametrize("name,mode,launch,lq,special", list(_dropin_params()))
def test_dropin_kernels_f16_against_float64(knobs, name, mode, launch, lq, special):
    """devis_msda_forward / backward with DEVIS_MSDA_F16 at every shape of DROPIN, default and deterministic mode, at the
    heuristic's launch shape in each Lq band and at every forced (threads, QPG); plus a +-60000 value in live corners and
    a non-finite pixel that no tap reads"""
    cfg = DROPIN[name]
    inputs, ref = _dropin_case(name, lq, special)
    if launch is not None:
        t, q = launch
        knobs(k0=t, k1=q, k2=t, k3=q)
    with _launches() as delta:
        got = _dropin_run(inputs, mode == "deterministic")
    if cfg["grouped"]:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    else:
        _expect(delta, FWD_GENERIC=1, BWD_GENERIC=1)
    _check(f"f16-dropin-{name}-{mode}-{launch}-{lq}-{special}", got, ref, ("out", "grad_value"))


# ---- whole-clip op (TemporalMSDeformAttnFunction, ClipTable kernels) ----------------------------------------------------
CLIP_SHAPES = ((12, 16), (6, 8), (3, 4), (2, 2))
CLIP_FRAMES = 3
CLIP_NAMES = ("value", "loc_curr", "aw_curr", "loc_temporal", "aw_temporal")
CLIP = {
    # encoder form with a tile order: msda_fwd8v_kernel<F16, QPG, ClipTable, 512>, msda_bwd_kernel<F16, 8, QPG, ClipTable>,
    # deterministic: msda_bwds_kernel<F16, true>
    "d32p4m8": dict(d=32, m=8, pc=4, pt=4, grouped=True),
    "d32p4m3": dict(d=32, m=3, pc=4, pt=4, grouped=True),       # msda_fwd8v_kernel<F16, QPG, ClipTable, 0>
    "d32p2": dict(d=32, m=8, pc=4, pt=2, grouped=True),         # msda_fwd_kernel<F16, 8, QPG, ClipTable>
    "d16": dict(d=16, m=8, pc=4, pt=4, grouped=True),           # msda_fwd_kernel<F16, 4, QPG, ClipTable>
    "d30": dict(d=30, m=4, pc=4, pt=3, grouped=False),          # msda_{fwd,bwd}_generic_kernel<__half, ClipTable>
}
# (threads, QPG) forced through keys 0-3: every QPG the ClipTable kernels are instantiated with
CLIP_FORCED = ((64, 1), (128, 2), (256, 4), (32, 4))


def _clip_params():
    for name, cfg in CLIP.items():
        for mode in ("default", "deterministic"):
            runs = [(None, None), (None, LQ_SMALL), (None, LQ_LARGE)]
            if cfg["grouped"]:
                runs += [(f, None) for f in CLIP_FORCED]
            for launch, queries in runs:
                tag = "auto" if launch is None else f"t{launch[0]}q{launch[1]}"
                yield pytest.param(name, mode, launch, queries, id=f"{name}-{mode}-{tag}-q{queries or 'enc'}")


@functools.lru_cache(maxsize=None)
def _clip_case(name, queries):
    from devis_b200 import synthetic
    from oracle import temporal_torch
    cfg = CLIP[name]
    clip = synthetic.make_clip(n_frames=CLIP_FRAMES, shapes=CLIP_SHAPES, heads=cfg["m"], channels=cfg["d"], pc=cfg["pc"],
                               pt=cfg["pt"], queries=queries, dist="local", seed=40 + list(CLIP).index(name),
                               dtype=F16, device="cpu")
    leaves = [clip[k].double().requires_grad_(True) for k in CLIP_NAMES]
    offs = [torch.tensor([f - t for f in row]) for t, row in enumerate(clip["frame_table"])]
    out = temporal_torch.temporal_core_per_frame(*leaves, torch.tensor(CLIP_SHAPES), offs)
    out.backward(clip["grad_out"].double())
    ref = {"out": out.detach()}
    ref.update({"grad_" + k: x.grad for k, x in zip(CLIP_NAMES, leaves)})
    return clip, ref


def _clip_run(clip, order):
    from devis_b200 import clip_geometry, temporal_ms_deform_attn
    geom = clip_geometry.ClipGeometry(CLIP_SHAPES, CLIP_FRAMES, clip["frame_table"])
    q_order = geom.tile_order("cuda") if order else None
    leaves = [clip[k].cuda().requires_grad_(True) for k in CLIP_NAMES]
    out = temporal_ms_deform_attn(*leaves, geom, q_order)
    out.backward(clip["grad_out"].cuda())
    got = {"out": out.detach()}
    got.update({"grad_" + k: x.grad for k, x in zip(CLIP_NAMES, leaves)})
    return got


@pytest.mark.parametrize("name,mode,launch,queries", list(_clip_params()))
def test_whole_clip_op_f16_against_float64(knobs, name, mode, launch, queries):
    """temporal_ms_deform_attn on an fp16 clip: encoder form (one query per pixel, tile order for the D = 32, P = 4
    shapes: its deterministic backward is the sorted kernel) or decoder form with Lq in the small and large bands"""
    cfg = CLIP[name]
    clip, ref = _clip_case(name, queries)
    order = queries is None and cfg["grouped"] and cfg["pt"] % 4 == 0 and cfg["pc"] % 4 == 0 and cfg["d"] == 32
    if launch is not None:
        t, q = launch
        knobs(k0=t, k1=q, k2=t, k3=q)
    with _mode(mode), _launches() as delta:
        got = _clip_run(clip, order)
    assert got["out"].dtype == F16 and got["grad_value"].dtype == F16 and got["grad_loc_curr"].dtype == torch.float32
    if not cfg["grouped"]:
        _expect(delta, FWD_GENERIC=1, BWD_GENERIC=1)
    elif mode == "deterministic" and order:
        _expect(delta, FWD_GROUPED=1, BWD_SORTED=1)
    else:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    _check(f"f16-clip-{name}-{mode}-{launch}-{queries}", got, ref, ("out", "grad_value"))


def test_whole_clip_op_f16_above_2gib(knobs):
    """value of 3 GiB (2 frames x 3 x 2^20 pixels x 8 heads x 32 fp16 channels): the dead-corner kernels' signed
    32-bit offsets do not reach, so msda_fwd_kernel<F16, 8> / msda_bwd_kernel<F16, 8> serve it with unsigned ones;
    half of the taps read rows above the 2 GiB mark.  The reference runs on the 64 right-most columns the taps touch
    (W = 2^20: locations on a 1/16-pixel grid are exact in fp32, so the kernel's coordinates equal the reference's)."""
    from devis_b200 import clip_geometry, temporal_ms_deform_attn
    from oracle import temporal_torch
    T, H, W, M, D, LQ, P, WC = 2, 3, 1 << 20, 8, 32, 64, 4, 64
    assert T * H * W * M * D * 2 > (1 << 31)
    g = torch.Generator().manual_seed(77)

    def locs(n_slots):
        # pixel x in crop coordinates on a 1/16 grid, away from the crop's left edge, some right corners off the map
        k = torch.randint(16 * 2, 16 * WC, (T, LQ, M, n_slots, P), generator=g)
        k = k + (k % 16 == 8).long()                     # x_im never on a cell border
        x_crop = k.double() / 16.0                       # = x_im + 0.5 in crop pixels
        y_im = torch.rand(T, LQ, M, n_slots, P, generator=g, dtype=torch.float64) * 2.6 - 0.8
        y_im = torch.floor(y_im) + (y_im - torch.floor(y_im)).clamp(0.05, 0.95)
        x_full = ((x_crop + (W - WC)) / W).float()       # exact: (k + 16 (W - WC)) / 2^24
        y = ((y_im + 0.5) / H).float()
        crop = torch.stack([x_crop / WC, y.double()], -1)
        return torch.stack([x_full, y], -1).contiguous(), crop

    lc, lc_crop = locs(1)
    lt, lt_crop = locs(1)
    aw = torch.softmax(torch.randn(T, LQ, M, 2 * P, generator=g), -1)
    ac, at = aw[..., :P].reshape(T, LQ, M, 1, P).contiguous(), aw[..., P:].reshape(T, LQ, M, 1, P).contiguous()
    crop = torch.randn(T, H, WC, M, D, generator=g).to(F16)
    gout = torch.randn(T, LQ, M * D, generator=g).to(F16)

    value = torch.randn(T, H, W, M, D, device="cuda", dtype=F16)
    value[:, :, W - WC:] = crop.cuda()
    value = value.view(T, H * W, M, D).detach().requires_grad_(True)
    geom = clip_geometry.ClipGeometry(((H, W),), T, [[1], [0]])
    leaves = [x.cuda().requires_grad_(True) for x in (lc, ac, lt, at)]
    with _launches() as delta:
        out = temporal_ms_deform_attn(value, *leaves, geom, None)
        out.backward(gout.cuda())
    _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    gv = value.grad.view(T, H, W, M, D)
    got = {"out": out.detach(), "grad_value": gv[:, :, W - WC:].reshape(T, H * WC, M, D).clone()}
    got.update({k: x.grad for k, x in zip(("grad_loc_curr", "grad_aw_curr", "grad_loc_temporal", "grad_aw_temporal"),
                                           leaves)})
    assert gv[:, :, :W - WC].abs().sum().item() == 0           # nothing scattered outside the sampled columns
    del value, gv

    rl = [x.requires_grad_(True) for x in (crop.double().view(T, H * WC, M, D), lc_crop, ac.double(), lt_crop,
                                           at.double())]
    ref_out = temporal_torch.temporal_core_per_frame(*rl, torch.tensor([[H, WC]]), [torch.tensor([1]), torch.tensor([-1])])
    ref_out.backward(gout.double())
    ref = {"out": ref_out.detach(), "grad_value": rl[0].grad, "grad_aw_curr": rl[2].grad, "grad_aw_temporal": rl[4].grad}
    # x_crop = (x W - (W - WC)) / WC, so d/d(x) on the full map is W / WC times d/d(x_crop)
    for name, i in (("grad_loc_curr", 1), ("grad_loc_temporal", 3)):
        gr = rl[i].grad.clone()
        gr[..., 0] *= W / WC
        ref[name] = gr
    _check("f16-clip-above-2gib", got, ref, ("out", "grad_value"))


# ---- fused op (TemporalMSDeformAttnFusedFunction) -----------------------------------------------------------------------
def _fused_params():
    for name in FUSED_CASES:
        for mode in ("default", "deterministic"):
            threads = (None,) if mode != "default" else (None, 32, 64, 128, 256)
            for t in threads:
                yield pytest.param(name, mode, t, id=f"{name}-{mode}-" + ("auto" if t is None else f"fwd{t}"))


@functools.lru_cache(maxsize=None)
def _fused_case(name):
    return _fused_inputs(FUSED_CASES[name], F16, FUSED_SHAPES, FUSED_FRAMES, FUSED_PC, FUSED_PT,
                         seed=900 + list(FUSED_CASES).index(name))


@pytest.mark.parametrize("name,mode,fwd_threads", list(_fused_params()))
def test_fused_op_f16_against_float64(knobs, name, mode, fwd_threads):
    """fused op on an fp16 clip: encoder form -> tmsda_fused_fwd8_kernel<F16, 512 | 0>, tmsda_fused_bwd_kernel<F16, false,
    false, DET>; general form (boxes, TREF_OWN / TREF_SAMPLED, by-products, reference points with grad outside the
    deterministic mode) -> tmsda_fused_fwd_kernel<F16, 1, true, 512>, tmsda_fused_bwd_kernel<F16, false, true, DET>"""
    from devis_b200 import _lib
    cfg = FUSED_CASES[name]
    x, ref = _fused_case(name)
    general = cfg["form"] == "box"
    tref = {"own": _lib.TREF_OWN, "sampled": _lib.TREF_SAMPLED}.get(cfg.get("tref"), _lib.TREF_LEVEL0)
    ref_grad = general and mode == "default"
    order = x["geom"].tile_order("cuda") if not general else None
    if fwd_threads is not None:
        knobs(k0=fwd_threads)
    with _mode(mode), _launches() as delta:
        got = _fused_run(x, ref_grad=ref_grad, want_sampling=general, tref=tref, order=order)
    _expect(delta, FUSED_FWD=1, FUSED_BWD=1)
    assert got["out"].dtype == F16 and got["grad_value"].dtype == F16
    f32 = FUSED_GRADS + (("grad_ref",) if ref_grad else ()) + (FUSED_SAMPLING if general else ())
    want = {k: ref[k] for k in ("out", "grad_value") + f32}
    _check(f"f16-fused-{name}-{mode}-{fwd_threads}", got, want, ("out", "grad_value"))


# ---- deterministic mode -------------------------------------------------------------------------------------------------
def _aux_launches():
    from devis_b200 import _lib
    return _lib.kernel_launches(_lib.KERNEL_AUX)


@pytest.mark.parametrize("form", ["clip_encoder", "clip_decoder", "fused"])
def test_deterministic_mode_is_bit_reproducible_for_f16(form):
    """torch.use_deterministic_algorithms(True): two runs give the same bits (the fixed-point helpers ran), and the
    results are those of the default mode up to the order of the float sums of grad_value"""
    if form == "fused":
        x, _ = _fused_case("enc_m8")
        run = lambda: _fused_run(x, order=x["geom"].tile_order("cuda"))
    else:
        clip, _ = _clip_case("d32p4m8", None if form == "clip_encoder" else LQ_MID)
        run = lambda: _clip_run(clip, form == "clip_encoder")
    base = run()
    torch.use_deterministic_algorithms(True)
    try:
        aux = _aux_launches()
        with _launches() as delta:
            a = run()
        assert _aux_launches() > aux, "the fixed-point helpers did not run"
        if form == "clip_encoder":
            assert delta["KERNEL_BWD_SORTED"] == 1
        b = run()
    finally:
        torch.use_deterministic_algorithms(False)
    for k in a:
        assert torch.equal(a[k], b[k]), k
        if k == "grad_value":
            d = (a[k].double() - base[k].double()).abs()
            assert (d <= 2 * U_F16 * base[k].double().abs() + 1e-6 * base[k].double().abs().max()).all()
        else:
            assert nmax(a[k].double().cpu().numpy(), base[k].double().cpu().numpy()) < 1e-5, k


# ---- modules under torch.autocast("cuda") -------------------------------------------------------------------------------
# bound of |module output / input gradient - fp32 run| / max|fp32 run| under fp16 autocast.  Measured on an NVIDIA B200
# (1000 W power limit): 2.2e-3 at most over the module cases (the unfused decoder's value-input gradient), 3.5e-4 for the
# GradScaler step's parameter gradients; the bf16 autocast test allows 4e-2 (test_transformer_gpu.py).
TOL_AUTOCAST = 1e-2


def _pyramid(shapes_l, T, device="cuda"):
    from devis_b200 import synthetic
    shapes = torch.tensor(shapes_l, device=device)
    lsi = torch.tensor(synthetic.level_start_index(shapes_l), device=device)
    tshapes = shapes.repeat(T - 1, 1)
    tlsi = torch.cat([tshapes.new_zeros(1), tshapes.prod(1).cumsum(0)[:-1]])
    offsets = [torch.tensor([d for d in range(-t, T - t) if d != 0], device=device) for t in range(T)]
    return (shapes, tshapes), (lsi, tlsi), offsets


def _compare(case, got, want):
    errs = {}
    for i, (g_, w_) in enumerate(zip(got, want)):
        errs[str(i)] = nmax(g_.detach().float().cpu().numpy(), w_.detach().float().cpu().numpy())
    _record(case, errs)
    assert all(v < TOL_AUTOCAST for v in errs.values()), errs


@pytest.mark.parametrize("fused", [True, False])
def test_temporal_encoder_under_f16_autocast(fused):
    from devis_b200 import TemporalMSDeformAttnEncoder, synthetic
    torch.manual_seed(0)
    T, shapes_l = 3, ((18, 30), (9, 15))
    S = sum(h * w for h, w in shapes_l)
    enc = TemporalMSDeformAttnEncoder(n_frames=T, d_model=256, n_levels=2, t_window=T - 1, n_heads=8, n_curr_points=4,
                                      n_temporal_points=4).cuda()
    with torch.no_grad():
        for lin in (enc.attention_weights, enc.temporal_attention_weights):
            lin.weight.normal_(0, 0.05)
    query, inp = torch.randn(T, S, 256, device="cuda"), torch.randn(T, S, 256, device="cuda")
    ref = synthetic.pixel_reference_points(shapes_l, T, "cuda")
    shapes, lsi, offsets = _pyramid(shapes_l, T)
    gout = torch.randn(T, S, 256, device="cuda")

    def run(amp):
        enc.fuse_prologue = fused
        enc.zero_grad(set_to_none=True)
        q, x = query.clone().requires_grad_(True), inp.clone().requires_grad_(True)
        with torch.autocast("cuda", enabled=amp):
            out, _ = enc(q, ref, x, shapes, lsi, offsets)
        assert out.dtype == (F16 if amp else torch.float32)
        out.float().backward(gout)
        return out.detach().float(), q.grad, x.grad

    want = run(False)
    with _launches() as delta:
        got = run(True)
    if fused:
        _expect(delta, FUSED_FWD=1, FUSED_BWD=1)
    else:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    _compare(f"autocast-encoder-fused{fused}", got, want)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("instance_aware", [True, False])
def test_temporal_decoder_under_f16_autocast(fused, ref_dim, instance_aware):
    """decoder module, 2-d or box reference points, instance-aware on / off: output, the 5-tuple's locations and
    weights, and the gradients of query, value input and reference points within bounds of the fp32 run"""
    from devis_b200 import TemporalMSDeformAttnDecoder
    torch.manual_seed(1)
    T, shapes_l, q = 3, ((18, 30), (9, 15)), 30
    S = sum(h * w for h, w in shapes_l)
    dec = TemporalMSDeformAttnDecoder(n_frames=T, d_model=256, n_levels=2, t_window=T - 1, n_heads=8, n_curr_points=4,
                                      n_temporal_points=4, dec_instance_aware_att=instance_aware).cuda()
    with torch.no_grad():
        for lin in (dec.attention_weights, dec.temporal_attention_weights):
            lin.weight.normal_(0, 0.05)
    query, inp = torch.randn(1, T * q, 256, device="cuda"), torch.randn(T, S, 256, device="cuda")
    xy = torch.rand(1, T * q, 1, 2, device="cuda") * 0.8 + 0.1
    ref = xy.expand(-1, -1, 2, -1)
    if ref_dim == 4:
        ref = torch.cat([ref, torch.rand(1, T * q, 2, 2, device="cuda") * 0.3 + 0.1], -1)
    ref = ref.contiguous()
    shapes, lsi, offsets = _pyramid(shapes_l, T)
    gout = torch.randn(1, T * q, 256, device="cuda")

    def run(amp):
        dec.fuse_prologue = fused
        dec.zero_grad(set_to_none=True)
        qq, x = query.clone().requires_grad_(True), inp.clone().requires_grad_(True)
        r = ref.clone().requires_grad_(True)
        with torch.autocast("cuda", enabled=amp):
            out, lc, lt, awc, awt = dec(qq, r, x, shapes, lsi, offsets)
        assert out.dtype == (F16 if amp else torch.float32) and len(lc) == T and len(lt) == T
        out.float().backward(gout)
        return (out.detach().float(), torch.stack(lc).detach(), torch.stack(lt).detach(), awc.detach(), awt.detach(),
                qq.grad, x.grad, r.grad)

    want = run(False)
    with _launches() as delta:
        got = run(True)
    if fused:
        _expect(delta, FUSED_FWD=1, FUSED_BWD=1)
    else:
        _expect(delta, FWD_GROUPED=1, BWD_GROUPED=1)
    _compare(f"autocast-decoder-fused{fused}-ref{ref_dim}-ia{instance_aware}", got, want)


def test_gradscaler_step_of_a_small_transformer():
    """one torch.amp.GradScaler step of a DeVISTransformer (1 encoder + 1 decoder layer, D = 32 per head: the fused
    kernels) under fp16 autocast: finite gradients, within bounds of the fp32 step after unscale_"""
    from devis_b200 import DeVISTransformer
    torch.manual_seed(2)
    T, shapes_l, C, nq = 3, ((16, 24), (8, 12)), 256, 10
    tr = DeVISTransformer(d_model=C, num_frames=T, num_encoder_layers=1, num_decoder_layers=1, dim_feedforward=512,
                          dropout=0.0, num_feature_levels=2, enc_n_temporal_points=4, dec_n_temporal_points=4).cuda()
    query_embed = torch.nn.Embedding(T * nq, 2 * C).cuda()
    params = list(tr.parameters()) + list(query_embed.parameters())
    srcs = [torch.randn(T, C, h, w, device="cuda") for h, w in shapes_l]
    pos = [torch.randn(T, C, h, w, device="cuda") for h, w in shapes_l]
    masks = [torch.zeros(T, h, w, dtype=torch.bool, device="cuda") for h, w in shapes_l]

    def step(amp):
        for p in params:
            p.grad = None
        scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 12, enabled=amp)
        with torch.autocast("cuda", enabled=amp):
            hs, _, memories, *_ = tr(srcs, masks, pos, query_embed.weight)
            loss = hs[-1].float().square().mean() + 1e-3 * sum(m.float().square().mean() for m in memories)
        opt = torch.optim.SGD(params, lr=0.0)
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        grads = torch.cat([p.grad.flatten() for p in params if p.grad is not None])
        scaler.step(opt)
        scaler.update()
        return grads

    want = step(False)
    with _launches() as delta:
        got = step(True)
    assert delta["KERNEL_FUSED_FWD"] >= 2 and delta["KERNEL_FUSED_BWD"] >= 2
    assert torch.isfinite(got).all()
    err = nmax(got.cpu().numpy(), want.cpu().numpy())
    _record("autocast-gradscaler-step", {"grads.nmax": err})
    assert err < TOL_AUTOCAST, err


# ---- performance guard --------------------------------------------------------------------------------------------------
def test_f16_whole_clip_kernels_meet_the_bf16_bounds():
    """the DeVIS layer-clip forward / backward in fp16 against the bf16 bounds of test_perf_guard_gpu.py"""
    if torch.cuda.get_device_properties(0).multi_processor_count < 140:
        pytest.skip("bounds are B200 numbers")
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from benchmarks.sweep import RawClip
    from devis_b200 import clip_geometry, synthetic
    from test_perf_guard_gpu import _median_us
    clip = synthetic.make_clip(device="cuda", dtype=F16, dist="local")
    geom = clip_geometry.ClipGeometry(clip["shapes"], 6, clip["frame_table"])
    rc = RawClip(clip, geom.tile_order("cuda"))
    fwd, bwd = _median_us(rc.fwd), _median_us(rc.bwd)
    assert fwd < 540.0, f"fp16 forward {fwd:.0f} us"
    assert bwd < 2080.0, f"fp16 backward {bwd:.0f} us"
