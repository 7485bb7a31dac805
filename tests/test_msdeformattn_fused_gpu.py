"""MSDeformAttn on the fused-prologue kernels, with the input padding mask applied inside them (D = 32, M = 8, L = 4,
P = 4: the Deformable-DETR head layout, which is what selects the fused path).

  * module level: fused float32 (and bfloat16) MSDeformAttn against the same module in float64 on the unfused path --
    the path the mod_msda_* goldens pin -- for no mask, DETR-style rectangular masks, random masks and a fully masked
    image; 2-d reference points (encoder, Lq = S, and decoder) and boxes (decoder, Lq = 300); N = 1, 2, 3.  Each case
    also asserts which kernel families ran.
  * op level: the masked fused call against value.masked_fill + the unmasked fused call, NaN / Inf in masked rows,
    and bit-identical deterministic backward runs with a mask.

Inputs of the module tests are dyadic where they reach the sampling locations (query, sampling_offsets, reference
points; power-of-two maps), so float32 and float64 form the very same locations and pick the same bilinear cells: the
comparison measures the kernels, not a floor() that flips between precisions.
"""
import pytest
import torch
import torch.nn.functional as F

from conftest import nmax

pytestmark = pytest.mark.gpu

D_MODEL, M, L, P = 256, 8, 4, 4
POW2 = ((16, 32), (8, 16), (4, 8), (2, 4))          # module tests: exact locations in float32 and float64
ODD = ((13, 21), (7, 11), (4, 6), (2, 3))           # op tests: both sides run the same float32 arithmetic


def _families():
    from devis_b200 import _lib
    return {k: _lib.kernel_launches(getattr(_lib, k)) for k in
            ("KERNEL_FWD_GROUPED", "KERNEL_FWD_GENERIC", "KERNEL_BWD_GROUPED", "KERNEL_BWD_GENERIC",
             "KERNEL_FUSED_FWD", "KERNEL_FUSED_BWD")}


def _delta(before):
    after = _families()
    return {k: after[k] - before[k] for k in after}


def _pyramid(shapes):
    from devis_b200 import clip_geometry
    return clip_geometry.pyramid_tensors(shapes, "cuda")


def detr_mask(n, shapes, valid):
    """Deformable DETR's mask: True on the padding of each image in the padded batch, resized to every level with
    nearest interpolation (models/backbone.py: F.interpolate(m[None].float(), size=x.shape[-2:]).to(torch.bool)[0])"""
    h0, w0 = shapes[0][0] * 8, shapes[0][1] * 8
    m = torch.ones(n, h0, w0, dtype=torch.bool, device="cuda")
    for i in range(n):
        fh, fw = valid[i % len(valid)]
        m[i, :max(1, round(h0 * fh)), :max(1, round(w0 * fw))] = False
    levels = [F.interpolate(m[None].float(), size=hw).to(torch.bool)[0].flatten(1) for hw in shapes]
    return torch.cat(levels, 1)


def make_mask(kind, n, shapes, gen):
    s = sum(h * w for h, w in shapes)
    if kind == "none":
        return None
    if kind == "detr":
        return detr_mask(n, shapes, [(1.0, 1.0), (0.75, 0.75), (0.5, 0.625)])
    if kind == "random":
        return (torch.rand(n, s, generator=gen) < 0.3).cuda()
    mask = torch.zeros(n, s, dtype=torch.bool)
    mask[0] = True                                   # one fully masked image
    return mask.cuda()


def _dyadic(shape, lo, hi, scale, gen):
    return torch.randint(lo, hi + 1, shape, generator=gen).double() / scale


def make_module_case(n, kind, seed, dtype):
    """module parameters, inputs and the grad of the output, in float64 on the CPU"""
    from devis_b200.modules import MSDeformAttn
    gen = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    mod = MSDeformAttn(D_MODEL, L, M, P).double()
    with torch.no_grad():
        mod.sampling_offsets.weight.copy_(_dyadic(mod.sampling_offsets.weight.shape, -2, 2, 256, gen))
        if dtype == torch.bfloat16:
            mod.sampling_offsets.weight.zero_()     # bf16 Linear outputs are exact only for few-bit sums
        mod.sampling_offsets.bias.copy_(_dyadic(mod.sampling_offsets.bias.shape, -12, 12, 4, gen))
        mod.attention_weights.weight.normal_(0, 0.05, generator=gen)
        mod.attention_weights.bias.normal_(0, 0.5, generator=gen)
        mod.value_proj.bias.normal_(0, 0.1, generator=gen)
        mod.output_proj.bias.normal_(0, 0.1, generator=gen)
    s = sum(h * w for h, w in POW2)
    lq = s if kind == "enc" else 300
    query = _dyadic((n, lq, D_MODEL), -4, 4, 8, gen)
    inp = torch.randn(n, s, D_MODEL, generator=gen, dtype=torch.float64)
    if kind == "box":
        ref = torch.cat([_dyadic((n, lq, L, 2), 32, 224, 256, gen), _dyadic((n, lq, L, 2), 16, 128, 256, gen)], -1)
    else:
        ref = _dyadic((n, lq, L, 2), 0, 255, 256, gen)
    gout = torch.randn(n, lq, D_MODEL, generator=gen, dtype=torch.float64)
    # both precisions start from the same numbers: everything rounded to the tested type once
    with torch.no_grad():
        for prm in mod.parameters():
            prm.copy_(prm.to(dtype).double())
    return mod, query, ref, inp.to(dtype).double(), gout.to(dtype).double()


def run_module(mod, query, ref, inp, gout, mask, dtype, fuse=True):
    import copy
    mod = copy.deepcopy(mod).to("cuda", dtype)
    mod.fuse_prologue = fuse
    shapes, lsi = _pyramid(POW2)
    q = query.to("cuda", dtype).requires_grad_(True)
    x = inp.to("cuda", dtype).requires_grad_(True)
    r = ref.to("cuda", torch.float64 if dtype == torch.float64 else torch.float32)
    before = _families()
    out, _ = mod(q, r, x, shapes, lsi, mask)
    out.backward(gout.to("cuda", dtype))
    torch.cuda.synchronize()
    grads = {"query": q.grad, "input_flatten": x.grad}
    grads.update({"param." + k: p.grad for k, p in mod.named_parameters()})
    return out.detach(), grads, _delta(before)


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("kind", ["enc", "dec", "box"])
@pytest.mark.parametrize("mask_kind", ["none", "detr", "random", "full_image"])
def test_fused_module_matches_float64_unfused(n, kind, mask_kind):
    mod, query, ref, inp, gout = make_module_case(n, kind, 100 * n + len(kind) + len(mask_kind), torch.float32)
    mask = make_mask(mask_kind, n, POW2, torch.Generator().manual_seed(n))
    want, want_g, d64 = run_module(mod, query, ref, inp, gout, mask, torch.float64)
    assert d64["KERNEL_FWD_GENERIC"] == 1 and d64["KERNEL_FUSED_FWD"] == 0, d64
    got, got_g, d32 = run_module(mod, query, ref, inp, gout, mask, torch.float32)
    assert d32["KERNEL_FUSED_FWD"] == 1 and d32["KERNEL_FUSED_BWD"] == 1, d32
    assert d32["KERNEL_FWD_GROUPED"] == d32["KERNEL_BWD_GROUPED"] == 0, d32
    assert nmax(got.cpu(), want.cpu()) <= 1e-5
    for k in want_g:
        assert nmax(got_g[k].cpu(), want_g[k].cpu()) <= 1e-4, k


@pytest.mark.parametrize("kind", ["enc", "box"])
@pytest.mark.parametrize("mask_kind", ["none", "detr"])
def test_fused_module_bf16_value(kind, mask_kind):
    n = 2
    mod, query, ref, inp, gout = make_module_case(n, kind, 7, torch.bfloat16)
    mask = make_mask(mask_kind, n, POW2, None)
    want, want_g, _ = run_module(mod, query, ref, inp, gout, mask, torch.float64)
    got, got_g, d = run_module(mod, query, ref, inp, gout, mask, torch.bfloat16)
    assert d["KERNEL_FUSED_FWD"] == 1 and d["KERNEL_FUSED_BWD"] == 1 and d["KERNEL_FWD_GROUPED"] == 0, d
    assert nmax(got.float().cpu(), want.cpu()) <= 1e-2
    for k in want_g:
        assert nmax(got_g[k].float().cpu(), want_g[k].cpu()) <= 1e-2, k


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fuse_prologue_off_keeps_the_unfused_kernels(dtype):
    mod, query, ref, inp, gout = make_module_case(2, "enc", 3, dtype)
    mask = make_mask("detr", 2, POW2, None)
    fused, fused_g, df = run_module(mod, query, ref, inp, gout, mask, dtype, fuse=True)
    plain, plain_g, dp = run_module(mod, query, ref, inp, gout, mask, dtype, fuse=False)
    assert df["KERNEL_FUSED_FWD"] == 1 and df["KERNEL_FWD_GROUPED"] == 0, df
    assert dp["KERNEL_FWD_GROUPED"] == 1 and dp["KERNEL_BWD_GROUPED"] == 1, dp
    assert dp["KERNEL_FUSED_FWD"] == dp["KERNEL_FUSED_BWD"] == 0, dp
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-5
    assert nmax(fused.float().cpu(), plain.float().cpu()) <= tol
    for k in plain_g:
        assert nmax(fused_g[k].float().cpu(), plain_g[k].float().cpu()) <= 10 * tol, k


def test_float16_module_still_raises():
    from devis_b200.modules import MSDeformAttn
    mod = MSDeformAttn(D_MODEL, L, M, P).cuda().half()
    shapes, lsi = _pyramid(POW2)
    s = sum(h * w for h, w in POW2)
    q = torch.randn(1, 10, D_MODEL, device="cuda", dtype=torch.float16)
    x = torch.randn(1, s, D_MODEL, device="cuda", dtype=torch.float16)
    with pytest.raises(RuntimeError, match="not implemented for 'torch.float16'"):
        mod(q, torch.rand(1, 10, L, 2, device="cuda"), x, shapes, lsi)


# ---- op level -----------------------------------------------------------------------------------------------------

def make_op_case(n, lq, ref_dim, dtype, seed):
    from devis_b200 import clip_geometry
    gen = torch.Generator().manual_seed(seed)
    s = sum(h * w for h, w in ODD)
    geom = clip_geometry.ClipGeometry(ODD, n, None)
    value = torch.randn(n, s, M, 32, generator=gen).to("cuda", dtype)
    if ref_dim == 2:
        ref = torch.rand(n, lq, L, 2, generator=gen)
    else:
        ref = torch.cat([torch.rand(n, lq, L, 2, generator=gen) * 0.8 + 0.1,
                         torch.rand(n, lq, L, 2, generator=gen) * 0.4 + 0.05], -1)
    off = torch.randn(n, lq, M, L, P, 2, generator=gen) * 3
    logit = torch.randn(n, lq, M, L * P, generator=gen)
    gout = torch.randn(n, lq, M * 32, generator=gen).to("cuda", dtype)
    order = geom.tile_order("cuda") if lq == s else None
    return geom, value, ref.cuda(), off.cuda(), logit.cuda(), gout, order


def run_op(geom, value, ref, off, logit, gout, order, mask):
    from devis_b200.functions import TemporalMSDeformAttnFusedFunction
    from devis_b200 import _lib
    v = value.clone().requires_grad_(True)
    o = off.clone().requires_grad_(True)
    lg = logit.clone().requires_grad_(True)
    out = TemporalMSDeformAttnFusedFunction.apply(v, ref, o, lg, None, None, geom, order, _lib.TREF_LEVEL0, False,
                                                  mask)
    out.backward(gout)
    torch.cuda.synchronize()
    return out.detach(), v.grad, o.grad, lg.grad


OP_CASES = [("enc", 2), ("dec", 2), ("dec", 4)]    # (queries, ref_dim): encoder Lq = S with the tile order


def _op_args(kind, ref_dim, dtype, n=2, seed=11):
    s = sum(h * w for h, w in ODD)
    return make_op_case(n, s if kind == "enc" else 300, ref_dim, dtype, seed)


@pytest.mark.parametrize("kind,ref_dim", OP_CASES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mask_kind", ["detr", "random", "full_image"])
def test_masked_op_equals_masked_fill(kind, ref_dim, dtype, mask_kind):
    geom, value, ref, off, logit, gout, order = _op_args(kind, ref_dim, dtype)
    mask = make_mask(mask_kind, 2, ODD, torch.Generator().manual_seed(5))
    got = run_op(geom, value, ref, off, logit, gout, order, mask)
    want = run_op(geom, value.masked_fill(mask[..., None, None], 0), ref, off, logit, gout, order, None)
    keep = ~mask[..., None, None]
    assert torch.equal(got[0], want[0])                                  # the same sums, the dropped terms were +0
    assert torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])  # d/d(offset), d/d(logit)
    assert torch.all(got[1][mask] == 0)                                   # masked rows receive no grad_value
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-6                      # float atomics: order only
    assert nmax(got[1].float().cpu(), (want[1] * keep).float().cpu()) <= tol


@pytest.mark.parametrize("kind,ref_dim", OP_CASES)
@pytest.mark.parametrize("mode", ["default", "deterministic"])
def test_nan_and_inf_in_masked_rows_change_nothing(kind, ref_dim, mode):
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    geom, value, ref, off, logit, gout, order = _op_args(kind, ref_dim, torch.float32, seed=13)
    mask = make_mask("random", 2, ODD, torch.Generator().manual_seed(6))
    clean = value.masked_fill(mask[..., None, None], 0)
    poison = clean.clone()
    rows = mask.nonzero()
    poison[rows[::2, 0], rows[::2, 1]] = float("nan")
    poison[rows[1::2, 0], rows[1::2, 1]] = float("inf")
    try:
        if mode == "deterministic":
            MSDA.set_deterministic(True)
        got = run_op(geom, poison, ref, off, logit, gout, order, mask)
        want = run_op(geom, clean, ref, off, logit, gout, order, mask)
    finally:
        MSDA.set_deterministic(False)
    for g, w in zip(got, want):
        assert torch.isfinite(g).all()
        if mode == "deterministic":
            assert torch.equal(g, w)
    if mode == "default":
        assert nmax(got[1].cpu(), want[1].cpu()) <= 1e-6                # float atomics: order only
    assert torch.equal(got[0], want[0]) and torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])
    assert torch.all(got[1][mask] == 0)


def make_exact_case(kind, ref_dim, seed):
    """Operands whose every grad_value partial sum is exact in bfloat16, in any order: power-of-two maps, taps on pixel
    centres (a single bilinear corner with factor 1), softmax weights 1/16 (equal logits), grad_output in {-1, 0, 1}
    and mostly 0.  Then the packed bf16 reductions of DEVIS_MSDA_FLAG_BF16_GRAD_VALUE add multiples of 1/16 and the
    result does not depend on their arrival order, so it can be compared bit for bit."""
    from devis_b200 import clip_geometry
    gen = torch.Generator().manual_seed(seed)
    n, s = 2, sum(h * w for h, w in POW2)
    lq = s if kind == "enc" else 300
    geom = clip_geometry.ClipGeometry(POW2, n, None)
    wh = torch.tensor([[w, h] for h, w in POW2], dtype=torch.float64)                   # (L, 2) as (W, H)
    cell = torch.floor(torch.rand(n, lq, L, 2, generator=gen, dtype=torch.float64) * wh)
    xy = (cell + 0.5) / wh                                                              # pixel centres
    step = torch.randint(-2, 3, (n, lq, M, L, P, 2), generator=gen).double()
    if ref_dim == 2:
        ref, off = xy, step                                 # loc = ref + off / (W, H): whole pixels
    else:
        ref = torch.cat([xy, (2.0 / wh).expand(n, lq, L, 2)], -1)
        off = 4 * step                                      # loc = ref.xy + off / 4 * wh / 2 = ref.xy + step / (W, H)
    value = torch.randn(n, s, M, 32, generator=gen).to("cuda", torch.bfloat16)
    logit = torch.zeros(n, lq, M, L * P)
    gout = torch.randint(-1, 2, (n, lq, M * 32), generator=gen) * (torch.rand(n, lq, M * 32, generator=gen) < 0.125)
    order = geom.tile_order("cuda") if lq == s else None
    return (geom, value, ref.float().cuda(), off.float().cuda(), logit.cuda(), gout.to("cuda", torch.bfloat16),
            order)


@pytest.mark.parametrize("kind,ref_dim", OP_CASES)
def test_nan_and_inf_in_masked_rows_with_bf16_grad_value_accumulation(kind, ref_dim):
    """the MASK kernels of the packed bf16 grad_value reductions: on operands where bf16 accumulation is exact, the
    poisoned masked call, the clean masked call and the float-accumulated clean call agree bit for bit"""
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    geom, value, ref, off, logit, gout, order = make_exact_case(kind, ref_dim, 19)
    mask = make_mask("random", 2, POW2, torch.Generator().manual_seed(7))
    clean = value.masked_fill(mask[..., None, None], 0)
    poison = clean.clone()
    rows = mask.nonzero()
    poison[rows[::2, 0], rows[::2, 1]] = float("nan")
    poison[rows[1::2, 0], rows[1::2, 1]] = float("inf")
    # precondition of exactness: sum_k |contribution_k| <= 16 for every element (the weights are >= 0, so this is
    # grad_value for |grad_output|), i.e. every partial sum is a multiple of 1/16 of at most 8 significant bits
    bound = run_op(geom, clean, ref, off, logit, gout.abs(), order, mask)[1]
    assert 0 < float(bound.float().max()) <= 15          # (15: margin for the bf16 rounding of the bound itself)
    exact = run_op(geom, clean, ref, off, logit, gout, order, mask)              # float32 accumulation
    try:
        MSDA.set_bf16_grad_value_accumulation(True)
        got = run_op(geom, poison, ref, off, logit, gout, order, mask)
        want = run_op(geom, clean, ref, off, logit, gout, order, mask)
    finally:
        MSDA.set_bf16_grad_value_accumulation(False)
    for g, w in zip(got, want):
        assert torch.isfinite(g).all()
        assert torch.equal(g, w)
    assert torch.equal(got[1], exact[1])
    assert torch.all(got[1][mask] == 0)


@pytest.mark.parametrize("kind,ref_dim", OP_CASES)
def test_deterministic_masked_backward_is_bit_identical(kind, ref_dim):
    geom, value, ref, off, logit, gout, order = _op_args(kind, ref_dim, torch.float32, seed=17)
    mask = make_mask("detr", 2, ODD, None)
    torch.use_deterministic_algorithms(True)
    try:
        a = run_op(geom, value, ref, off, logit, gout, order, mask)
        b = run_op(geom, value, ref, off, logit, gout, order, mask)
    finally:
        torch.use_deterministic_algorithms(False)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert torch.all(a[1][mask] == 0)
