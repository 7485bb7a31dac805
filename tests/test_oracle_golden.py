"""Pins oracle/ (the CPU restatements) against fixtures produced by the reference's own code
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import load_golden, nmax
from oracle import c_oracle, msda_torch, temporal_torch

OP_CASES = ["op_testpy", "op_ragged", "op_d32", "op_d1", "op_d30", "op_d71", "op_border"]
# op_testpy uses torch.rand locations (test.py:32); its taps are not kept away from cell borders,
# but in float64 both coordinate formulas agree on the cell for this seed.


@pytest.mark.parametrize("name", OP_CASES)
def test_c_oracle_f64_matches_reference_pytorch_core(name):
    g = load_golden(name)
    out = c_oracle.forward(g["value"], g["shapes"], g["lsi"], g["loc"], g["aw"])
    assert nmax(out, g["out"]) < 1e-12
    gv, gl, ga = c_oracle.backward(g["value"], g["shapes"], g["lsi"], g["loc"], g["aw"], g["gout"])
    assert nmax(gv, g["gvalue"]) < 1e-12
    assert nmax(gl, g["gloc"]) < 1e-11
    assert nmax(ga, g["gaw"]) < 1e-12


@pytest.mark.parametrize("name", [n for n in OP_CASES if n != "op_testpy"])
def test_c_oracle_f32_within_north_star_tolerance(name):
    """fp32 restatement vs fp64 reference on boundary-safe taps: fwd 1e-5, grads 1e-4."""
    g = load_golden(name)
    f = lambda k: g[k].astype(np.float32)
    out = c_oracle.forward(f("value"), g["shapes"], g["lsi"], f("loc"), f("aw"))
    assert nmax(out, g["out"]) < 1e-5
    gv, gl, ga = c_oracle.backward(f("value"), g["shapes"], g["lsi"], f("loc"), f("aw"), f("gout"))
    assert nmax(gv, g["gvalue"]) < 1e-4
    assert nmax(gl, g["gloc"]) < 1e-4
    assert nmax(ga, g["gaw"]) < 1e-4


@pytest.mark.parametrize("name", OP_CASES)
def test_torch_port_matches_reference_pytorch_core(name):
    g = load_golden(name)
    t = lambda k: torch.from_numpy(g[k])
    out, gv, gl, ga = msda_torch.msda_forward_backward_torch(t("value"), t("shapes"), t("loc"), t("aw"), t("gout"))
    assert nmax(out.numpy(), g["out"]) < 1e-13
    assert nmax(gv.numpy(), g["gvalue"]) < 1e-13
    assert nmax(gl.numpy(), g["gloc"]) < 1e-13
    assert nmax(ga.numpy(), g["gaw"]) < 1e-13
    assert torch.equal(msda_torch.level_start_index_of(t("shapes")), t("lsi"))


def test_c_oracle_handles_empty_query_set():
    g = load_golden("op_ragged")
    loc = g["loc"][:, :0]
    aw = g["aw"][:, :0]
    out = c_oracle.forward(g["value"], g["shapes"], g["lsi"], loc, aw)
    assert out.shape == (2, 0, 24)
    gv, gl, ga = c_oracle.backward(g["value"], g["shapes"], g["lsi"], loc, aw, g["gout"][:, :0])
    assert not gv.any() and gl.size == 0 and ga.size == 0


def _sd(g):
    # the d32p4 fixtures store their (bfloat16-representable) parameters and inputs as float32
    return {k[3:]: torch.from_numpy(v).double() for k, v in g.items() if k.startswith("sd.")}


@pytest.mark.parametrize("tag", ["all", "window", "d32p4_all", "d32p4_window"])
def test_temporal_encoder_port_matches_reference_module(tag):
    g = load_golden(f"mod_tenc_{tag}")
    t_frames, c, nl, t_window, heads, pc, pt = [int(x) for x in g["cfg"]]
    t = lambda k: torch.from_numpy(g[k]).double() if g[k].dtype.kind == "f" else torch.from_numpy(g[k])
    offs = [row for row in t("temporal_offsets")]
    out = temporal_torch.temporal_encoder_forward(_sd(g), t("query"), t("ref"), t("inp"), t("shapes"), offs,
                                                  heads, nl, t_window, pc, pt)
    assert nmax(out.numpy(), g["out"]) < 1e-12


@pytest.mark.parametrize("tag", ["2d_ia", "2d_noia", "4d_ia", "4d_noia", "d32p4_2d", "d32p4_4d"])
def test_temporal_decoder_port_matches_reference_module(tag):
    g = load_golden(f"mod_tdec_{tag}")
    t_frames, c, nl, t_window, heads, pc, pt, ia = [int(x) for x in g["cfg"]]
    t = lambda k: torch.from_numpy(g[k]).double() if g[k].dtype.kind == "f" else torch.from_numpy(g[k])
    offs = [row for row in t("temporal_offsets")]
    out, lc, lt, awc, awt = temporal_torch.temporal_decoder_forward(
        _sd(g), t("query"), t("ref"), t("inp"), t("shapes"), offs, heads, nl, t_window, pc, pt, bool(ia))
    assert nmax(out.numpy(), g["out"]) < 1e-12
    assert nmax(torch.stack(lc).numpy(), g["loc_curr"]) < 1e-13
    assert nmax(torch.stack(lt).numpy(), g["loc_temporal"]) < 1e-13
    assert nmax(awc.numpy(), g["aw_curr"]) < 1e-13 and nmax(awt.numpy(), g["aw_temporal"]) < 1e-13


def test_temporal_tables_match_reference_transformer():
    g = load_golden("book_enc_all")
    offs = temporal_torch.all_frames_offsets(3)
    assert np.array_equal(torch.stack(offs).numpy(), g["temporal_offsets"])
    g = load_golden("book_enc_window")
    offs = temporal_torch.window_offsets(4, int(g["t_window"]))
    assert np.array_equal(torch.stack(offs).numpy(), g["temporal_offsets"])
    tl = temporal_torch.temporal_level_start_index(torch.from_numpy(g["tshapes"]))
    assert np.array_equal(tl.numpy(), g["tlsi"])


DCN_CASES = ["dcn_k3_mask", "dcn_k3_c24", "dcn_k3_c40", "dcn_stride2_dil2_nomask", "dcn_k1", "dcn_c33",
             "dcn_fused_c32_o16", "dcn_fused_c72_o32", "dcn_fused_c16_o1", "dcn_fused_c8_o4_s2", "dcn_fused_c40_o64",
             "dcn_fused_c20_o2", "dcn_fused_c136_o8_k1", "dcn_fused_c16_o16_s2"]


def _dcn_run(fn, g, dtype=torch.float64):
    t = lambda k: torch.from_numpy(g[k]).to(dtype)
    st, pd, dl, use_mask = [int(v) for v in g["cfg"]]
    names = ["x", "offset", "weight", "bias"] + (["mask"] if use_mask else [])
    leaves = [t(k).clone().requires_grad_(True) for k in names]
    out = fn(leaves[0], leaves[1], leaves[2], leaves[3], stride=(st, st), padding=(pd, pd), dilation=(dl, dl),
             mask=leaves[4] if use_mask else None)
    out.backward(t("gout"))
    return out.detach(), dict(zip(names, [x.grad for x in leaves]))


@pytest.mark.parametrize("name", DCN_CASES)
def test_deform_conv_restatement_matches_torchvision_fixtures(name):
    """oracle/deform_conv_torch.py against outputs of torchvision.ops.deform_conv2d (CPU, float64) -- the operator the
    reference's mask head calls (deformable_segmentation.py:265) -- forward and every gradient"""
    from oracle import deform_conv_torch
    g = load_golden(name)
    out, grads = _dcn_run(deform_conv_torch.deform_conv2d_torch, g)
    assert nmax(out.numpy(), g["out"]) < 1e-13
    for k, key in (("x", "gx"), ("offset", "goffset"), ("weight", "gweight"), ("bias", "gbias"), ("mask", "gmask")):
        if k in grads:
            assert nmax(grads[k].numpy(), g[key]) < 1e-12, k


def test_deform_conv_restatement_matches_installed_torchvision_directly():
    """same pin without the fixtures: the torchvision in this image, random problem, float64"""
    tv = pytest.importorskip("torchvision.ops")
    from oracle import deform_conv_torch
    g = load_golden("dcn_k3_mask")
    a, ga = _dcn_run(deform_conv_torch.deform_conv2d_torch, g)
    b, gb = _dcn_run(tv.deform_conv2d, g)
    assert nmax(a.numpy(), b.numpy()) < 1e-13
    for k in ga:
        assert nmax(ga[k].numpy(), gb[k].numpy()) < 1e-12


def _edge_problem(case, seed, poisoned):
    """float64 problem of dcn_cases: offsets on a 2^-10 grid with a quarter of the coordinates on the edges of the map;
    ``poisoned``: pixels (0..1, 0..1) non-finite, reached only by taps outside the map"""
    import dcn_cases as dc
    x, off, weight, bias, mask, gout = dc.operands(case, seed, edge_share=0.25)
    if poisoned:
        x, _, off = dc.poison(case, x, off)
    return x, off, weight, bias, mask, gout


def _fwd_bwd(fn, case, x, off, weight, bias, mask, gout):
    leaves = [t.clone().requires_grad_(True) for t in (x, off, weight, bias, mask)]
    out = fn(leaves[0], leaves[1], leaves[2], leaves[3], stride=case.stride, padding=case.pad, dilation=case.dil,
             mask=leaves[4])
    out.backward(gout)
    return [out.detach()] + [t.grad for t in leaves]


@pytest.mark.parametrize("poisoned", [False, True], ids=["finite", "nonfinite_outside"])
@pytest.mark.parametrize("geometry", ["k3", "asym"])
def test_deform_conv_restatement_matches_torchvision_at_edges(geometry, poisoned):
    """the oracle against the installed torchvision (CPU, float64), forward and every gradient: taps on integer
    coordinates, on H - 1 / W - 1, inside (-1, 0) and exactly on -1 and H / W; a 2 x 3 kernel with unequal stride,
    padding and dilation; and non-finite pixels that only taps outside the map reach (torchvision never reads a corner
    outside the map, so they must not turn the result into NaN).

    One convention differs, at a single point: a tap exactly on -1 is void (value 0, the same on both sides), and its
    offset gradient is 0 here and in this library's kernels, while torchvision's coordinate gradient takes the one-sided
    derivative from inside the map.  Both offset components of such a tap are checked to be 0 here; the component whose
    coordinate is -1 is left out of the comparison with torchvision."""
    tv = pytest.importorskip("torchvision.ops")
    import dcn_cases as dc
    from oracle import deform_conv_torch
    geo = dict(kh=2, kw=3, stride=(2, 1), pad=(1, 2), dil=(1, 2)) if geometry == "asym" else {}
    case = dc.Case("edges", 2, 5, 3, 9, 11, **geo)
    ops = _edge_problem(case, 5, poisoned)
    a = _fwd_bwd(deform_conv_torch.deform_conv2d_torch, case, *ops)
    b = _fwd_bwd(tv.deform_conv2d, case, *ops)
    by, bx = dc._base(case)
    o = ops[1].view(case.n, case.k, 2, case.ho, case.wo)
    # the offset component whose own coordinate is exactly -1; the other component of such a tap is compared too, except
    # where torchvision's own value is not finite (its coordinate gradient reads the edge row of a void tap at weight 0,
    # 0 * Inf when that row is poisoned)
    comp = torch.stack([(by + o[:, :, 0]) == -1, (bx + o[:, :, 1]) == -1], dim=2)
    tap = (comp[:, :, 0] | comp[:, :, 1])[:, :, None].expand_as(comp)
    comp, tap = comp.reshape(ops[1].shape), tap.reshape(ops[1].shape)
    assert comp.any()
    assert (a[2][tap] == 0).all()
    b[2] = torch.where(comp | (tap & ~torch.isfinite(b[2])), 0, b[2])
    for name, p, q in zip(("out", "gx", "goffset", "gweight", "gbias", "gmask"), a, b):
        assert torch.isfinite(q).all() or name == "gx", name          # torchvision's own result is finite
        if name == "gx" and poisoned:                                  # nothing reaches the poisoned pixels
            assert (q[:, :, :2, :2] == 0).all() and (p[:, :, :2, :2] == 0).all()
        assert torch.isfinite(p).all(), name
        assert nmax(p.numpy(), q.numpy()) < 1e-12, name
