"""Offset groups of the deformable convolution, without a GPU: host-side validation of the _og C-ABI entry points, which
fused forms serve a layer, the packed-weight sizes, and the dcn_og_*.npz fixtures against torchvision's CPU operator."""
import glob
import os

import pytest
import torch

from conftest import GOLDEN, load_golden, nmax

ERR_NULL, ERR_BAD_SHAPE, ERR_TOO_LARGE, ERR_UNSUPPORTED = -1, -2, -5, -8
F32, F64 = 0, 1
SMALL_COUT = (1, 2, 4, 8, 16)
# (Cin, Cout): the mask-head layers (benchmarks/dcn_bench.py LAYERS) and the fixture layers
LAYER_SHAPES = [(264, 264), (264, 128), (136, 64), (72, 32), (32, 16), (16, 1), (8, 5), (24, 6), (40, 6), (33, 3),
                (16, 16), (8, 4), (40, 64), (20, 2), (136, 8), (30, 16), (64, 8), (72, 4)]


def _lib():
    from devis_b200 import _lib
    return _lib.load()


def test_og_entry_points_validate_on_the_host():
    """offset_groups < 1 and channels % offset_groups != 0 -> BAD_SHAPE, G * kh * kw beyond the grid -> TOO_LARGE, fused
    calls for layers the fused form does not serve -> UNSUPPORTED; all before any CUDA call (null pointers throughout)"""
    lib = _lib()
    null = None
    dims = (1, 4, 4, 8, 4, 4, 3, 3, 1, 1, 1, 1, 1, 1)
    im2col = lambda dims, og, dtype=F32: lib.devis_dcn_im2col_og(null, null, null, null, *dims, og, dtype, null)
    col2im = lambda dims, og, dtype=F32: lib.devis_dcn_col2im_og(*([null] * 7), *dims, og, dtype, 0, null, 0, null)
    fwd = lambda dims, og, cout: lib.devis_dcn_fused_forward_og(*([null] * 6), *dims, og, cout, null)
    bwd = lambda dims, og, cout: lib.devis_dcn_fused_backward_og(*([null] * 8), *dims, og, cout, 0, null, 0, null)
    for call in (im2col, col2im):
        for og in (0, -1, 3, 5):
            assert call(dims, og) == ERR_BAD_SHAPE, og
        for og in (1, 2, 4, 8):
            assert call(dims, og) == ERR_NULL, og
            assert call(dims, og, F64) == ERR_NULL, og
        big = dims[:6] + (91, 91) + dims[8:]                    # 91 * 91 = 8281 kernel positions
        assert call(big, 1) == ERR_NULL and call(big, 8) == ERR_TOO_LARGE
    for call in (fwd, bwd):
        for og in (0, 3):
            assert call(dims, og, 16) == ERR_BAD_SHAPE, og
        assert call(dims, 2, 16) == ERR_NULL                     # Cg = 4
        assert call(dims, 4, 16) == ERR_UNSUPPORTED              # Cg = 2: no float4 pieces
        assert call(dims, 2, 5) == ERR_UNSUPPORTED
    wide = dims[:3] + (32,) + dims[4:]
    assert fwd(wide, 1, 32) == ERR_NULL                          # constant-bank forward at G = 1 ...
    assert fwd(wide, 2, 32) == ERR_UNSUPPORTED                   # ... not at G > 1
    assert lib.devis_dcn_pack_weight_og(null, null, 8, 16, 3, 3, 0, null) == ERR_BAD_SHAPE
    assert lib.devis_dcn_pack_weight_og(null, null, 8, 16, 3, 3, 3, null) == ERR_BAD_SHAPE
    assert lib.devis_dcn_pack_weight_og(null, null, 8, 5, 3, 3, 2, null) == ERR_UNSUPPORTED
    assert lib.devis_dcn_pack_weight_og(null, null, 8, 16, 3, 3, 2, null) == ERR_NULL
    # empty batches are fine with null pointers and launch nothing
    before = lib.devis_msda_launch_count()
    empty = (0,) + dims[1:]
    assert im2col(empty, 2) == 0 and col2im(empty, 2) == 0 and fwd(empty, 2, 16) == 0 and bwd(empty, 2, 16) == 0
    assert lib.devis_msda_launch_count() == before


def test_fused_form_table():
    """G = 1: the _og query equals the old one.  G > 1: the lane-group kernels serve the layer (forward and data
    backward) iff float32, (Cin / G) % 4 == 0 and Cout in {1, 2, 4, 8, 16}; the constant-bank forward never does"""
    lib = _lib()
    for c, cout in LAYER_SHAPES:
        for dtype in (F32, F64):
            assert lib.devis_dcn_fused_form_og(c, cout, 3, 3, 1, dtype) == lib.devis_dcn_fused_form(c, cout, 3, 3, dtype)
            assert lib.devis_dcn_fused_form_og(c, cout, 1, 1, 1, dtype) == lib.devis_dcn_fused_form(c, cout, 1, 1, dtype)
        for og in (2, 3, 4, 8):
            served = c % og == 0 and (c // og) % 4 == 0 and cout in SMALL_COUT
            assert lib.devis_dcn_fused_form_og(c, cout, 3, 3, og, F32) == (3 if served else 0), (c, cout, og)
            assert lib.devis_dcn_fused_form_og(c, cout, 3, 3, og, F64) == 0
    assert lib.devis_dcn_fused_form_og(32, 16, 3, 3, 2, F32) == 3 and lib.devis_dcn_fused_form_og(16, 1, 3, 3, 4, F32) == 3
    assert lib.devis_dcn_fused_form_og(72, 32, 3, 3, 2, F32) == 0 and lib.devis_dcn_fused_form_og(264, 8, 3, 3, 4, F32) == 0
    assert lib.devis_dcn_fused_form_og(136, 8, 3, 3, 2, F32) == 3 and lib.devis_dcn_fused_form_og(16, 1, 3, 3, 0, F32) == 0


def test_packed_weight_sizes():
    """G = 1: the old size.  G > 1: K * G * nblk * Cout * lanes * 4 floats, nblk = ceil(Cg / 4 / lanes), lanes = 8 when
    Cg / 4 > 4 else 4; 0 for layers the fused form does not serve"""
    lib = _lib()
    for c, cout in LAYER_SHAPES:
        for kh, kw in ((3, 3), (1, 1), (3, 1)):
            assert lib.devis_dcn_packed_weight_elems_og(c, cout, kh, kw, 1) == lib.devis_dcn_packed_weight_elems(c, cout, kh, kw)
        for og in (2, 4):
            got = lib.devis_dcn_packed_weight_elems_og(c, cout, 3, 3, og)
            if lib.devis_dcn_fused_form_og(c, cout, 3, 3, og, F32):
                c4 = c // og // 4
                lanes = 8 if c4 > 4 else 4
                assert got == 9 * og * -(-c4 // lanes) * cout * lanes * 4, (c, cout, og)
            else:
                assert got == 0
    assert lib.devis_dcn_packed_weight_elems_og(32, 16, 3, 3, 2) == 9 * 2 * 1 * 16 * 4 * 4


def _fixtures():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "dcn_og_*.npz")))


def test_fixture_set_is_complete():
    from golden.make_dcn_offset_groups import CASES
    assert _fixtures() == sorted(CASES)


@pytest.mark.parametrize("name", _fixtures())
def test_fixtures_match_torchvision_cpu(name):
    """the committed fixtures, re-run through torchvision's CPU operator"""
    pytest.importorskip("torchvision.ops")
    from golden.make_dcn_offset_groups import reference
    g = load_golden(name)
    t = lambda k: torch.from_numpy(g[k])
    mask = t("mask") if "mask" in g else None
    assert g["offset"].shape[1] // (2 * g["weight"].shape[2] * g["weight"].shape[3]) > 1
    out, leaves = reference(t("x"), t("offset"), t("weight"), t("bias"), mask, g["cfg"])
    out.backward(t("gout"))
    assert nmax(out.detach().numpy(), g["out"]) <= 1e-13
    for leaf, key in zip(leaves, ("gx", "goffset", "gweight", "gbias", "gmask")):
        assert nmax(leaf.grad.numpy(), g[key]) <= 1e-13, key
