"""The torch.library custom ops (devis::*) without a GPU: every op on meta tensors against a table of the output
shapes, dtypes and strides the CUDA bodies produce, the op schemas, and registration on import without loading the
library."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

M = "meta"


def _t(*shape, dtype=torch.float32):
    return torch.empty(shape, dtype=dtype, device=M)


def _cl(*shape):
    return torch.empty(shape, device=M).to(memory_format=torch.channels_last)


def _contig(shape):
    st, acc = [], 1
    for s in reversed(shape):
        st.append(acc)
        acc *= max(s, 1)
    return tuple(reversed(st))


def _nchw_of_nhwc(n, c, h, w):
    """strides of an NCHW view of a contiguous (N, H, W, C) buffer"""
    return (h * w * c, 1, w * c, c)


T, S, LQ, NH, D, NL, PC, PT, WT = 3, 80, 10, 8, 32, 2, 4, 4, 2
SHAPES = torch.tensor([[8, 8], [4, 4]])
LSI = torch.tensor([0, 64])
OFFS = [torch.tensor([[1, 2], [-1, 1], [-2, -1]])]
FLAT = [1, 2, -1, 1, -2, -1]


def _msda(dtype):
    v = _t(2, S, NH, D, dtype=dtype)
    loc, aw = _t(2, LQ, NH, NL, PC, 2), _t(2, LQ, NH, NL, PC)
    out = torch.ops.devis.ms_deform_attn(v, SHAPES.to(M), LSI.to(M), loc, aw, 64, False)
    grads = torch.ops.devis.ms_deform_attn_backward(_t(2, LQ, NH * D, dtype=dtype), v, SHAPES.to(M), LSI.to(M), loc,
                                                    aw, 64, True)
    return [out, *grads]


def _tmsda(dtype, need_gv=True):
    v = _t(T, S, NH, D, dtype=dtype)
    lc, ac = _t(T, LQ, NH, NL, PC, 2), _t(T, LQ, NH, NL, PC)
    lt, at = _t(T, LQ, NH, WT * NL, PT, 2), _t(T, LQ, NH, WT * NL, PT)
    out = torch.ops.devis.tmsda(v, lc, ac, lt, at, SHAPES, LSI, None, None, OFFS, [], None, 0, 0)
    grads = torch.ops.devis.tmsda_backward(_t(T, LQ, NH * D, dtype=dtype), v, lc, ac, lt, at, SHAPES, LSI, [], FLAT,
                                           None, 0, 0, need_gv)
    return [out, *grads]


def _fused(dtype, want_sampling, temporal, ref_dim=2, need_gref=False):
    v = _t(T, S, NH, D, dtype=dtype)
    ref = _t(T, LQ, NL, ref_dim)
    oc, lgc = _t(T, LQ, NH, NL, PC, 2), _t(T, LQ, NH, NL * PC)
    ot, lgt = (_t(T, LQ, NH, WT * NL, PT, 2), _t(T, LQ, NH, WT * NL * PT)) if temporal else (None, None)
    offs, flat = (OFFS, []) if temporal else ([], [])
    res = torch.ops.devis.tmsda_fused(v, ref, oc, lgc, ot, lgt, SHAPES, LSI, None, None, offs, flat, None, 8, 8, 0,
                                      want_sampling, _t(T, S, dtype=torch.bool), False)
    grads = torch.ops.devis.tmsda_fused_backward(_t(T, LQ, NH * D, dtype=dtype), v, ref, oc, lgc, ot, lgt, SHAPES, LSI,
                                                 [], FLAT if temporal else [], None, 8, 8, 0, None, True, need_gref)
    return [*res, *grads]


def _dcn(form, channels_last, need=(True, True, True, True, True)):
    n, c, h, w, cout = 2, 8, 6, 10, 4
    x = _cl(n, c, h, w) if channels_last else _t(n, c, h, w)
    off, wt, b, m = _t(n, 18, h, w), _t(cout, c, 3, 3), _t(cout), _t(n, 9, h, w)
    geo = (1, 1, 1, 1, 1, 1)
    g = _t(n, cout, h, w)
    if form == "fused":
        out, xc, packed = torch.ops.devis.deform_conv2d_fused(x, off, wt, b, m, *geo, 123)
        grads = torch.ops.devis.deform_conv2d_fused_backward(g, x, xc, off, wt, b, m, packed, *geo, 3, *need)
        return [out, xc, packed, *grads]
    if form == "im2col":
        out, xc, cols = torch.ops.devis.deform_conv2d_im2col(x, off, wt, b, m, *geo)
        grads = torch.ops.devis.deform_conv2d_im2col_backward(g, x, xc, off, wt, b, m, cols, *geo, *need)
        return [out, xc, cols, *grads]
    out, xc = torch.ops.devis.deform_conv2d_igemm(x, off, wt, b, m, *geo)
    grads = torch.ops.devis.deform_conv2d_igemm_backward(g, x, xc, off, wt, b, m, *geo, *need)
    return [out, xc, *grads]


F32, BF16, F16, F64, E = torch.float32, torch.bfloat16, torch.float16, torch.float64, ((0,), (1,))
GV = (T, S, NH, D)
DCN_OUT = ((2, 4, 6, 10), _nchw_of_nhwc(2, 4, 6, 10))
DCN_GIN = ((2, 8, 6, 10), _nchw_of_nhwc(2, 8, 6, 10))
DCN_GW = ((4, 8, 3, 3), _nchw_of_nhwc(4, 8, 3, 3))
DCN_XC = ((2, 6, 10, 8), _contig((2, 6, 10, 8)))
DCN_GRADS = [DCN_GIN, ((2, 18, 6, 10), None), DCN_GW, ((4,), None), ((2, 9, 6, 10), None)]

# (case, call, [(shape, strides or None for contiguous, dtype or None for the value dtype)])
CASES = [
    ("msda_f32", lambda: _msda(F32), [((2, LQ, NH * D), None, F32), ((2, S, NH, D), None, F32),
                                      ((2, LQ, NH, NL, PC, 2), None, F32), ((2, LQ, NH, NL, PC), None, F32)]),
    ("msda_bf16", lambda: _msda(BF16), [((2, LQ, NH * D), None, BF16), ((2, S, NH, D), None, BF16),
                                        ((2, LQ, NH, NL, PC, 2), None, F32), ((2, LQ, NH, NL, PC), None, F32)]),
    ("msda_f64", lambda: _msda(F64), [((2, LQ, NH * D), None, F64), ((2, S, NH, D), None, F64),
                                      ((2, LQ, NH, NL, PC, 2), None, F32), ((2, LQ, NH, NL, PC), None, F32)]),
    ("tmsda_f16", lambda: _tmsda(F16), [((T, LQ, NH * D), None, F16), (GV, None, F16),
                                        ((T, LQ, NH, NL, PC, 2), None, F32), ((T, LQ, NH, NL, PC), None, F32),
                                        ((T, LQ, NH, WT * NL, PT, 2), None, F32), ((T, LQ, NH, WT * NL, PT), None, F32)]),
    ("tmsda_no_grad_value", lambda: _tmsda(F32, need_gv=False),
     [((T, LQ, NH * D), None, F32), ((0,), None, F32), ((T, LQ, NH, NL, PC, 2), None, F32),
      ((T, LQ, NH, NL, PC), None, F32), ((T, LQ, NH, WT * NL, PT, 2), None, F32), ((T, LQ, NH, WT * NL, PT), None, F32)]),
    ("fused_bf16_sampling", lambda: _fused(BF16, True, True),
     [((T, LQ, NH * D), None, BF16), ((T, LQ, NH, NL, PC, 2), None, F32), ((T, LQ, NH, NL, PC), None, F32),
      ((T, LQ, NH, WT * NL, PT, 2), None, F32), ((T, LQ, NH, WT * NL, PT), None, F32),
      (GV, None, BF16), ((0,), None, BF16), ((T, LQ, NH, NL, PC, 2), None, F32), ((T, LQ, NH, NL * PC), None, F32),
      ((T, LQ, NH, WT * NL, PT, 2), None, F32), ((T, LQ, NH, WT * NL * PT), None, F32)]),
    ("fused_batch_boxes", lambda: _fused(F32, False, False, ref_dim=4, need_gref=True),
     [((T, LQ, NH * D), None, F32), ((0,), None, F32), ((0,), None, F32), ((0,), None, F32), ((0,), None, F32),
      (GV, None, F32), ((T, LQ, NL, 4), None, F32), ((T, LQ, NH, NL, PC, 2), None, F32),
      ((T, LQ, NH, NL * PC), None, F32), ((0,), None, F32), ((0,), None, F32)]),
    ("fused_sampling_no_temporal", lambda: _fused(F16, True, False),
     [((T, LQ, NH * D), None, F16), ((T, LQ, NH, NL, PC, 2), None, F32), ((T, LQ, NH, NL, PC), None, F32),
      ((0,), None, F32), ((0,), None, F32), (GV, None, F16), ((0,), None, F16), ((T, LQ, NH, NL, PC, 2), None, F32),
      ((T, LQ, NH, NL * PC), None, F32), ((0,), None, F32), ((0,), None, F32)]),
    ("dcn_fused_nchw", lambda: _dcn("fused", False),
     [DCN_OUT, DCN_XC, ((123,), None), *DCN_GRADS]),
    ("dcn_fused_channels_last_weight_only", lambda: _dcn("fused", True, (False, False, True, False, False)),
     [DCN_OUT, E, ((123,), None), E, E, DCN_GW, E, E]),
    ("dcn_im2col_channels_last", lambda: _dcn("im2col", True),
     [DCN_OUT, E, ((2 * 6 * 10, 9 * 8), None), *DCN_GRADS]),
    ("dcn_igemm_nchw", lambda: _dcn("igemm", False), [DCN_OUT, DCN_XC, *DCN_GRADS]),
]


@pytest.mark.parametrize("name,call,expected", CASES, ids=[c[0] for c in CASES])
def test_fake_outputs_on_meta_tensors(name, call, expected):
    import devis_b200  # noqa: F401  (registers the ops)
    got = call()
    assert len(got) == len(expected)
    for i, (t, exp) in enumerate(zip(got, expected)):
        shape, strides = exp[0], exp[1]
        assert t.device.type == "meta", (name, i)
        assert tuple(t.shape) == shape, (name, i, tuple(t.shape), shape)
        assert t.stride() == (strides if strides is not None else _contig(shape)), (name, i, t.stride())
        if len(exp) > 2 and exp[2] is not None and shape != (0,):       # (placeholders of absent outputs: any dtype)
            assert t.dtype == exp[2], (name, i, t.dtype)


SCHEMAS = {
    "ms_deform_attn": "devis::ms_deform_attn(Tensor value, Tensor spatial_shapes, Tensor level_start_index, "
                      "Tensor sampling_loc, Tensor attn_weight, SymInt im2col_step, bool check_levels) -> Tensor",
    "tmsda": "devis::tmsda(Tensor value, Tensor loc_curr, Tensor aw_curr, Tensor? loc_temporal, Tensor? aw_temporal, "
             "Tensor spatial_shapes, Tensor level_start_index, Tensor? temporal_spatial_shapes, "
             "Tensor? temporal_level_start_index, Tensor[] temporal_offsets, SymInt[] frame_offsets, "
             "Tensor? query_order, SymInt tile_h, "
             "SymInt tile_w) -> Tensor",
    "tmsda_fused": "devis::tmsda_fused(Tensor value, Tensor ref, Tensor off_curr, Tensor logit_curr, "
                   "Tensor? off_temporal, Tensor? logit_temporal, Tensor spatial_shapes, Tensor level_start_index, "
                   "Tensor? temporal_spatial_shapes, Tensor? temporal_level_start_index, Tensor[] temporal_offsets, "
                   "SymInt[] frame_offsets, Tensor? query_order, SymInt tile_h, SymInt tile_w, SymInt temporal_ref_mode, bool want_sampling, "
                   "Tensor? padding_mask, bool check_levels) -> (Tensor, Tensor, Tensor, Tensor, Tensor)",
    "deform_conv2d_fused": "devis::deform_conv2d_fused(Tensor input, Tensor offset, Tensor weight, Tensor? bias, "
                           "Tensor? mask, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, SymInt dil_h, "
                           "SymInt dil_w, SymInt packed_elems) -> (Tensor, Tensor, Tensor)",
    "deform_conv2d_im2col": "devis::deform_conv2d_im2col(Tensor input, Tensor offset, Tensor weight, Tensor? bias, "
                            "Tensor? mask, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, SymInt dil_h, "
                            "SymInt dil_w) -> (Tensor, Tensor, Tensor)",
    "deform_conv2d_igemm": "devis::deform_conv2d_igemm(Tensor input, Tensor offset, Tensor weight, Tensor? bias, "
                           "Tensor? mask, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, SymInt dil_h, "
                           "SymInt dil_w) -> (Tensor, Tensor)",
}
OPS = ["ms_deform_attn", "tmsda", "tmsda_fused", "deform_conv2d_fused", "deform_conv2d_im2col", "deform_conv2d_igemm"]


def test_schemas_are_functional_and_as_documented():
    import devis_b200  # noqa: F401
    for name in OPS:
        for op_name in (name, name + "_backward"):
            schema = getattr(torch.ops.devis, op_name).default._schema
            assert not schema.is_mutable, op_name
            assert all(a.alias_info is None for a in list(schema.arguments) + list(schema.returns)), op_name
            # no defaults: the dispatcher would drop such arguments, and the autograd formulas count them
            assert all(not a.has_default_value() for a in schema.arguments), op_name
        assert str(getattr(torch.ops.devis, name).default._schema) == SCHEMAS[name]


def test_cpu_tensors_raise_runtime_error_from_the_op():
    import devis_b200  # noqa: F401
    v = torch.zeros(1, 80, 8, 32)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        torch.ops.devis.ms_deform_attn(v, SHAPES, LSI, torch.zeros(1, 5, 8, 2, 4, 2), torch.zeros(1, 5, 8, 2, 4), 64,
                                       False)
    with pytest.raises(RuntimeError, match="not implemented on the CPU"):
        torch.ops.devis.deform_conv2d_im2col(torch.zeros(1, 4, 5, 5), torch.zeros(1, 18, 5, 5), torch.zeros(2, 4, 3, 3),
                                             None, None, 1, 1, 1, 1, 1, 1)


def test_import_registers_the_ops_without_loading_the_library():
    code = ("import sys\nsys.path.insert(0, %r)\nimport torch, devis_b200\nfrom devis_b200 import _lib\n"
            "names = %r\n"
            "ok = all(hasattr(torch.ops.devis, n) and hasattr(torch.ops.devis, n + '_backward') for n in names)\n"
            "v = torch.empty(2, 80, 8, 32, device='meta')\n"
            "out = torch.ops.devis.tmsda_fused(v, torch.empty(2, 5, 2, 2, device='meta'), "
            "torch.empty(2, 5, 8, 2, 4, 2, device='meta'), torch.empty(2, 5, 8, 8, device='meta'), None, None, "
            "torch.tensor([[8, 8], [4, 4]]), torch.tensor([0, 64]), None, None, [], [], None, 8, 8, 0, False, None, True)\n"
            "print('REGISTERED', ok, 'LOADED', _lib._lib is not None, tuple(out[0].shape))\n" % (ROOT, OPS))
    env = dict(os.environ, DEVIS_MSDA_LIB="/nonexistent/libdevis_msda.so")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert "REGISTERED True LOADED False (2, 5, 256)" in out.stdout, out.stdout + out.stderr


def test_no_autograd_function_launches_a_kernel():
    """the ops are the implementation: no torch.autograd.Function subclass is left in the package"""
    pkg = os.path.join(ROOT, "devis_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "(Function)" not in src and "torch.autograd import Function" not in src, f
