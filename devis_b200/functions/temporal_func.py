"""Whole-clip temporal multi-scale deformable attention as ONE autograd op.

The reference computes a layer's temporal attention with a Python loop over the T query frames:
per frame one ``MSDeformAttnFunction.apply`` on the frame's own value, a gather copy
``value[temporal_frames].flatten(0, 1)``, a second ``apply`` on that copy with the temporal frames
stacked along the level axis, and an add (modules/ms_deform_attn.py:435-460 encoder, :325-404
decoder) -- 2T launches, T copies and 2T materialised outputs forward, the same again backward.
``TemporalMSDeformAttnFunction`` does the whole clip in one launch each way: value (T,S,M,D) is read
in place through the frame table, current and temporal taps accumulate into the same registers, and
the backward scatters straight into grad_value (T,S,M,D) -- no copies, no index_add.

Both ops are ``torch.library`` custom ops (``devis::tmsda``, ``devis::tmsda_fused`` and their ``*_backward``), so
torch.compile and torch.export trace each one as a single node.  Their arguments are tensors and ints only: the clip
geometry travels as the pyramid tensors and the frame offsets, and the op body rebuilds the memoised ClipGeometry from
their host copies (clip_geometry.op_geometry) -- every host read and data-dependent check happens inside the op.
"""
from typing import Optional

import torch

from .. import _lib
from .. import MultiScaleDeformableAttention as MSDA
from .. import clip_geometry

# float16 value (what torch.autocast("cuda") hands the op by default) is served like bfloat16: 16-bit value, output and
# grad_output, float32 locations, weights and gradients
_DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
_16BIT = (torch.bfloat16, torch.float16)

# argument types of the op schemas
Tensor, OptTensor, Tensors = torch.Tensor, Optional[torch.Tensor], list[torch.Tensor]


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def _aux(t, value):
    want = torch.float32 if value.dtype in _16BIT else value.dtype
    t = t if t.dtype == want else t.to(want)
    return t if t.is_contiguous() else t.contiguous()


def _none(t):
    """the placeholder of an absent optional output (ops return tensors only) -> None"""
    return None if t is None or t.numel() == 0 and t.dim() == 1 else t


def _no_grad_list(ints):
    """the 'gradient' of an int[] argument: autograd reads an empty list as an (empty) tensor list"""
    return [] if not ints else None


def _dims(value, loc_curr, loc_temporal, geom):
    t, s, m, d = value.shape
    lq = loc_curr.shape[1]
    pc = loc_curr.shape[4]
    pt = loc_temporal.shape[4] if loc_temporal is not None and geom.t_window else 0
    if t != geom.n_frames or s != geom.spatial_size:
        raise RuntimeError(f"value {tuple(value.shape)} does not match the clip geometry "
                           f"(frames {geom.n_frames}, rows {geom.spatial_size})")
    if loc_curr.shape[3] != geom.n_levels:
        raise RuntimeError("loc_curr level axis does not match the clip geometry")
    if pt and loc_temporal.shape[3] != geom.t_window * geom.n_levels:
        raise RuntimeError("loc_temporal level axis must be t_window * n_levels")
    return t, s, m, d, lq, pc, pt


def _wt(temporal_offsets, frame_offsets, n_frames):
    """t_window from the shapes of the frame offsets alone (what the fake implementations may use)"""
    if frame_offsets:
        return len(frame_offsets) // n_frames
    if not temporal_offsets:
        return 0
    return temporal_offsets[0].shape[-1]


def _order(geom, query_order, tile_h, tile_w, lq, device):
    """the explicit query order, else the 2-D tile walk of the pixel-grid queries when asked for and Lq == S"""
    if query_order is not None or tile_h <= 0 or lq != geom.spatial_size:
        return query_order
    return geom.tile_order(device, tile_h, tile_w)


# ------------------------------------------------------------------------------------------------------------------------
# devis::tmsda -- whole-clip op on sampling locations and weights
# ------------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("devis::tmsda", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _tmsda_op(value: Tensor, loc_curr: Tensor, aw_curr: Tensor, loc_temporal: OptTensor, aw_temporal: OptTensor,
              spatial_shapes: Tensor, level_start_index: Tensor, temporal_spatial_shapes: OptTensor,
              temporal_level_start_index: OptTensor, temporal_offsets: Tensors, frame_offsets: list[int], query_order: OptTensor,
              tile_h: int, tile_w: int) -> Tensor:
    if not value.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if value.dtype not in _DTYPES:
        raise RuntimeError(f'"temporal_ms_deform_attn" not implemented for \'{value.dtype}\'')
    geometry = clip_geometry.op_geometry(value.shape[0], spatial_shapes, level_start_index, temporal_spatial_shapes,
                                         temporal_level_start_index, temporal_offsets, frame_offsets)
    value = value if value.is_contiguous() else value.contiguous()
    lc, ac = _aux(loc_curr, value), _aux(aw_curr, value)
    has_t = geometry.t_window > 0 and loc_temporal is not None
    lt = _aux(loc_temporal, value) if has_t else None
    at = _aux(aw_temporal, value) if has_t else None
    t, s, m, d, lq, pc, pt = _dims(value, lc, lt, geometry)
    query_order = _order(geometry, query_order, tile_h, tile_w, lq, value.device)
    out = torch.empty((t, lq, m * d), dtype=value.dtype, device=value.device)
    with torch.cuda.device(value.device):
        stream = torch.cuda.current_stream().cuda_stream
        _lib.check(_lib.load().devis_tmsda_forward(
            _ptr(value), geometry.shapes_ptr, geometry.lsi_ptr, geometry.frames_ptr,
            _ptr(lc), _ptr(ac), _ptr(lt), _ptr(at), _ptr(out), _ptr(query_order),
            t, s, m, d, geometry.n_levels, lq, pc, pt, geometry.t_window if has_t else 0,
            _DTYPES[value.dtype], stream))
    return out


@_tmsda_op.register_fake
def _(value, loc_curr, aw_curr, loc_temporal, aw_temporal, spatial_shapes, level_start_index, temporal_spatial_shapes,
      temporal_level_start_index, temporal_offsets, frame_offsets, query_order, tile_h, tile_w):
    t, _, m, d = value.shape
    return value.new_empty((t, loc_curr.shape[1], m * d))


@torch.library.custom_op("devis::tmsda_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _tmsda_backward_op(grad_output: Tensor, value: Tensor, loc_curr: Tensor, aw_curr: Tensor, loc_temporal: OptTensor,
                       aw_temporal: OptTensor, spatial_shapes: Tensor, level_start_index: Tensor,
                       temporal_offsets: Tensors, frame_offsets: list[int], query_order: OptTensor, tile_h: int, tile_w: int,
                       need_grad_value: bool) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """(grad_value, grad_loc_curr, grad_aw_curr, grad_loc_temporal, grad_aw_temporal), each in its input's dtype; an
    empty tensor stands for a gradient that is not computed"""
    geometry = clip_geometry.op_geometry(value.shape[0], spatial_shapes, level_start_index, None, None,
                                         temporal_offsets, frame_offsets)
    value = value if value.is_contiguous() else value.contiguous()
    lc, ac = _aux(loc_curr, value), _aux(aw_curr, value)
    has_t = geometry.t_window > 0 and loc_temporal is not None
    lt = _aux(loc_temporal, value) if has_t else None
    at = _aux(aw_temporal, value) if has_t else None
    t, s, m, d, lq, pc, pt = _dims(value, lc, lt, geometry)
    query_order = _order(geometry, query_order, tile_h, tile_w, lq, value.device)
    gout = grad_output if grad_output.dtype == value.dtype else grad_output.to(value.dtype)
    gout = gout if gout.is_contiguous() else gout.contiguous()
    need_gv = need_grad_value
    half_acc = need_gv and MSDA.bf16_accumulate_enabled(value)
    acc_dtype = torch.float32 if (value.dtype in _16BIT and not half_acc) else value.dtype
    gv = torch.empty(value.shape, dtype=acc_dtype, device=value.device) if need_gv else None
    glc, gac = torch.empty_like(lc), torch.empty_like(ac)
    glt = torch.empty_like(lt) if has_t else None
    gat = torch.empty_like(at) if has_t else None
    flags = (_lib.FLAG_DETERMINISTIC if MSDA.deterministic_enabled(value.dtype) else 0) \
        | (0 if need_gv else _lib.FLAG_NO_GRAD_VALUE) | (_lib.FLAG_BF16_GRAD_VALUE if half_acc else 0)
    lib = _lib.load()
    code = _DTYPES[value.dtype]
    with torch.cuda.device(value.device):
        stream = torch.cuda.current_stream().cuda_stream
        ws_bytes = lib.devis_tmsda_backward_workspace_bytes(t, s, m, d, geometry.n_levels, lq, pc, pt,
                                                            geometry.t_window if has_t else 0, code, flags)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=value.device) if ws_bytes else None
        _lib.check(lib.devis_tmsda_backward(
            _ptr(value), geometry.shapes_ptr, geometry.lsi_ptr, geometry.frames_ptr,
            _ptr(lc), _ptr(ac), _ptr(lt), _ptr(at), _ptr(gout),
            _ptr(gv), _ptr(glc), _ptr(gac), _ptr(glt), _ptr(gat), _ptr(query_order),
            t, s, m, d, geometry.n_levels, lq, pc, pt, geometry.t_window if has_t else 0,
            code, flags, _ptr(ws), ws_bytes, stream))
    cast = lambda g, like: value.new_empty(0) if g is None else (g if g.dtype == like.dtype else g.to(like.dtype))
    return (cast(gv, value), cast(glc, loc_curr), cast(gac, aw_curr), cast(glt, loc_temporal),
            cast(gat, aw_temporal))


@_tmsda_backward_op.register_fake
def _(grad_output, value, loc_curr, aw_curr, loc_temporal, aw_temporal, spatial_shapes, level_start_index,
      temporal_offsets, frame_offsets, query_order, tile_h, tile_w, need_grad_value):
    has_t = _wt(temporal_offsets, frame_offsets, value.shape[0]) > 0 and loc_temporal is not None
    like = lambda x, on: torch.empty_like(x, memory_format=torch.contiguous_format) if on else value.new_empty(0)
    return (like(value, need_grad_value), like(loc_curr, True), like(aw_curr, True), like(loc_temporal, has_t),
            like(aw_temporal, has_t))


def _tmsda_setup_context(ctx, inputs, output):
    (value, loc_curr, aw_curr, loc_temporal, aw_temporal, shapes, lsi, _, _, offsets, frame_offsets, query_order,
     tile_h, tile_w) = inputs
    ctx.tile = (tile_h, tile_w)
    ctx.frame_offsets = frame_offsets
    ctx.n_offsets = len(offsets)
    ctx.save_for_backward(value, loc_curr, aw_curr, loc_temporal, aw_temporal, shapes, lsi, query_order, *offsets)


def _tmsda_backward(ctx, grad_output):
    value, lc, ac, lt, at, shapes, lsi, query_order, *offsets = ctx.saved_tensors
    gv, glc, gac, glt, gat = _tmsda_backward_op(grad_output, value, lc, ac, lt, at, shapes, lsi, offsets,
                                                ctx.frame_offsets, query_order, *ctx.tile, ctx.needs_input_grad[0])
    return (_none(gv), glc, gac, _none(glt), _none(gat), None, None, None, None, [None] * ctx.n_offsets,
            _no_grad_list(ctx.frame_offsets), None, None, None)


_tmsda_op.register_autograd(_tmsda_backward, setup_context=_tmsda_setup_context)


class TemporalMSDeformAttnFunction:
    """apply(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None) -> (T, Lq, M*D)

    value (T,S,M,D); loc_curr (T,Lq,M,L,Pc,2); aw_curr (T,Lq,M,L,Pc); loc_temporal (T,Lq,M,Wt*L,Pt,2);
    aw_temporal (T,Lq,M,Wt*L,Pt) -- exactly the tensors the reference's per-frame loop slices
    (ms_deform_attn.py:437-457); geometry is a devis_b200.clip_geometry.ClipGeometry.  Entry point of the op
    ``devis::tmsda`` (once differentiable)."""

    @staticmethod
    def apply(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None):
        shapes, lsi, offsets = geometry.op_args()
        return _tmsda_op(value, loc_curr, aw_curr, loc_temporal, aw_temporal, shapes, lsi, None, None, [], offsets,
                         query_order, 0, 0)


# ------------------------------------------------------------------------------------------------------------------------
# devis::tmsda_fused -- whole-clip op on the Linear outputs (softmax and location arithmetic in the kernels)
# ------------------------------------------------------------------------------------------------------------------------
def _f32(t):
    return (t if t.dtype == torch.float32 else t.float()).contiguous()


@torch.library.custom_op("devis::tmsda_fused", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _fused_op(value: Tensor, ref: Tensor, off_curr: Tensor, logit_curr: Tensor, off_temporal: OptTensor,
              logit_temporal: OptTensor, spatial_shapes: Tensor, level_start_index: Tensor,
              temporal_spatial_shapes: OptTensor, temporal_level_start_index: OptTensor, temporal_offsets: Tensors,
              frame_offsets: list[int], query_order: OptTensor, tile_h: int, tile_w: int, temporal_ref_mode: int, want_sampling: bool,
              padding_mask: OptTensor, check_levels: bool) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """(out, loc_curr, aw_curr, loc_temporal, aw_temporal): the sampling by-products are empty tensors unless
    ``want_sampling`` (and the temporal ones unless the clip has temporal slots).  ``check_levels``: MSDeformAttn's
    ``sum(H*W) == S`` assertion."""
    if not value.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if value.dtype not in (torch.float32,) + _16BIT:
        raise RuntimeError(f'"temporal_ms_deform_attn_fused" not implemented for \'{value.dtype}\'')
    geometry = clip_geometry.op_geometry(value.shape[0], spatial_shapes, level_start_index, temporal_spatial_shapes,
                                         temporal_level_start_index, temporal_offsets, frame_offsets)
    if check_levels:
        assert sum(h * w for h, w in geometry.shapes) == value.shape[1]
    value = value if value.is_contiguous() else value.contiguous()
    ref, oc, lc = _f32(ref), _f32(off_curr), _f32(logit_curr)
    has_t = geometry.t_window > 0 and off_temporal is not None
    ot = _f32(off_temporal) if has_t else None
    lt = _f32(logit_temporal) if has_t else None
    t, s, m, d = value.shape
    lq, pc = oc.shape[1], oc.shape[4]
    pt = ot.shape[4] if has_t else 0
    ref_dim = ref.shape[-1]
    if t != geometry.n_frames or s != geometry.spatial_size or oc.shape[3] != geometry.n_levels:
        raise RuntimeError("operands do not match the clip geometry")
    if tuple(ref.shape) != (t, lq, geometry.n_levels, ref_dim) or ref_dim not in (2, 4):
        raise RuntimeError(f"reference points {tuple(ref.shape)} must be (T, Lq, L, 2|4)")
    if padding_mask is not None:
        if tuple(padding_mask.shape) != (t, s) or padding_mask.dtype not in (torch.bool, torch.uint8) \
                or padding_mask.device != value.device:
            raise RuntimeError(f"padding mask {tuple(padding_mask.shape)} {padding_mask.dtype} must be a bool tensor "
                               f"(T, S) = {(t, s)} on the device of value")
        padding_mask = padding_mask.detach().contiguous()
    query_order = _order(geometry, query_order, tile_h, tile_w, lq, value.device)
    out = torch.empty((t, lq, m * d), dtype=value.dtype, device=value.device)
    samp = [None] * 4
    if want_sampling:
        samp[0], samp[1] = torch.empty_like(oc), torch.empty((t, lq, m, geometry.n_levels, pc), dtype=torch.float32,
                                                             device=value.device)
        if has_t:
            samp[2] = torch.empty_like(ot)
            samp[3] = torch.empty((t, lq, m, geometry.t_window * geometry.n_levels, pt), dtype=torch.float32,
                                  device=value.device)
    with torch.cuda.device(value.device):
        _lib.check(_lib.load().devis_tmsda_fused_forward_ex(
            _ptr(value), geometry.shapes_ptr, geometry.lsi_ptr, geometry.frames_ptr, _ptr(ref), _ptr(oc), _ptr(lc),
            _ptr(ot), _ptr(lt), _ptr(out), _ptr(samp[0]), _ptr(samp[1]), _ptr(samp[2]), _ptr(samp[3]),
            _ptr(query_order), _ptr(padding_mask), t, s, m, d, geometry.n_levels, lq, pc, pt,
            geometry.t_window if has_t else 0, ref_dim, int(temporal_ref_mode), _DTYPES[value.dtype],
            torch.cuda.current_stream().cuda_stream))
    return (out,) + tuple(value.new_empty(0, dtype=torch.float32) if x is None else x for x in samp)


@_fused_op.register_fake
def _(value, ref, off_curr, logit_curr, off_temporal, logit_temporal, spatial_shapes, level_start_index,
      temporal_spatial_shapes, temporal_level_start_index, temporal_offsets, frame_offsets, query_order, tile_h, tile_w,
      temporal_ref_mode, want_sampling, padding_mask, check_levels):
    t, _, m, d = value.shape
    lq, nl, pc = off_curr.shape[1], off_curr.shape[3], off_curr.shape[4]
    has_t = _wt(temporal_offsets, frame_offsets, t) > 0 and off_temporal is not None
    f32 = lambda shape: value.new_empty(shape, dtype=torch.float32)
    samp = [f32(0) for _ in range(4)]
    if want_sampling:
        samp[0], samp[1] = f32(tuple(off_curr.shape)), f32((t, lq, m, nl, pc))
        if has_t:
            samp[2], samp[3] = f32(tuple(off_temporal.shape)), f32(tuple(off_temporal.shape[:5]))
    return (value.new_empty((t, lq, m * d)),) + tuple(samp)


@torch.library.custom_op("devis::tmsda_fused_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _fused_backward_op(grad_output: Tensor, value: Tensor, ref: Tensor, off_curr: Tensor, logit_curr: Tensor,
                       off_temporal: OptTensor, logit_temporal: OptTensor, spatial_shapes: Tensor,
                       level_start_index: Tensor, temporal_offsets: Tensors, frame_offsets: list[int], query_order: OptTensor, tile_h: int,
                       tile_w: int, temporal_ref_mode: int, padding_mask: OptTensor, need_grad_value: bool,
                       need_grad_ref: bool) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """(grad_value, grad_ref, grad_off_curr, grad_logit_curr, grad_off_temporal, grad_logit_temporal), each in its
    input's dtype; an empty tensor stands for a gradient that is not computed"""
    geometry = clip_geometry.op_geometry(value.shape[0], spatial_shapes, level_start_index, None, None,
                                         temporal_offsets, frame_offsets)
    in_dtypes = (off_curr.dtype, logit_curr.dtype, off_temporal.dtype if off_temporal is not None else None,
                 logit_temporal.dtype if logit_temporal is not None else None, ref.dtype)
    value = value if value.is_contiguous() else value.contiguous()
    ref, oc, lc = _f32(ref), _f32(off_curr), _f32(logit_curr)
    has_t = geometry.t_window > 0 and off_temporal is not None
    ot = _f32(off_temporal) if has_t else None
    lt = _f32(logit_temporal) if has_t else None
    t, s, m, d = value.shape
    lq, pc = oc.shape[1], oc.shape[4]
    pt = ot.shape[4] if has_t else 0
    ref_dim = ref.shape[-1]
    if padding_mask is not None:
        padding_mask = padding_mask.detach().contiguous()
    query_order = _order(geometry, query_order, tile_h, tile_w, lq, value.device)
    gout = grad_output if grad_output.dtype == value.dtype else grad_output.to(value.dtype)
    gout = gout if gout.is_contiguous() else gout.contiguous()
    need_gv = need_grad_value
    need_gref = need_grad_ref
    half_acc = need_gv and MSDA.bf16_accumulate_enabled(value)
    det = MSDA.deterministic_enabled(value.dtype)
    if det and need_gref:
        raise RuntimeError("temporal_ms_deform_attn_fused: deterministic mode has no gradient for the reference points "
                           "(use the unfused path: TemporalMSDeformAttnFusedFunction.supported() says so)")
    gv = torch.empty(value.shape, dtype=value.dtype if half_acc else torch.float32, device=value.device) \
        if need_gv else None
    goc, glc = torch.empty_like(oc), torch.empty_like(lc)
    got = torch.empty_like(ot) if has_t else None
    glt = torch.empty_like(lt) if has_t else None
    gref = torch.empty_like(ref) if need_gref else None
    flags = (0 if need_gv else _lib.FLAG_NO_GRAD_VALUE) | (_lib.FLAG_BF16_GRAD_VALUE if half_acc else 0) | \
        (_lib.FLAG_DETERMINISTIC if det else 0)
    with torch.cuda.device(value.device):
        ws_bytes = _lib.load().devis_tmsda_fused_backward_workspace_bytes(t, s, m, d, flags)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=value.device) if ws_bytes else None
        _lib.check(_lib.load().devis_tmsda_fused_backward_ex(
            _ptr(value), geometry.shapes_ptr, geometry.lsi_ptr, geometry.frames_ptr, _ptr(ref), _ptr(oc), _ptr(lc),
            _ptr(ot), _ptr(lt), _ptr(gout), _ptr(gv), _ptr(goc), _ptr(glc), _ptr(got), _ptr(glt), _ptr(gref),
            _ptr(query_order), _ptr(padding_mask), t, s, m, d, geometry.n_levels, lq, pc, pt, geometry.t_window if has_t else 0,
            ref_dim, int(temporal_ref_mode), _DTYPES[value.dtype], flags, _ptr(ws), ws_bytes,
            torch.cuda.current_stream().cuda_stream))
    doc, dlc, dot, dlt, dref = in_dtypes
    if gv is not None and gv.dtype != value.dtype:
        gv = gv.to(value.dtype)
    cast = lambda g, dt: value.new_empty(0) if g is None else (g if g.dtype == dt else g.to(dt))
    return (cast(gv, value.dtype), cast(gref, dref), cast(goc, doc), cast(glc, dlc), cast(got, dot), cast(glt, dlt))


@_fused_backward_op.register_fake
def _(grad_output, value, ref, off_curr, logit_curr, off_temporal, logit_temporal, spatial_shapes, level_start_index,
      temporal_offsets, frame_offsets, query_order, tile_h, tile_w, temporal_ref_mode, padding_mask, need_grad_value,
      need_grad_ref):
    has_t = _wt(temporal_offsets, frame_offsets, value.shape[0]) > 0 and off_temporal is not None
    like = lambda x, on: torch.empty_like(x, memory_format=torch.contiguous_format) if on else value.new_empty(0)
    return (like(value, need_grad_value), like(ref, need_grad_ref), like(off_curr, True), like(logit_curr, True),
            like(off_temporal, has_t), like(logit_temporal, has_t))


def _fused_setup_context(ctx, inputs, output):
    (value, ref, off_curr, logit_curr, off_temporal, logit_temporal, shapes, lsi, _, _, offsets, frame_offsets,
     query_order, tile_h, tile_w, tref, want_sampling, padding_mask, _) = inputs
    ctx.args = (tile_h, tile_w, tref)
    ctx.frame_offsets = frame_offsets
    ctx.n_offsets = len(offsets)
    ctx.mark_non_differentiable(*output[1:])
    ctx.save_for_backward(value, ref, off_curr, logit_curr, off_temporal, logit_temporal, shapes, lsi, query_order,
                          padding_mask, *offsets)


def _fused_backward(ctx, grad_output, *_unused):
    value, ref, oc, lc, ot, lt, shapes, lsi, query_order, padding_mask, *offsets = ctx.saved_tensors
    tile_h, tile_w, tref = ctx.args
    gv, gref, goc, glc, got, glt = _fused_backward_op(
        grad_output, value, ref, oc, lc, ot, lt, shapes, lsi, offsets, ctx.frame_offsets, query_order, tile_h, tile_w,
        tref, padding_mask, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
    return (_none(gv), _none(gref), goc, glc, _none(got), _none(glt), None, None, None, None, [None] * ctx.n_offsets,
            _no_grad_list(ctx.frame_offsets), None, None, None, None, None, None, None)


_fused_op.register_autograd(_fused_backward, setup_context=_fused_setup_context)


class TemporalMSDeformAttnFusedFunction:
    """apply(value, ref, off_curr, logit_curr, off_temporal, logit_temporal, geometry, query_order=None,
             temporal_ref_mode=TREF_LEVEL0, want_sampling=False, padding_mask=None) -> out (T, Lq, M*D)
                                                           | (out, loc_curr, aw_curr, loc_temporal, aw_temporal)

    Whole-clip temporal attention straight from the Linear outputs: the joint softmax over all taps and the sampling
    location arithmetic (encoder: ms_deform_attn.py:240-260, 437-452; decoder: :320-404, points or boxes, instance
    aware or not) happen inside the kernels, and the backward returns the gradients of the raw offsets and logits (and of
    the reference points when they require grad).  value (T,S,M,32) fp32|bf16|fp16; ref (T,Lq,L,2|4); off_curr
    (T,Lq,M,L,Pc,2); logit_curr (T,Lq,M,L*Pc); off_temporal (T,Lq,M,Wt*L,Pt,2); logit_temporal (T,Lq,M,Wt*L*Pt).
    temporal_ref_mode: _lib.TREF_LEVEL0 (encoder) | TREF_OWN | TREF_SAMPLED (decoder, instance aware).
    want_sampling: also return the sampling locations and softmax weights the kernel computed (non-differentiable
    by-products: what TemporalMSDeformAttnDecoder.forward hands to visualize_att_maps.py).
    padding_mask: optional CUDA bool (or uint8) tensor (T, S), True = padding.  Equivalent to
    value.masked_fill(padding_mask[..., None], 0) before the op, NaN / Inf in masked rows included; no gradient.
    MSDeformAttn passes its input_padding_mask here (its batch is the frame axis).  Entry point of the op
    ``devis::tmsda_fused`` (once differentiable)."""

    @staticmethod
    def supported(value, reference_points, n_curr_points=4, n_temporal_points=4):
        """`value`: the projected value tensor (T,S,M,D) (or any tensor with its device, dtype and shape)"""
        return (value.is_cuda and value.dtype in (torch.float32,) + _16BIT and value.shape[-1] == 32
                and n_curr_points % 4 == 0 and n_temporal_points % 4 == 0
                and reference_points.shape[-1] in (2, 4) and value.numel() * value.element_size() < (1 << 31)
                # deterministic mode: grad_value goes through fixed point inside the kernel; d/d(reference points) is a
                # float-atomic sum there, so learnable reference points take the unfused path in that mode
                and not (MSDA.deterministic_enabled(value.dtype) and reference_points.requires_grad))

    @staticmethod
    def apply(value, ref, off_curr, logit_curr, off_temporal, logit_temporal, geometry, query_order=None,
              temporal_ref_mode=_lib.TREF_LEVEL0, want_sampling=False, padding_mask=None):
        shapes, lsi, offsets = geometry.op_args()
        res = _fused_op(value, ref, off_curr, logit_curr, off_temporal, logit_temporal, shapes, lsi, None, None,
                        [], offsets, query_order, 0, 0, int(temporal_ref_mode), bool(want_sampling), padding_mask,
                        False)
        if not want_sampling:
            return res[0]
        has_t = geometry.t_window > 0 and off_temporal is not None
        return res if has_t else res[:3]


def temporal_ms_deform_attn(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None):
    return TemporalMSDeformAttnFunction.apply(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry,
                                              query_order)
