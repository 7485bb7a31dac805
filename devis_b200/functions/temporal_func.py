"""Whole-clip temporal multi-scale deformable attention as ONE autograd op.

The reference computes a layer's temporal attention with a Python loop over the T query frames:
per frame one ``MSDeformAttnFunction.apply`` on the frame's own value, a gather copy
``value[temporal_frames].flatten(0, 1)``, a second ``apply`` on that copy with the temporal frames
stacked along the level axis, and an add (modules/ms_deform_attn.py:435-460 encoder, :325-404
decoder) -- 2T launches, T copies and 2T materialised outputs forward, the same again backward.
``TemporalMSDeformAttnFunction`` does the whole clip in one launch each way: value (T,S,M,D) is read
in place through the frame table, current and temporal taps accumulate into the same registers, and
the backward scatters straight into grad_value (T,S,M,D) -- no copies, no index_add.
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import _lib
from .. import MultiScaleDeformableAttention as MSDA

# float16 value (what torch.autocast("cuda") hands the op by default) is served like bfloat16: 16-bit value, output and
# grad_output, float32 locations, weights and gradients
_DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
_16BIT = (torch.bfloat16, torch.float16)


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def _aux(t, value):
    want = torch.float32 if value.dtype in _16BIT else value.dtype
    t = t if t.dtype == want else t.to(want)
    return t if t.is_contiguous() else t.contiguous()


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


class TemporalMSDeformAttnFunction(Function):
    """apply(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None) -> (T, Lq, M*D)

    value (T,S,M,D); loc_curr (T,Lq,M,L,Pc,2); aw_curr (T,Lq,M,L,Pc); loc_temporal (T,Lq,M,Wt*L,Pt,2);
    aw_temporal (T,Lq,M,Wt*L,Pt) -- exactly the tensors the reference's per-frame loop slices
    (ms_deform_attn.py:437-457); geometry is a devis_b200.clip_geometry.ClipGeometry."""

    @staticmethod
    def forward(ctx, value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None):
        if not value.is_cuda:
            raise RuntimeError("Not implemented on the CPU")
        if value.dtype not in _DTYPES:
            raise RuntimeError(f'"temporal_ms_deform_attn" not implemented for \'{value.dtype}\'')
        value = value if value.is_contiguous() else value.contiguous()
        lc, ac = _aux(loc_curr, value), _aux(aw_curr, value)
        has_t = geometry.t_window > 0 and loc_temporal is not None
        lt = _aux(loc_temporal, value) if has_t else None
        at = _aux(aw_temporal, value) if has_t else None
        t, s, m, d, lq, pc, pt = _dims(value, lc, lt, geometry)
        out = torch.empty((t, lq, m * d), dtype=value.dtype, device=value.device)
        with torch.cuda.device(value.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(_lib.load().devis_tmsda_forward(
                _ptr(value), geometry.shapes_ptr, geometry.lsi_ptr, geometry.frames_ptr,
                _ptr(lc), _ptr(ac), _ptr(lt), _ptr(at), _ptr(out), _ptr(query_order),
                t, s, m, d, geometry.n_levels, lq, pc, pt, geometry.t_window if has_t else 0,
                _DTYPES[value.dtype], stream))
        ctx.geometry = geometry
        ctx.has_t = has_t
        ctx.in_dtypes = (loc_curr.dtype, aw_curr.dtype,
                         loc_temporal.dtype if has_t else None, aw_temporal.dtype if has_t else None)
        ctx.save_for_backward(value, lc, ac, lt, at, query_order)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, lc, ac, lt, at, query_order = ctx.saved_tensors
        geometry, has_t = ctx.geometry, ctx.has_t
        t, s, m, d, lq, pc, pt = _dims(value, lc, lt, geometry)
        gout = grad_output if grad_output.dtype == value.dtype else grad_output.to(value.dtype)
        gout = gout if gout.is_contiguous() else gout.contiguous()
        need_gv = ctx.needs_input_grad[0]
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
        dl, da, dlt, dat = ctx.in_dtypes
        if gv is not None and gv.dtype != value.dtype:
            gv = gv.to(value.dtype)
        glc = glc if glc.dtype == dl else glc.to(dl)
        gac = gac if gac.dtype == da else gac.to(da)
        if has_t:
            glt = glt if glt.dtype == dlt else glt.to(dlt)
            gat = gat if gat.dtype == dat else gat.to(dat)
        return gv, glc, gac, glt, gat, None, None


class TemporalMSDeformAttnFusedFunction(Function):
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
    MSDeformAttn passes its input_padding_mask here (its batch is the frame axis)."""

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
    def forward(ctx, value, ref, off_curr, logit_curr, off_temporal, logit_temporal, geometry, query_order=None,
                temporal_ref_mode=_lib.TREF_LEVEL0, want_sampling=False, padding_mask=None):
        if not value.is_cuda:
            raise RuntimeError("Not implemented on the CPU")
        if value.dtype not in (torch.float32,) + _16BIT:
            raise RuntimeError(f'"temporal_ms_deform_attn_fused" not implemented for \'{value.dtype}\'')
        f32 = lambda t: (t if t.dtype == torch.float32 else t.float()).contiguous()
        value = value if value.is_contiguous() else value.contiguous()
        ref_in_dtype = ref.dtype
        ref, oc, lc = f32(ref), f32(off_curr), f32(logit_curr)
        has_t = geometry.t_window > 0 and off_temporal is not None
        ot = f32(off_temporal) if has_t else None
        lt = f32(logit_temporal) if has_t else None
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
        ctx.geometry, ctx.has_t, ctx.tref = geometry, has_t, int(temporal_ref_mode)
        ctx.dims = (t, s, m, d, lq, pc, pt, ref_dim)
        ctx.in_dtypes = (off_curr.dtype, logit_curr.dtype, off_temporal.dtype if has_t else None,
                         logit_temporal.dtype if has_t else None, ref_in_dtype)
        ctx.save_for_backward(value, ref, oc, lc, ot, lt, query_order, padding_mask)
        if not want_sampling:
            return out
        extras = tuple(x for x in samp if x is not None)
        ctx.mark_non_differentiable(*extras)
        ctx.n_extras = len(extras)
        return (out,) + extras

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output, *_unused):
        value, ref, oc, lc, ot, lt, query_order, padding_mask = ctx.saved_tensors
        geometry, has_t = ctx.geometry, ctx.has_t
        t, s, m, d, lq, pc, pt, ref_dim = ctx.dims
        gout = grad_output if grad_output.dtype == value.dtype else grad_output.to(value.dtype)
        gout = gout if gout.is_contiguous() else gout.contiguous()
        need_gv = ctx.needs_input_grad[0]
        need_gref = ctx.needs_input_grad[1]
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
                ref_dim, ctx.tref, _DTYPES[value.dtype], flags, _ptr(ws), ws_bytes,
                torch.cuda.current_stream().cuda_stream))
        doc, dlc, dot, dlt, dref = ctx.in_dtypes
        if gv is not None and gv.dtype != value.dtype:
            gv = gv.to(value.dtype)
        cast = lambda g, dt: g if (g is None or g.dtype == dt) else g.to(dt)
        return (gv, cast(gref, dref), cast(goc, doc), cast(glc, dlc), cast(got, dot), cast(glt, dlt), None, None, None,
                None, None)


def temporal_ms_deform_attn(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry, query_order=None):
    return TemporalMSDeformAttnFunction.apply(value, loc_curr, aw_curr, loc_temporal, aw_temporal, geometry,
                                              query_order)
