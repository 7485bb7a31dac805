"""Drop-in for the reference's compiled extension module ``MultiScaleDeformableAttention``
(built from src/models/ops/src/vision.cpp:13-16): same two functions, same argument order, same
return values, same error behaviour -- implemented as a thin shim that checks the tensors like
cuda/ms_deform_attn_cuda.cu:28-52,93-119 does, allocates the outputs and hands raw pointers plus the
current CUDA stream to the C-ABI library.

``import devis_b200.MultiScaleDeformableAttention as MSDA`` can replace
``import MultiScaleDeformableAttention as MSDA`` in functions/ms_deform_attn_func.py:18.

The two functions are the torch.library custom ops ``devis::ms_deform_attn`` / ``devis::ms_deform_attn_backward``
(the forward op carries the autograd formula of MSDeformAttnFunction), so torch.compile and torch.export trace the op
as one node.  Every op of this package is tagged ``needs_exact_strides``: a compiled graph hands it its operands in the
layout eager code would, which is what the contiguity checks below expect.
"""
import torch

from . import _lib

_DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.bfloat16: _lib.BF16}

# process-wide default for the backward mode; see set_deterministic()
_deterministic = False


def set_deterministic(flag):
    """Select the bit-reproducible grad_value accumulation (the reference's float atomicAdd scatter is
    run-to-run non-deterministic; SURVEY.md section 5).  Also switched on by
    torch.use_deterministic_algorithms(True)."""
    global _deterministic
    _deterministic = bool(flag)


def deterministic_enabled(value_dtype=None):
    on = _deterministic or torch.are_deterministic_algorithms_enabled()
    return on and value_dtype != torch.float64      # fp64 keeps native double atomics (gradcheck path)


# process-wide switch for the bf16 grad_value accumulation; see set_bf16_grad_value_accumulation()
_bf16_accumulate = False


def set_bf16_grad_value_accumulation(flag):
    """bf16 value only.  False (default): grad_value is accumulated in float32 and rounded to bf16 once.  True: the
    scatter adds straight into a bf16 grad_value with packed bf16 reductions (DEVIS_MSDA_FLAG_BF16_GRAD_VALUE) --
    half the bytes leave the SM, which is what bounds the backward, at the precision of PyTorch's own bf16
    atomicAdd scatters (every partial sum rounds to bf16).  Ignored in deterministic mode and for head dims other
    than 16 / 32."""
    global _bf16_accumulate
    _bf16_accumulate = bool(flag)


def bf16_accumulate_enabled(value):
    return (_bf16_accumulate and value.dtype == torch.bfloat16 and value.shape[-1] in (16, 32)
            and value.numel() * 2 < (1 << 32) and not deterministic_enabled(value.dtype))


def _check(named, like=None):
    for name, t in named:
        if not t.is_contiguous():
            raise RuntimeError(f"{name} tensor has to be contiguous")
    for name, t in named:
        if not t.is_cuda:
            if name == "value":
                raise RuntimeError("Not implemented on the CPU")
            raise RuntimeError(f"{name} must be a CUDA tensor")


def _dtype_code(value):
    try:
        return _DTYPES[value.dtype]
    except KeyError:
        raise RuntimeError(f'"ms_deform_attn" not implemented for \'{value.dtype}\'') from None


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def _aux(t, value):
    """sampling locations / attention weights in the dtype the kernels read: value's dtype for
    fp32/fp64, float32 next to a bf16 value."""
    want = torch.float32 if value.dtype == torch.bfloat16 else value.dtype
    return t if t.dtype == want else t.to(want)


def _level_area(spatial_shapes):
    """sum of H*W over the levels, from the memoised host copy (one synchronising read per tensor object)"""
    from .clip_geometry import host_list
    return sum(int(h) * int(w) for h, w in host_list(spatial_shapes))


@torch.library.custom_op("devis::ms_deform_attn", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _forward_op(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
                sampling_loc: torch.Tensor, attn_weight: torch.Tensor, im2col_step: int,
                check_levels: bool) -> torch.Tensor:
    """vision.cpp:14 / ms_deform_attn.h:20-39.  Returns (N, Lq, M*D) in value's dtype.  ``check_levels``: MSDeformAttn's
    ``sum(H*W) == S`` assertion (ms_deform_attn.py:95), made here where the pyramid's host copy is read."""
    if not value.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    _check([("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
            ("sampling_loc", sampling_loc), ("attn_weight", attn_weight)])
    code = _dtype_code(value)
    n, s, m, d = value.shape
    if check_levels:
        assert _level_area(spatial_shapes) == s
    nl = spatial_shapes.shape[0]
    lq, p = sampling_loc.shape[1], sampling_loc.shape[4]
    step = min(n, int(im2col_step)) if n > 0 else 1
    if n > 0 and n % step != 0:
        raise RuntimeError(f"batch({n}) must divide im2col_step({step})")
    loc, aw = _aux(sampling_loc, value), _aux(attn_weight, value)
    shapes = spatial_shapes.to(torch.int64) if spatial_shapes.dtype != torch.int64 else spatial_shapes
    lsi = level_start_index.to(torch.int64) if level_start_index.dtype != torch.int64 else level_start_index
    out = torch.empty((n, lq, m * d), dtype=value.dtype, device=value.device)
    with torch.cuda.device(value.device):
        stream = torch.cuda.current_stream().cuda_stream
        _lib.check(_lib.load().devis_msda_forward(
            _ptr(value), _ptr(shapes), _ptr(lsi), _ptr(loc), _ptr(aw), _ptr(out),
            n, s, m, d, nl, lq, p, max(int(im2col_step), 1), code, stream))
    return out


@_forward_op.register_fake
def _(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step, check_levels):
    n, _, m, d = value.shape
    return value.new_empty((n, sampling_loc.shape[1], m * d))


@torch.library.custom_op("devis::ms_deform_attn_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _backward_op(grad_output: torch.Tensor, value: torch.Tensor, spatial_shapes: torch.Tensor,
                 level_start_index: torch.Tensor, sampling_loc: torch.Tensor, attn_weight: torch.Tensor,
                 im2col_step: int, need_grad_value: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """vision.cpp:15 / ms_deform_attn.h:41-61.  Returns (grad_value, grad_sampling_loc, grad_attn_weight);
    grad_value is an empty tensor when ``need_grad_value`` is False (the scatter is skipped)."""
    if not value.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    _check([("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
            ("sampling_loc", sampling_loc), ("attn_weight", attn_weight), ("grad_output", grad_output)])
    code = _dtype_code(value)
    n, s, m, d = value.shape
    nl = spatial_shapes.shape[0]
    lq, p = sampling_loc.shape[1], sampling_loc.shape[4]
    step = min(n, int(im2col_step)) if n > 0 else 1
    if n > 0 and n % step != 0:
        raise RuntimeError(f"batch({n}) must divide im2col_step({step})")
    loc, aw = _aux(sampling_loc, value), _aux(attn_weight, value)
    gout = grad_output if grad_output.dtype == value.dtype else grad_output.to(value.dtype)
    shapes = spatial_shapes.to(torch.int64) if spatial_shapes.dtype != torch.int64 else spatial_shapes
    lsi = level_start_index.to(torch.int64) if level_start_index.dtype != torch.int64 else level_start_index
    half_acc = need_grad_value and bf16_accumulate_enabled(value)
    acc_dtype = torch.float32 if (value.dtype == torch.bfloat16 and not half_acc) else value.dtype
    grad_value = torch.empty(value.shape, dtype=acc_dtype, device=value.device) if need_grad_value else None
    grad_loc = torch.empty_like(loc)
    grad_aw = torch.empty_like(aw)
    flags = (_lib.FLAG_DETERMINISTIC if deterministic_enabled(value.dtype) else 0) | \
        (0 if need_grad_value else _lib.FLAG_NO_GRAD_VALUE) | (_lib.FLAG_BF16_GRAD_VALUE if half_acc else 0)
    lib = _lib.load()
    with torch.cuda.device(value.device):
        stream = torch.cuda.current_stream().cuda_stream
        ws_bytes = lib.devis_msda_backward_workspace_bytes(n, s, m, d, nl, lq, p, code, flags)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=value.device) if ws_bytes else None
        _lib.check(lib.devis_msda_backward(
            _ptr(value), _ptr(shapes), _ptr(lsi), _ptr(loc), _ptr(aw), _ptr(gout),
            _ptr(grad_value), _ptr(grad_loc), _ptr(grad_aw),
            n, s, m, d, nl, lq, p, max(int(im2col_step), 1), code, flags, _ptr(ws), ws_bytes, stream))
    if grad_value is None:
        grad_value = value.new_empty(0)
    elif grad_value.dtype != value.dtype:
        grad_value = grad_value.to(value.dtype)
    if grad_loc.dtype != sampling_loc.dtype:
        grad_loc = grad_loc.to(sampling_loc.dtype)
    if grad_aw.dtype != attn_weight.dtype:
        grad_aw = grad_aw.to(attn_weight.dtype)
    return grad_value, grad_loc, grad_aw


@_backward_op.register_fake
def _(grad_output, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step, need_grad_value):
    return (value.new_empty(value.shape if need_grad_value else (0,)), torch.empty_like(sampling_loc),
            torch.empty_like(attn_weight))


def _setup_context(ctx, inputs, output):
    value, shapes, lsi, loc, aw, im2col_step, _ = inputs
    ctx.im2col_step = im2col_step
    ctx.save_for_backward(value, shapes, lsi, loc, aw)


def _backward(ctx, grad_output):
    """once differentiable, like the reference's Function (functions/ms_deform_attn_func.py:30-38)"""
    value, shapes, lsi, loc, aw = ctx.saved_tensors
    need_gv, need_loc, need_aw = ctx.needs_input_grad[0], ctx.needs_input_grad[3], ctx.needs_input_grad[4]
    if not (need_gv or need_loc or need_aw):
        return None, None, None, None, None, None, None
    grad_value, grad_loc, grad_aw = _backward_op(grad_output.contiguous(), value, shapes, lsi, loc, aw,
                                                 ctx.im2col_step, need_gv)
    return (grad_value if need_gv else None), None, None, grad_loc, grad_aw, None, None


_forward_op.register_autograd(_backward, setup_context=_setup_context)


def ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    """vision.cpp:14 / ms_deform_attn.h:20-39.  Returns (N, Lq, M*D) in value's dtype (op ``devis::ms_deform_attn``)."""
    return _forward_op(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, int(im2col_step), False)


def ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output,
                            im2col_step, need_grad_value=True):
    """vision.cpp:15 / ms_deform_attn.h:41-61.  Returns [grad_value, grad_sampling_loc, grad_attn_weight].
    ``need_grad_value=False`` (extension, used by the autograd formula when value is frozen) skips the scatter and
    returns None in its place."""
    grad_value, grad_loc, grad_aw = _backward_op(grad_output, value, spatial_shapes, level_start_index, sampling_loc,
                                                 attn_weight, int(im2col_step), bool(need_grad_value))
    return [grad_value if need_grad_value else None, grad_loc, grad_aw]
