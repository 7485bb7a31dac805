"""Modulated deformable convolution for DeVIS's mask head: ``deform_conv2d`` with torchvision's signature.

The reference calls ``torchvision.ops.deform_conv2d(input, offset, weight, bias, padding=..., mask=...)`` in
ModulatedDeformableConv2d.forward (src/models/deformable_segmentation.py:262-267).  torchvision's operator
(torchvision/ops/deform_conv.py:14-99, C++ vision::ops::deform_conv2d) computes

    out[n, co, y, x] = bias[co] + sum_{ci, k} weight[co, ci, k] * mask[n, k, y, x] *
                       bilinear(input[n, ci], y*stride - pad + ky*dil + offset[n, 2k, y, x],
                                               x*stride - pad + kx*dil + offset[n, 2k+1, y, x])

with zero padding.  With G offset groups (``offset`` of 2 * G * kh * kw channels, ``mask`` of G * kh * kw) input channel
ci belongs to group g = ci // (Cin / G), and its samples use ``offset[n, 2 * (g * kh * kw + k) (+1)]`` and
``mask[n, g * kh * kw + k]``.  Here the gather (and, backward, the scatter plus the offset / mask gradients) are the hand-written
sm_100a kernels behind ``devis_dcn_im2col`` / ``devis_dcn_col2im`` (include/devis_deform_conv.h,
devis_b200/csrc/deform_conv.cuh); the contractions with ``weight`` are cuBLAS GEMMs, as in torchvision (at::addmm).
The input is read channels-last: pass a ``torch.channels_last`` tensor to avoid the layout copy; the result is returned
as an NCHW view of a channels-last buffer.

Two forms (both hand-written kernels of this library, chosen per layer by ``devis_dcn_fused_form``):
  * fused  -- float32, Cin % 4 == 0, few output channels (the high-resolution half of the mask head; exact rule:
              devis_dcn_fused_form): gather and contraction in ONE kernel, the column matrix (9x the input) is never
              written; backward = one kernel for the data gradients when Cout <= 16 (no grad_cols either; wider layers
              take the grad_cols GEMM + scatter kernel) + the weight gradient from columns recomputed in bounded chunks,
              so nothing of column size is kept between forward and backward;
  * im2col -- everything else: column matrix + cuBLAS GEMM, as torchvision does.
``set_fused(False)`` forces the im2col form (A/B tests).  The wide layers' forward runs on the tensor cores
(IGemmDeformConv2dFunction) and the narrow layers' weight gradient in one kernel (devis_dcn_weight_grad); both serve one
offset group only, so with G > 1 those layers take the im2col form and the weight gradient takes the GEMM on recomputed
columns.  The lane-group fused kernels serve G > 1 when (Cin / G) % 4 == 0 (devis_dcn_fused_form_og).

Supported: groups == 1, any offset_groups, float32 / float64 (half and bfloat16 are computed in float32 like
torchvision's autocast wrapper does), CUDA only -- there is no CPU fallback.

Each form is a ``torch.library`` custom op (``devis::deform_conv2d_{im2col,fused,igemm}`` and their ``*_backward``), so
torch.compile and torch.export trace a layer as one node; the choice of form stays in ``deform_conv2d`` (traceable
Python: grad mode, requires_grad, allow_tf32, the deterministic flag and the library's shape rules).  A forward op
returns what its backward needs besides its inputs as extra outputs: the channels-last copy of the input (empty when the
input is channels-last already, the backward then reads the input itself), the im2col form's columns, the fused form's
packed weight -- exactly what the backward kept before.
"""

import warnings
from typing import Optional

import torch
from torch.nn.modules.utils import _pair

from . import _lib

_DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def _out_size(size, k, stride, pad, dil):
    return (size + 2 * pad - (dil * (k - 1) + 1)) // stride + 1


_FUSED = True
_warned_nondeterministic = False


def _alert_not_deterministic():
    """float64 grad_input is scattered with float atomics: the sum order, hence the last bits, change from run to run
    (the fixed-point form of _grad_input_flags is float32 only).  Under ``torch.use_deterministic_algorithms(True)`` say
    so, the way ATen's non-deterministic kernels do (error, or a warning in warn_only mode)."""
    global _warned_nondeterministic
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = ("devis_b200.deform_conv2d backward does not have a deterministic implementation for float64 grad_input "
           "(float atomic scatter), but you set 'torch.use_deterministic_algorithms(True)'")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        if not _warned_nondeterministic:
            warnings.warn(msg, stacklevel=3)
            _warned_nondeterministic = True
        return
    raise RuntimeError(msg + ". You can turn off determinism just for this operation, or use warn_only=True.")
_COLS_CHUNK_BYTES = 256 << 20          # recomputed columns per weight-gradient chunk
_DET_ACC_CHUNK_BYTES = 256 << 20       # 64-bit grad_input accumulators per deterministic data-backward call


def _grad_input_flags(dtype):
    """backward flags of the grad_input scatter.  Under ``torch.use_deterministic_algorithms(True)`` float32 takes the
    64-bit fixed-point form (DEVIS_MSDA_FLAG_DETERMINISTIC: bit-identical run to run); float64 has none (2^-36 of the
    largest contribution is coarser than float64 accumulation) and raises torch's alert instead."""
    if not torch.are_deterministic_algorithms_enabled():
        return 0
    if dtype == torch.float32:
        return _lib.FLAG_DETERMINISTIC
    _alert_not_deterministic()
    return 0


def _data_chunk(n, h, w, c, flags, per):
    """batch items per data-backward call: ``per`` (the caller's bound), and with the fixed-point form at most
    _DET_ACC_CHUNK_BYTES of accumulators (8 B per input element; 6.6 GB for 1800 instances of a 32-channel 90 x 160 map).
    Each call has its own fixed-point scale, which depends on the shapes and the values only."""
    if flags:
        per = min(per, _DET_ACC_CHUNK_BYTES // max(1, h * w * c * 8))
    return max(1, min(n, per))


def _workspace(lib, per, h, w, c, flags, device):
    """(workspace, bytes) of a data-backward call over ``per`` batch items"""
    nbytes = int(lib.devis_dcn_backward_workspace_bytes(per, h, w, c, flags))
    return (torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes) if nbytes else (None, 0)


def _wgrad(g2, cols):
    """grad_out^T x columns: (rows, Cout)^T x (rows, K*C) -> (Cout, K*C).  The reduction runs over rows = N*Ho*Wo
    (10^5 .. 10^6) while the product is tiny for the narrow mask-head layers; as ONE GEMM cuBLAS picks sgemm_largek
    and runs at 4 TFLOP/s (512 us for 16 x 216000 x 288, `benchmarks/dcn_profile.py`).  Independent row slabs as a
    batched GEMM + a sum of the partial products read the columns at memory speed instead."""
    rows, cout = g2.shape
    kc = cols.shape[1]
    slab = 2048
    if cout > 1 and cout * kc <= (1 << 17) and rows >= 8 * slab:
        s = rows // slab
        main = s * slab
        out = torch.bmm(g2[:main].view(s, slab, cout).transpose(1, 2), cols[:main].view(s, slab, kc)).sum(0)
        if main < rows:
            out.addmm_(g2[main:].t(), cols[main:rows])
        return out
    return g2.t() @ cols[:rows]


def set_fused(enabled):
    """enable / disable the fused gather+contraction kernels (default on); returns the previous setting"""
    global _FUSED
    old, _FUSED = _FUSED, bool(enabled)
    return old


@torch.compiler.assume_constant_result
def _library_fused_form(c, cout, kh, kw, offset_groups):
    """the library's shape rule (a pure function of the ints): a constant to torch.compile, not a graph break"""
    return int(_lib.load().devis_dcn_fused_form_og(c, cout, kh, kw, offset_groups, _lib.F32))


def _fused_form(c, cout, kh, kw, dtype, offset_groups=1):
    """bit 0: fused forward kernel serves the layer, bit 1: fused data-backward kernel does (devis_dcn_fused_form_og)"""
    if not _FUSED or dtype != torch.float32:
        return 0
    return _library_fused_form(int(c), int(cout), int(kh), int(kw), int(offset_groups))


@torch.compiler.assume_constant_result
def _packed_weight_elems(c, cout, kh, kw, offset_groups):
    """floats of the fused kernels' weight layout for the layer (the library's rule; a constant to torch.compile)"""
    return int(_lib.load().devis_dcn_packed_weight_elems_og(c, cout, kh, kw, offset_groups))


def _offset_groups(offset, kh, kw):
    return offset.shape[1] // (2 * kh * kw)


def _packed_weight(weight, offset_groups=1):
    """weight (Cout, Cin, kh, kw) in the layout the fused kernels read.  Repacked on EVERY call: one small kernel over
    <= 100 KB for the layers the fused form serves.  (Round 1 cached the packed copy per tensor object and ``_version``;
    writes through ``Parameter.data`` -- ``nn.Module.to()``, EMA / weight-swap code -- do not bump ``_version``, so the
    fused path could run with stale weights, or with a pointer on the wrong device after ``model.to('cuda:1')``.)"""
    cout, c, kh, kw = weight.shape
    lib = _lib.load()
    w = weight.detach()
    w = w if w.is_contiguous() else w.contiguous()
    packed = torch.empty(int(lib.devis_dcn_packed_weight_elems_og(c, cout, kh, kw, offset_groups)), dtype=torch.float32,
                         device=weight.device)
    with torch.cuda.device(weight.device):
        _lib.check(lib.devis_dcn_pack_weight_og(_ptr(w), _ptr(packed), c, cout, kh, kw, offset_groups,
                                                torch.cuda.current_stream().cuda_stream))
    return packed


OptTensor = Optional[torch.Tensor]


def _nhwc(input):
    """(input read channels-last, the copy to keep for the backward): an empty tensor when no copy was made (the
    backward then permutes the input again, which costs nothing)"""
    x = input.permute(0, 2, 3, 1)
    if x.is_contiguous():
        return x, input.new_empty(0)
    x = x.contiguous()
    return x, x


def _saved_nhwc(input, x_copy):
    return x_copy if x_copy.dim() == 4 else input.permute(0, 2, 3, 1)


def _contig(t):
    return t if t is None or t.is_contiguous() else t.contiguous()


def _fake_forward(input, offset, weight, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w):
    """(NCHW view of a channels-last output, the channels-last input copy or an empty tensor) as the forms return them"""
    n, c, h, w = input.shape
    cout, _, kh, kw = weight.shape
    ho, wo = _out_size(h, kh, stride_h, pad_h, dil_h), _out_size(w, kw, stride_w, pad_w, dil_w)
    out = input.new_empty((n, ho, wo, cout)).permute(0, 3, 1, 2)
    x_copy = input.new_empty(0) if input.permute(0, 2, 3, 1).is_contiguous() else input.new_empty((n, h, w, c))
    return out, x_copy


def _fake_backward(input, offset, weight, bias, mask, need_in, need_off, need_w, need_b, need_m):
    """gradients as the backward ops return them: grad_input and grad_weight are NCHW views of channels-last buffers,
    an empty tensor stands for one that is not computed (the offset and mask gradients come with the data backward)"""
    n, c, h, w = input.shape
    cout, _, kh, kw = weight.shape
    empty = lambda: input.new_empty(0)
    data = need_in or need_off or (need_m and mask is not None)
    like = lambda t: torch.empty_like(t, memory_format=torch.contiguous_format)
    grad_in = input.new_empty((n, h, w, c)).permute(0, 3, 1, 2) if need_in else empty()
    grad_off = like(offset) if data else empty()
    grad_w = input.new_empty((cout, kh, kw, c)).permute(0, 3, 1, 2) if need_w else empty()
    grad_b = input.new_empty((cout,)) if need_b and bias is not None else empty()
    grad_m = like(mask) if data and mask is not None else empty()
    return grad_in, grad_off, grad_w, grad_b, grad_m


def _needs(ctx):
    """(need_in, need_off, need_w, need_b, need_m)"""
    return tuple(ctx.needs_input_grad[:5])


def _autograd_result(grads, n_args):
    """backward-op results -> autograd's: None for the empty placeholders and for the non-tensor arguments"""
    return tuple(None if g.numel() == 0 and g.dim() == 1 else g for g in grads) + (None,) * n_args


# ------------------------------------------------------------------------------------------------------------------------
# fused form: gather and contraction in one kernel
# ------------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("devis::deform_conv2d_fused", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _fused_op(input: torch.Tensor, offset: torch.Tensor, weight: torch.Tensor, bias: OptTensor, mask: OptTensor,
              stride_h: int, stride_w: int, pad_h: int, pad_w: int, dil_h: int, dil_w: int,
              packed_elems: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(out (N, Cout, Ho, Wo), channels-last input copy or empty, packed weight of ``packed_elems`` floats: the
    library's size for the layer, _packed_weight_elems)"""
    if not input.is_cuda:
        raise RuntimeError("deform_conv2d: not implemented on the CPU (no fallback in this library)")
    n, c, h, w = input.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    x, x_copy = _nhwc(input)
    offset, mask, bias = _contig(offset), _contig(mask), _contig(bias)
    og = _offset_groups(offset, kh, kw)
    packed = _packed_weight(weight) if og == 1 else _packed_weight(weight, og)   # G = 1: the hook's original signature
    if packed.numel() != packed_elems:
        raise RuntimeError(f"deform_conv2d: packed weight has {packed.numel()} elements, expected {packed_elems}")
    out = torch.empty((n, ho, wo, cout), dtype=input.dtype, device=input.device)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    with torch.cuda.device(input.device):
        _lib.check(_lib.load().devis_dcn_fused_forward_og(_ptr(x), _ptr(offset), _ptr(mask), _ptr(packed), _ptr(bias),
                                                          _ptr(out), *dims, og, cout,
                                                          torch.cuda.current_stream().cuda_stream))
    return out.permute(0, 3, 1, 2), x_copy, packed


@_fused_op.register_fake
def _(input, offset, weight, bias, mask, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, packed_elems):
    out, x_copy = _fake_forward(input, offset, weight, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w)
    return out, x_copy, input.new_empty((packed_elems,), dtype=torch.float32)


@torch.library.custom_op("devis::deform_conv2d_fused_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _fused_backward_op(grad_out: torch.Tensor, input: torch.Tensor, x_copy: torch.Tensor, offset: torch.Tensor,
                       weight: torch.Tensor, bias: OptTensor, mask: OptTensor, packed: torch.Tensor, stride_h: int,
                       stride_w: int, pad_h: int, pad_w: int, dil_h: int, dil_w: int, form: int, need_in: bool,
                       need_off: bool, need_w: bool, need_b: bool,
                       need_m: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(grad_input, grad_offset, grad_weight, grad_bias, grad_mask); ``form``: the forward's _fused_form"""
    x = _saved_nhwc(input, x_copy)
    offset, mask = _contig(offset), _contig(mask)
    n, h, w, c = x.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    k, og = kh * kw, _offset_groups(offset, kh, kw)
    g = grad_out.permute(0, 2, 3, 1)
    g = g if g.is_contiguous() else g.contiguous()                    # (N, Ho, Wo, Cout)
    grad_w = grad_b = grad_in = grad_off = grad_m = None
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    with torch.cuda.device(x.device):
        if need_in or need_off or (need_m and mask is not None):
            flags = _grad_input_flags(x.dtype) if need_in else 0
            gx = torch.empty_like(x, memory_format=torch.contiguous_format) if need_in else None
            grad_off = torch.empty_like(offset)
            grad_m = torch.empty_like(mask) if mask is not None else None
            if form & 2:
                per = _data_chunk(n, h, w, c, flags, n)
                ws, ws_bytes = _workspace(lib, per, h, w, c, flags, x.device)
                for n0 in range(0, n, per):
                    n1 = min(n, n0 + per)
                    _lib.check(lib.devis_dcn_fused_backward_og(
                        _ptr(x[n0:n1]), _ptr(offset[n0:n1]), _ptr(mask[n0:n1]) if mask is not None else None,
                        _ptr(packed), _ptr(g[n0:n1]), _ptr(gx[n0:n1]) if need_in else None, _ptr(grad_off[n0:n1]),
                        _ptr(grad_m[n0:n1]) if mask is not None else None, n1 - n0, *dims[1:], og, cout, flags,
                        _ptr(ws), ws_bytes, stream))
            else:
                # wider layers: column gradient by GEMM (a bounded chunk of the batch at a time) + scatter kernel
                w2 = weight.detach().permute(0, 2, 3, 1).reshape(cout, k * c)
                per = _data_chunk(n, h, w, c, flags, _COLS_CHUNK_BYTES // max(1, ho * wo * k * c * 4))
                ws, ws_bytes = _workspace(lib, per, h, w, c, flags, x.device)
                g2 = g.view(n * ho * wo, cout)
                for n0 in range(0, n, per):
                    n1 = min(n, n0 + per)
                    grad_cols = g2[n0 * ho * wo:n1 * ho * wo] @ w2
                    _lib.check(lib.devis_dcn_col2im_og(_ptr(x[n0:n1]), _ptr(offset[n0:n1]),
                                                       _ptr(mask[n0:n1]) if mask is not None else None, _ptr(grad_cols),
                                                       _ptr(gx[n0:n1]) if need_in else None, _ptr(grad_off[n0:n1]),
                                                       _ptr(grad_m[n0:n1]) if mask is not None else None, n1 - n0,
                                                       *dims[1:], og, _DTYPES[x.dtype], flags, _ptr(ws), ws_bytes,
                                                       stream))
            grad_in = gx.permute(0, 3, 1, 2) if need_in else None
        if need_w and og == 1 and x.dtype == torch.float32 and not torch.are_deterministic_algorithms_enabled() \
                and lib.devis_dcn_wgrad_supported(c, cout, kh, kw, _DTYPES[x.dtype]):
            # narrow layers: gather + contraction with grad_out in one kernel, no column matrix (dcn_wgrad_kernel,
            # one offset group only).  Its cross-block float atomics are order-dependent: under
            # torch.use_deterministic_algorithms the GEMM route below, deterministic like torchvision's, is taken.
            gw3 = torch.empty((cout, k, c), dtype=x.dtype, device=x.device)
            _lib.check(lib.devis_dcn_weight_grad(_ptr(x), _ptr(offset), _ptr(mask), _ptr(g), _ptr(gw3), *dims,
                                                 cout, stream))
            grad_w = gw3.view(cout, kh, kw, c).permute(0, 3, 1, 2)
        elif need_w:
            # cols^T x grad_out from columns recomputed a bounded chunk of the batch at a time
            per = max(1, min(n, _COLS_CHUNK_BYTES // max(1, ho * wo * k * c * 4)))
            cols = torch.empty((per * ho * wo, k * c), dtype=x.dtype, device=x.device)
            gw2 = torch.zeros((cout, k * c), dtype=x.dtype, device=x.device)
            g2 = g.view(n * ho * wo, cout)
            for n0 in range(0, n, per):
                n1 = min(n, n0 + per)
                rows = (n1 - n0) * ho * wo
                _lib.check(lib.devis_dcn_im2col_og(_ptr(x[n0:n1]), _ptr(offset[n0:n1]),
                                                   _ptr(mask[n0:n1]) if mask is not None else None, _ptr(cols),
                                                   n1 - n0, *dims[1:], og, _DTYPES[x.dtype], stream))
                gw2 += _wgrad(g2[n0 * ho * wo:n1 * ho * wo], cols[:rows])
            grad_w = gw2.view(cout, kh, kw, c).permute(0, 3, 1, 2)
    if need_b and bias is not None:
        grad_b = g.sum((0, 1, 2))
    return tuple(x.new_empty(0) if t is None else t for t in (grad_in, grad_off, grad_w, grad_b, grad_m))


@_fused_backward_op.register_fake
def _(grad_out, input, x_copy, offset, weight, bias, mask, packed, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
      form, need_in, need_off, need_w, need_b, need_m):
    return _fake_backward(input, offset, weight, bias, mask, need_in, need_off, need_w, need_b, need_m)


def _fused_setup_context(ctx, inputs, output):
    input, offset, weight, bias, mask, *geometry, _ = inputs
    _, x_copy, packed = output
    cout, c, kh, kw = weight.shape
    ctx.geometry = geometry
    ctx.form = _fused_form(c, cout, kh, kw, input.dtype, _offset_groups(offset, kh, kw))
    ctx.mark_non_differentiable(x_copy, packed)
    ctx.save_for_backward(input, x_copy, offset, weight, bias, mask, packed)


def _fused_backward(ctx, grad_out, *_unused):
    input, x_copy, offset, weight, bias, mask, packed = ctx.saved_tensors
    return _autograd_result(_fused_backward_op(grad_out, input, x_copy, offset, weight, bias, mask, packed,
                                               *ctx.geometry, ctx.form, *_needs(ctx)), 7)


_fused_op.register_autograd(_fused_backward, setup_context=_fused_setup_context)


class FusedDeformConv2dFunction:
    """apply(input, offset, weight, bias, mask, stride, padding, dilation) -> (N, Cout, Ho, Wo), fused kernels
    (op ``devis::deform_conv2d_fused``, once differentiable)"""

    @staticmethod
    def apply(input, offset, weight, bias, mask, stride, padding, dilation):
        cout, c, kh, kw = weight.shape
        elems = _packed_weight_elems(int(c), int(cout), int(kh), int(kw), int(_offset_groups(offset, kh, kw)))
        return _fused_op(input, offset, weight, bias, mask, *stride, *padding, *dilation, elems)[0]


# ------------------------------------------------------------------------------------------------------------------------
# im2col form: column matrix + cuBLAS GEMM
# ------------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("devis::deform_conv2d_im2col", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _im2col_op(input: torch.Tensor, offset: torch.Tensor, weight: torch.Tensor, bias: OptTensor, mask: OptTensor,
               stride_h: int, stride_w: int, pad_h: int, pad_w: int, dil_h: int,
               dil_w: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(out (N, Cout, Ho, Wo), channels-last input copy or empty, columns (N*Ho*Wo, K*Cin))"""
    if not input.is_cuda:
        raise RuntimeError("deform_conv2d: not implemented on the CPU (no fallback in this library)")
    n, c, h, w = input.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    x, x_copy = _nhwc(input)                                          # (N, H, W, C)
    offset, mask = _contig(offset), _contig(mask)
    k, og = kh * kw, _offset_groups(offset, kh, kw)
    cols = torch.empty((n * ho * wo, k * c), dtype=input.dtype, device=input.device)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    with torch.cuda.device(input.device):
        _lib.check(_lib.load().devis_dcn_im2col_og(_ptr(x), _ptr(offset), _ptr(mask), _ptr(cols), *dims, og,
                                                   _DTYPES[input.dtype], torch.cuda.current_stream().cuda_stream))
    w2 = weight.permute(0, 2, 3, 1).reshape(cout, k * c)              # columns are [k][ci]
    out = torch.addmm(bias, cols, w2.t()) if bias is not None else cols @ w2.t()
    return out.view(n, ho, wo, cout).permute(0, 3, 1, 2), x_copy, cols


@_im2col_op.register_fake
def _(input, offset, weight, bias, mask, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w):
    out, x_copy = _fake_forward(input, offset, weight, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w)
    n, _, ho, wo = out.shape
    cout, c, kh, kw = weight.shape
    return out, x_copy, input.new_empty((n * ho * wo, kh * kw * c))


@torch.library.custom_op("devis::deform_conv2d_im2col_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _im2col_backward_op(grad_out: torch.Tensor, input: torch.Tensor, x_copy: torch.Tensor, offset: torch.Tensor,
                        weight: torch.Tensor, bias: OptTensor, mask: OptTensor, cols: torch.Tensor, stride_h: int,
                        stride_w: int, pad_h: int, pad_w: int, dil_h: int, dil_w: int, need_in: bool, need_off: bool,
                        need_w: bool, need_b: bool,
                        need_m: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(grad_input, grad_offset, grad_weight, grad_bias, grad_mask) from the forward's columns"""
    x = _saved_nhwc(input, x_copy)
    offset, mask = _contig(offset), _contig(mask)
    n, h, w, c = x.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    og = _offset_groups(offset, kh, kw)
    w2 = weight.detach().permute(0, 2, 3, 1).reshape(cout, kh * kw * c)
    g2 = grad_out.permute(0, 2, 3, 1).reshape(n * ho * wo, cout)
    grad_w = grad_b = grad_in = grad_off = grad_m = None
    if need_w:
        grad_w = _wgrad(g2, cols).view(cout, kh, kw, c).permute(0, 3, 1, 2)
    if need_b and bias is not None:
        grad_b = g2.sum(0)
    if need_in or need_off or (need_m and mask is not None):
        grad_cols = g2 @ w2
        flags = _grad_input_flags(x.dtype) if need_in else 0
        gx = torch.empty_like(x, memory_format=torch.contiguous_format) if need_in else None
        grad_off = torch.empty_like(offset)
        grad_m = torch.empty_like(mask) if mask is not None else None
        lib = _lib.load()
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            per = _data_chunk(n, h, w, c, flags, n)
            ws, ws_bytes = _workspace(lib, per, h, w, c, flags, x.device)
            for n0 in range(0, n, per):
                n1 = min(n, n0 + per)
                _lib.check(lib.devis_dcn_col2im_og(_ptr(x[n0:n1]), _ptr(offset[n0:n1]),
                                                   _ptr(mask[n0:n1]) if mask is not None else None,
                                                   _ptr(grad_cols[n0 * ho * wo:n1 * ho * wo]),
                                                   _ptr(gx[n0:n1]) if need_in else None, _ptr(grad_off[n0:n1]),
                                                   _ptr(grad_m[n0:n1]) if mask is not None else None, n1 - n0,
                                                   *dims[1:], og, _DTYPES[x.dtype], flags, _ptr(ws),
                                                   ws_bytes, stream))
        grad_in = gx.permute(0, 3, 1, 2) if need_in else None
    return tuple(x.new_empty(0) if t is None else t for t in (grad_in, grad_off, grad_w, grad_b, grad_m))


@_im2col_backward_op.register_fake
def _(grad_out, input, x_copy, offset, weight, bias, mask, cols, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
      need_in, need_off, need_w, need_b, need_m):
    return _fake_backward(input, offset, weight, bias, mask, need_in, need_off, need_w, need_b, need_m)


def _im2col_setup_context(ctx, inputs, output):
    input, offset, weight, bias, mask, *geometry = inputs
    _, x_copy, cols = output
    ctx.geometry = geometry
    ctx.mark_non_differentiable(x_copy, cols)
    ctx.save_for_backward(input, x_copy, offset, weight, bias, mask, cols)


def _im2col_backward(ctx, grad_out, *_unused):
    input, x_copy, offset, weight, bias, mask, cols = ctx.saved_tensors
    return _autograd_result(_im2col_backward_op(grad_out, input, x_copy, offset, weight, bias, mask, cols,
                                                *ctx.geometry, *_needs(ctx)), 6)


_im2col_op.register_autograd(_im2col_backward, setup_context=_im2col_setup_context)


class DeformConv2dFunction:
    """apply(input, offset, weight, bias, mask, stride, padding, dilation) -> (N, Cout, Ho, Wo)
    (op ``devis::deform_conv2d_im2col``, once differentiable)"""

    @staticmethod
    def apply(input, offset, weight, bias, mask, stride, padding, dilation):
        return _im2col_op(input, offset, weight, bias, mask, *stride, *padding, *dilation)[0]


_TENSOR_CORE = True


def set_tensor_core(enabled):
    """enable / disable the tcgen05 implicit-GEMM forward of the wide layers (default on); returns the previous setting"""
    global _TENSOR_CORE
    old, _TENSOR_CORE = _TENSOR_CORE, bool(enabled)
    return old


@torch.compiler.assume_constant_result
def _library_igemm_supported(c, cout, kh, kw):
    return bool(_lib.load().devis_dcn_igemm_supported(c, cout, kh, kw, _lib.F32))


def _igemm_supported(c, cout, kh, kw, dtype):
    if not _TENSOR_CORE or dtype != torch.float32:
        return False
    return _library_igemm_supported(int(c), int(cout), int(kh), int(kw))


@torch.library.custom_op("devis::deform_conv2d_igemm", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _igemm_op(input: torch.Tensor, offset: torch.Tensor, weight: torch.Tensor, bias: OptTensor, mask: OptTensor,
              stride_h: int, stride_w: int, pad_h: int, pad_w: int, dil_h: int,
              dil_w: int) -> tuple[torch.Tensor, torch.Tensor]:
    """(out (N, Cout, Ho, Wo), channels-last input copy or empty).  Precision: torch.backends.cuda.matmul.allow_tf32
    as it is when the op runs"""
    if not input.is_cuda:
        raise RuntimeError("deform_conv2d: not implemented on the CPU (no fallback in this library)")
    n, c, h, w = input.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    x, x_copy = _nhwc(input)
    offset, mask, bias = _contig(offset), _contig(mask), _contig(bias)
    lib = _lib.load()
    wd = weight.detach()
    wd = wd if wd.is_contiguous() else wd.contiguous()
    packed = torch.empty(int(lib.devis_dcn_igemm_packed_weight_elems(c, cout, kh, kw)), dtype=torch.float32,
                         device=input.device)
    out = torch.empty((n, ho, wo, cout), dtype=input.dtype, device=input.device)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    precision = _lib.DCN_PRECISION_TF32 if torch.backends.cuda.matmul.allow_tf32 else _lib.DCN_PRECISION_3XTF32
    with torch.cuda.device(input.device):
        stream = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.devis_dcn_igemm_pack_weight(_ptr(wd), _ptr(packed), c, cout, kh, kw, stream))
        _lib.check(lib.devis_dcn_igemm_forward(_ptr(x), _ptr(offset), _ptr(mask), _ptr(packed), _ptr(bias), _ptr(out),
                                               *dims, cout, precision, stream))
    return out.permute(0, 3, 1, 2), x_copy


@_igemm_op.register_fake
def _(input, offset, weight, bias, mask, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w):
    return _fake_forward(input, offset, weight, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w)


@torch.library.custom_op("devis::deform_conv2d_igemm_backward", mutates_args=(), tags=(torch.Tag.needs_exact_strides,))
def _igemm_backward_op(grad_out: torch.Tensor, input: torch.Tensor, x_copy: torch.Tensor, offset: torch.Tensor,
                       weight: torch.Tensor, bias: OptTensor, mask: OptTensor, stride_h: int, stride_w: int, pad_h: int,
                       pad_w: int, dil_h: int, dil_w: int, need_in: bool, need_off: bool, need_w: bool, need_b: bool,
                       need_m: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(grad_input, grad_offset, grad_weight, grad_bias, grad_mask): the im2col form's backward with the columns
    recomputed in bounded chunks"""
    x = _saved_nhwc(input, x_copy)
    offset, mask = _contig(offset), _contig(mask)
    n, h, w, c = x.shape
    cout, _, kh, kw = weight.shape
    sh, sw, ph, pw, dh, dw = stride_h, stride_w, pad_h, pad_w, dil_h, dil_w
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    dims = (n, h, w, c, ho, wo, kh, kw, sh, sw, ph, pw, dh, dw)
    k = kh * kw
    weight = weight.detach()
    weight = weight if weight.is_contiguous() else weight.contiguous()
    g2 = grad_out.permute(0, 2, 3, 1).reshape(n * ho * wo, cout)
    g2 = g2 if g2.is_contiguous() else g2.contiguous()
    w2 = weight.permute(0, 2, 3, 1).reshape(cout, k * c)
    grad_w = grad_b = grad_in = grad_off = grad_m = None
    lib = _lib.load()
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream().cuda_stream
        if need_w:
            per = max(1, min(n, _COLS_CHUNK_BYTES // max(1, ho * wo * k * c * 4)))
            cols = torch.empty((per * ho * wo, k * c), dtype=x.dtype, device=x.device)
            gw2 = torch.zeros((cout, k * c), dtype=x.dtype, device=x.device)
            for n0 in range(0, n, per):
                n1 = min(n, n0 + per)
                rows = (n1 - n0) * ho * wo
                _lib.check(lib.devis_dcn_im2col(_ptr(x[n0:n1]), _ptr(offset[n0:n1]),
                                                _ptr(mask[n0:n1]) if mask is not None else None, _ptr(cols),
                                                n1 - n0, *dims[1:], _DTYPES[x.dtype], stream))
                gw2 += _wgrad(g2[n0 * ho * wo:n1 * ho * wo], cols[:rows])
            del cols
            grad_w = gw2.view(cout, kh, kw, c).permute(0, 3, 1, 2)
        if need_b and bias is not None:
            grad_b = g2.sum(0)
        if need_in or need_off or (need_m and mask is not None):
            flags = _grad_input_flags(x.dtype) if need_in else 0
            gx = torch.empty_like(x, memory_format=torch.contiguous_format) if need_in else None
            grad_off = torch.empty_like(offset)
            grad_m = torch.empty_like(mask) if mask is not None else None
            per = _data_chunk(n, h, w, c, flags, _COLS_CHUNK_BYTES // max(1, ho * wo * k * c * 4))
            ws, ws_bytes = _workspace(lib, per, h, w, c, flags, x.device)
            for n0 in range(0, n, per):
                n1 = min(n, n0 + per)
                grad_cols = g2[n0 * ho * wo:n1 * ho * wo] @ w2
                _lib.check(lib.devis_dcn_col2im_ex(_ptr(x[n0:n1]), _ptr(offset[n0:n1]),
                                                   _ptr(mask[n0:n1]) if mask is not None else None, _ptr(grad_cols),
                                                   _ptr(gx[n0:n1]) if need_in else None, _ptr(grad_off[n0:n1]),
                                                   _ptr(grad_m[n0:n1]) if mask is not None else None, n1 - n0,
                                                   *dims[1:], _DTYPES[x.dtype], flags, _ptr(ws), ws_bytes,
                                                   stream))
            grad_in = gx.permute(0, 3, 1, 2) if need_in else None
    return tuple(x.new_empty(0) if t is None else t for t in (grad_in, grad_off, grad_w, grad_b, grad_m))


@_igemm_backward_op.register_fake
def _(grad_out, input, x_copy, offset, weight, bias, mask, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, need_in,
      need_off, need_w, need_b, need_m):
    return _fake_backward(input, offset, weight, bias, mask, need_in, need_off, need_w, need_b, need_m)


def _igemm_setup_context(ctx, inputs, output):
    input, offset, weight, bias, mask, *geometry = inputs
    ctx.geometry = geometry
    ctx.mark_non_differentiable(output[1])
    ctx.save_for_backward(input, output[1], offset, weight, bias, mask)


def _igemm_backward(ctx, grad_out, *_unused):
    input, x_copy, offset, weight, bias, mask = ctx.saved_tensors
    return _autograd_result(_igemm_backward_op(grad_out, input, x_copy, offset, weight, bias, mask, *ctx.geometry,
                                               *_needs(ctx)), 6)


_igemm_op.register_autograd(_igemm_backward, setup_context=_igemm_setup_context)


class IGemmDeformConv2dFunction:
    """apply(input, offset, weight, bias, mask, stride, padding, dilation) -> (N, Cout, Ho, Wo)

    Forward of the wide mask-head layers as an implicit GEMM on the tensor cores (devis_dcn_igemm_forward, tcgen05 /
    TMEM): no column matrix is written or kept.  One offset group only.  Precision follows ``torch.backends.cuda.matmul.allow_tf32`` exactly as
    torchvision's ``addmm`` would: off (the default) -> 3xTF32, fp32-grade; on -> one TF32 pass.  The backward is the
    im2col form's (cuBLAS GEMMs + devis_dcn_col2im), with the columns RECOMPUTED for the weight gradient, so nothing of
    column size lives between forward and backward.  Op ``devis::deform_conv2d_igemm``, once differentiable."""

    @staticmethod
    def apply(input, offset, weight, bias, mask, stride, padding, dilation):
        return _igemm_op(input, offset, weight, bias, mask, *stride, *padding, *dilation)[0]


def deform_conv2d(input, offset, weight, bias=None, stride=(1, 1), padding=(0, 0), dilation=(1, 1), mask=None):
    """torchvision.ops.deform_conv2d (torchvision/ops/deform_conv.py:14), same arguments and result."""
    stride, padding, dilation = _pair(stride), _pair(padding), _pair(dilation)
    if input.dim() != 4 or weight.dim() != 4 or offset.dim() != 4:
        raise RuntimeError("deform_conv2d: input, offset and weight must be 4-dimensional")
    if not input.is_cuda:
        raise RuntimeError("deform_conv2d: not implemented on the CPU (no fallback in this library)")
    n, c, h, w = input.shape
    cout, cin_g, kh, kw = weight.shape
    if cin_g != c:
        raise RuntimeError(f"deform_conv2d: groups = {c // max(cin_g, 1)} is not supported by this build (groups = 1 only)")
    k = kh * kw
    if offset.shape[1] == 0 or offset.shape[1] % (2 * k):
        raise RuntimeError(f"deform_conv2d: offset.shape[1] must be a multiple of 2 * kernel_h * kernel_w = {2 * k}, "
                           f"got {offset.shape[1]}")
    og = _offset_groups(offset, kh, kw)
    if c % og:
        raise RuntimeError(f"deform_conv2d: input channels ({c}) must be divisible by offset_groups ({og})")
    ho, wo = _out_size(h, kh, stride[0], padding[0], dilation[0]), _out_size(w, kw, stride[1], padding[1], dilation[1])
    if ho <= 0 or wo <= 0:
        raise RuntimeError(f"deform_conv2d: calculated output size too small ({ho} x {wo})")
    if tuple(offset.shape) != (n, 2 * og * k, ho, wo):
        raise RuntimeError(f"deform_conv2d: offset must be {(n, 2 * og * k, ho, wo)}, got {tuple(offset.shape)}")
    if mask is not None and tuple(mask.shape) != (n, og * k, ho, wo):
        raise RuntimeError(f"deform_conv2d: mask must be {(n, og * k, ho, wo)}, got {tuple(mask.shape)}")
    if bias is not None and tuple(bias.shape) != (cout,):
        raise RuntimeError("deform_conv2d: bias must have out_channels elements")
    out_dtype = input.dtype
    if out_dtype in (torch.float16, torch.bfloat16):          # torchvision's autocast wrapper computes in float32 too
        cast = lambda t: None if t is None else t.float()
        input, offset, weight, bias, mask = cast(input), cast(offset), cast(weight), cast(bias), cast(mask)
    elif out_dtype not in _DTYPES:
        raise RuntimeError(f'"deform_conv2d" not implemented for \'{out_dtype}\'')
    same = lambda t: None if t is None else (t if t.dtype == input.dtype else t.to(input.dtype))
    # fused forward when the layer is served; when gradients are needed only if its data backward is fused as well
    # (otherwise the im2col form, which keeps its columns for the backward, is the faster training path)
    # (the layer's channel counts are read from the weight: a parameter, static for torch.compile even when the input
    # shapes are dynamic; c == cin_g was checked above)
    form = _fused_form(cin_g, cout, kh, kw, input.dtype, og) if n > 0 else 0
    needs_grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (input, offset, weight, bias, mask))
    fn = FusedDeformConv2dFunction if form & 1 and (form & 2 or not needs_grad) else DeformConv2dFunction
    # Forward on the tensor cores (tcgen05 implicit GEMM) for the layers with enough contraction to pay for it: everything
    # the CUDA-core fused forms do not serve, and of those they do serve the ones with K*C >= 576 and >= 32 output channels
    # (measured, benchmarks/igemm_narrow.py: 72 -> 32 @45x80 385 us against 613 us; 32 -> 16 @90x160 629 against 486 us and
    # 16 -> 4 623 against 246 us stay where they are).  With gradients the 72 -> 32 layer keeps the im2col form: its backward
    # reuses the forward's columns, which is 270 us faster there than recomputing them (at 560 MB of columns for 60 instances).
    # The tensor-core forward serves one offset group only.
    if og == 1 and n > 0 and _igemm_supported(cin_g, cout, kh, kw, input.dtype) and \
            (not form & 1 or (cin_g * kh * kw >= 576 and cout >= 32 and not form & 2 and not needs_grad)):
        fn = IGemmDeformConv2dFunction
    out = fn.apply(input, same(offset), same(weight), same(bias), same(mask), stride, padding, dilation)
    return out if out.dtype == out_dtype else out.to(out_dtype)
