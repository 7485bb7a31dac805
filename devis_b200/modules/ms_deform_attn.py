"""Attention modules with the reference's class names, constructor arguments, parameter names
(checkpoints load unchanged), call signatures and return values
(/root/reference/src/models/ops/modules/ms_deform_attn.py), running on the sm_100a kernels.

  MSDeformAttn                  ms_deform_attn.py:30-132   one op call; with fuse_prologue the softmax, the location
                                                           arithmetic and the padding mask run inside the kernels
  TemporalMSDeformAttnBase      ms_deform_attn.py:137-285  projections + joint softmax
  TemporalMSDeformAttnEncoder   ms_deform_attn.py:417-464
  TemporalMSDeformAttnDecoder   ms_deform_attn.py:288-414

What differs from the reference is only HOW the temporal modules evaluate a clip: the reference loops
over the T frames in Python and issues two op calls and one gather copy of ``value`` per frame; here
the whole clip is one ``TemporalMSDeformAttnFunction`` call that reads ``value`` in place, and with
``fuse_prologue`` (default, encoder and decoder) the kernels also take over the joint softmax and the location
arithmetic (``TemporalMSDeformAttnFusedFunction``), reading the Linear outputs directly.

The modules call the custom ops (torch.ops.devis.*) with the pyramid tensors and the frame offsets themselves; the op
bodies read their host copies and validate them.  What is left here is traceable Python -- shapes, flags, the choice
of the fused path -- so torch.compile(fullgraph=True) and torch.export trace these modules without a graph break.
"""
import math
import warnings

import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.init import constant_, xavier_uniform_

from .. import MultiScaleDeformableAttention as MSDA
from .. import _lib
from ..functions import TemporalMSDeformAttnFusedFunction
from ..functions import temporal_func


def _is_power_of_2(n):
    if (not isinstance(n, int)) or (n < 0):
        raise ValueError("invalid input for _is_power_of_2: {} (type: {})".format(n, type(n)))
    return (n & (n - 1) == 0) and n != 0


def _head_directions(n_heads):
    """Unit-max-norm direction per head: the initial sampling pattern of Deformable DETR
    (ms_deform_attn.py:66-68,189-192)."""
    theta = torch.arange(n_heads, dtype=torch.float32) * (2.0 * math.pi / n_heads)
    d = torch.stack([theta.cos(), theta.sin()], -1)
    return d / d.abs().max(-1, keepdim=True)[0]


def _ray_bias(n_heads, n_slots, n_points):
    """(heads, slots, points, 2): point i of every slot sits i+1 steps along the head's direction."""
    steps = torch.arange(1, n_points + 1, dtype=torch.float32).view(1, 1, n_points, 1)
    return (_head_directions(n_heads).view(n_heads, 1, 1, 2) * steps).expand(n_heads, n_slots, n_points, 2)


def _wh(spatial_shapes, dtype):
    """(L,2) offset normaliser in (W, H) order (ms_deform_attn.py:113-114)."""
    return torch.stack([spatial_shapes[..., 1], spatial_shapes[..., 0]], -1).to(dtype)


def _pair_halves(arg):
    """the reference's (current, temporal) pair of shape / start-index tensors -> (current, temporal or None)"""
    if isinstance(arg, (tuple, list)):
        return arg[0], (arg[1] if len(arg) > 1 else None)
    return arg, None


def _offset_args(temporal_offsets):
    """the per-frame temporal offsets as the ops take them: (tensors, ints) -- T tensors (the reference's form, passed
    through so that their memoised host copy is reused) or one (T, t_window) tensor; python lists (what the trunk
    passes) as a row-major list of ints, which a compiled graph keeps as constants"""
    if isinstance(temporal_offsets, torch.Tensor):
        return [temporal_offsets], []
    if all(isinstance(o, torch.Tensor) for o in temporal_offsets):
        return list(temporal_offsets), []
    return [], [int(o) for row in temporal_offsets for o in row]


_FRAME_INDEX = {}


def _frame_index(temporal_offsets, n_frames, device):
    """(T, t_window) int64 frame indices on `device` from the per-frame offsets, by tensor ops (no host read)"""
    tensors, ints = _offset_args(temporal_offsets)
    if ints:
        wt = len(ints) // n_frames
        rows = tuple(tuple(t + o for o in ints[t * wt:(t + 1) * wt]) for t in range(n_frames))
        if torch.compiler.is_compiling():         # a constant of the graph
            return torch.tensor(rows, dtype=torch.long, device=device)
        # eager: uploaded once per table and device (a fresh upload per call would also break CUDA-graph capture)
        key = (rows, str(device))
        if key not in _FRAME_INDEX:
            if len(_FRAME_INDEX) > 64:
                _FRAME_INDEX.clear()
            _FRAME_INDEX[key] = torch.tensor(rows, dtype=torch.long, device=device)
        return _FRAME_INDEX[key]
    if len(tensors) == 1 and tensors[0].dim() == 2:
        table = tensors[0]
    else:
        table = torch.stack([o.reshape(-1) for o in tensors])
    return table.to(device=device, dtype=torch.long) + torch.arange(n_frames, device=device)[:, None]


def _tile(query_tile):
    return tuple(query_tile) if query_tile else (0, 0)


def _check_head_dim(d_model, n_heads):
    if d_model % n_heads != 0:
        raise ValueError("d_model must be divisible by n_heads, but got {} and {}".format(d_model, n_heads))
    if not _is_power_of_2(d_model // n_heads):
        warnings.warn("You'd better set d_model in MSDeformAttn to make the dimension of each attention head a "
                      "power of 2 which is more efficient in our CUDA implementation.")


class MSDeformAttn(nn.Module):
    def __init__(self, d_model=256, n_levels=4, n_heads=8, n_points=4):
        super().__init__()
        _check_head_dim(d_model, n_heads)
        self.im2col_step = 64
        self.d_model, self.n_levels, self.n_heads, self.n_points = d_model, n_levels, n_heads, n_points
        self.sampling_offsets = nn.Linear(d_model, n_heads * n_levels * n_points * 2)
        self.attention_weights = nn.Linear(d_model, n_heads * n_levels * n_points)
        self.value_proj = nn.Linear(d_model, d_model)
        self.output_proj = nn.Linear(d_model, d_model)
        # encoder self-attention (Lq == S): walk the pixel-grid queries in 2-D tiles (cache locality only)
        self.query_tile = (8, 8)
        # let the kernels read the raw Linear outputs and the padding mask (TemporalMSDeformAttnFusedFunction with the
        # batch as the frame axis): no softmax, location or masked_fill kernels and no copy of value, either way
        self.fuse_prologue = True
        self._reset_parameters()

    def _reset_parameters(self):
        constant_(self.sampling_offsets.weight.data, 0.)
        with torch.no_grad():
            self.sampling_offsets.bias = nn.Parameter(
                _ray_bias(self.n_heads, self.n_levels, self.n_points).reshape(-1).clone())
        constant_(self.attention_weights.weight.data, 0.)
        constant_(self.attention_weights.bias.data, 0.)
        xavier_uniform_(self.value_proj.weight.data)
        constant_(self.value_proj.bias.data, 0.)
        xavier_uniform_(self.output_proj.weight.data)
        constant_(self.output_proj.bias.data, 0.)

    def _fused_path(self, value, reference_points):
        """whether forward() takes the fused-prologue kernels for this projected value (N,S,M,D).  float32 and bfloat16
        only: float16 keeps the reference's dispatch (it raises), float64 and the shapes the fused kernels do not serve
        (D != 32, P % 4 != 0, value >= 2 GiB, deterministic mode with learnable reference points) keep the unfused op."""
        return (self.fuse_prologue and value.dtype in (torch.float32, torch.bfloat16) and value.shape[0] > 0
                and TemporalMSDeformAttnFusedFunction.supported(value, reference_points, self.n_points, self.n_points))

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                input_padding_mask=None):
        """query (N,Lq,C); reference_points (N,Lq,L,2|4); input_flatten (N,S,C); returns (out, None)."""
        n, lq, _ = query.shape
        s = input_flatten.shape[1]
        m, nl, p = self.n_heads, self.n_levels, self.n_points
        value = self.value_proj(input_flatten)
        # decided on the PROJECTED value (under autocast it is half precision while input_flatten is not)
        heads = value.view(n, s, m, self.d_model // m)
        if self._fused_path(heads, reference_points):
            return self._forward_fused(query, reference_points, heads, input_spatial_shapes, input_level_start_index,
                                       input_padding_mask)

        if input_padding_mask is not None:
            value = value.masked_fill(input_padding_mask[..., None], float(0))
        value = value.view(n, s, m, self.d_model // m)
        offsets = self.sampling_offsets(query).view(n, lq, m, nl, p, 2)
        weights = F.softmax(self.attention_weights(query).view(n, lq, m, nl * p), -1).view(n, lq, m, nl, p)
        if reference_points.shape[-1] == 2:
            loc = reference_points[:, :, None, :, None, :] \
                + offsets / _wh(input_spatial_shapes, offsets.dtype)[None, None, None, :, None, :]
        elif reference_points.shape[-1] == 4:
            loc = reference_points[:, :, None, :, None, :2] \
                + offsets / p * reference_points[:, :, None, :, None, 2:] * 0.5
        else:
            raise ValueError("Last dim of reference_points must be 2 or 4, but get {} instead.".format(
                reference_points.shape[-1]))
        # (the op asserts sum(H*W) == S on the pyramid's host copy)
        out = MSDA._forward_op(value, input_spatial_shapes, input_level_start_index, loc, weights, self.im2col_step,
                               True)
        return self.output_proj(out), None

    def _forward_fused(self, query, reference_points, value, input_spatial_shapes, input_level_start_index,
                       input_padding_mask):
        """One launch each way for the attention: the N images are the frames of a clip without temporal slots, the
        softmax, `ref + off / (W, H)` (points, encoder form) or the box form (GEN) and the padding mask are evaluated in
        the kernels.  Host values of the pyramid come from memoised reads inside the op: no device read-back the unfused
        path does not make."""
        n, lq, _ = query.shape
        m, nl, p = self.n_heads, self.n_levels, self.n_points
        step = min(n, self.im2col_step)
        if n % step != 0:
            raise RuntimeError(f"batch({n}) must divide im2col_step({step})")
        out = temporal_func._fused_op(
            value, reference_points, self.sampling_offsets(query).view(n, lq, m, nl, p, 2),
            self.attention_weights(query).view(n, lq, m, nl * p), None, None, input_spatial_shapes,
            input_level_start_index, None, None, [], [], None, *_tile(self.query_tile), _lib.TREF_LEVEL0, False,
            input_padding_mask, True)[0]
        return self.output_proj(out), None


class TemporalMSDeformAttnBase(nn.Module):
    def __init__(self, n_frames=36, d_model=256, n_levels=4, t_window=2, n_heads=8, n_curr_points=4,
                 n_temporal_points=2):
        super().__init__()
        _check_head_dim(d_model, n_heads)
        self.im2col_step = 64
        self.d_model, self.n_frames, self.n_levels, self.t_window = d_model, n_frames, n_levels, t_window
        self.n_heads, self.n_curr_points, self.n_temporal_points = n_heads, n_curr_points, n_temporal_points

        self.sampling_offsets = nn.Linear(d_model, n_heads * n_levels * n_curr_points * 2)
        self.attention_weights = nn.Linear(d_model, n_heads * n_levels * n_curr_points)
        self.temporal_sampling_offsets = nn.Linear(d_model, n_heads * n_levels * t_window * n_temporal_points * 2)
        self.temporal_attention_weights = nn.Linear(d_model, n_heads * n_levels * t_window * n_temporal_points)
        self.value_proj = nn.Linear(d_model, d_model)
        self.output_proj = nn.Linear(d_model, d_model)
        # encoder only: walk the pixel-grid queries in 2-D tiles (cache locality, see ClipGeometry.tile_order)
        self.query_tile = (8, 8)
        # let the kernels read the raw Linear outputs (joint softmax and the sampling-location arithmetic fused in)
        self.fuse_prologue = True
        self._reset_parameters()

    def _reset_parameters(self):
        constant_(self.sampling_offsets.weight.data, 0.)
        constant_(self.temporal_sampling_offsets.weight.data, 0.)
        with torch.no_grad():
            self.sampling_offsets.bias = nn.Parameter(
                _ray_bias(self.n_heads, self.n_levels, self.n_curr_points).reshape(-1).clone())
            self.temporal_sampling_offsets.bias = nn.Parameter(
                _ray_bias(self.n_heads, self.n_levels * self.t_window, self.n_temporal_points).reshape(-1).clone())
        for lin in (self.attention_weights, self.temporal_attention_weights):
            constant_(lin.weight.data, 0.)
            constant_(lin.bias.data, 0.)
        for lin in (self.value_proj, self.output_proj):
            xavier_uniform_(lin.weight.data)
            constant_(lin.bias.data, 0.)

    def _compute_deformable_attention(self, query, input_flatten):
        """ms_deform_attn.py:225-266.  Returns value (T,S,M,D), current offsets (T,Lq,M,L,Pc,2), temporal
        offsets (T,Lq,M,Wt*L,Pt,2) with the temporal axis frame-slot-major / level-minor, and the two
        halves of ONE softmax over all L*Pc + Wt*L*Pt taps.  (No padding-mask fill: the temporal
        modules never receive a mask, devis_transformer.py:120.)"""
        t, lq, _ = query.shape
        m, nl, wt, pc, pt = self.n_heads, self.n_levels, self.t_window, self.n_curr_points, self.n_temporal_points
        value = None
        if input_flatten is not None:     # None: the caller has projected value already
            value = self.value_proj(input_flatten).view(t, input_flatten.shape[1], m, self.d_model // m)
        off_t = self.temporal_sampling_offsets(query).view(t, lq, m, wt * nl, pt, 2)
        off_c = self.sampling_offsets(query).view(t, lq, m, nl, pc, 2)
        logits = torch.cat([self.attention_weights(query).view(t, lq, m, nl * pc),
                            self.temporal_attention_weights(query).view(t, lq, m, wt * nl * pt)], dim=3)
        joint = F.softmax(logits, -1)
        aw_c = joint[..., :nl * pc].reshape(t, lq, m, nl, pc)
        aw_t = joint[..., nl * pc:].reshape(t, lq, m, wt * nl, pt)
        return value, off_c, off_t, aw_c, aw_t

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                temporal_offsets):
        raise NotImplementedError


class TemporalMSDeformAttnEncoder(TemporalMSDeformAttnBase):
    def forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                temporal_offsets):
        """query (T,S,C); reference_points (T,S,L,2); input_flatten (T,S,C); input_spatial_shapes /
        input_level_start_index: (current, temporal) pairs; temporal_offsets: T tensors of t_window frame
        offsets.  Returns (out (T,S,C), None) -- ms_deform_attn.py:419-464."""
        cur_shapes, t_shapes = _pair_halves(input_spatial_shapes)
        cur_lsi, t_lsi = _pair_halves(input_level_start_index)
        offs, ints = _offset_args(temporal_offsets)
        assert reference_points.shape[-1] == 2
        tile = _tile(self.query_tile)

        t, lq, _ = query.shape
        m, nl, wt, pc, pt = self.n_heads, self.n_levels, self.t_window, self.n_curr_points, self.n_temporal_points
        value = self.value_proj(input_flatten).view(t, input_flatten.shape[1], m, self.d_model // m)
        # decided on the PROJECTED value (under autocast it is half precision while input_flatten is not)
        if self.fuse_prologue and TemporalMSDeformAttnFusedFunction.supported(value, reference_points, pc, pt):
            out = temporal_func._fused_op(
                value, reference_points,
                self.sampling_offsets(query).view(t, lq, m, nl, pc, 2),
                self.attention_weights(query).view(t, lq, m, nl * pc),
                self.temporal_sampling_offsets(query).view(t, lq, m, wt * nl, pt, 2),
                self.temporal_attention_weights(query).view(t, lq, m, wt * nl * pt), cur_shapes, cur_lsi, t_shapes,
                t_lsi, offs, ints, None, *tile, _lib.TREF_LEVEL0, False, None, False)[0]
            return self.output_proj(out), None

        _, off_c, off_t, aw_c, aw_t = self._compute_deformable_attention(query, None)

        wh = _wh(cur_shapes, off_c.dtype)
        loc_c = reference_points[:, :, None, :, None, :] + off_c / wh[None, None, None, :, None, :]
        # temporal taps start from the LEVEL-0 reference point on every temporal level (:447)
        loc_t = reference_points[:, :, 0][:, :, None, None, None, :] \
            + off_t / wh.repeat(self.t_window, 1)[None, None, None, :, None, :]

        out = temporal_func._tmsda_op(value, loc_c, aw_c, loc_t, aw_t, cur_shapes, cur_lsi, t_shapes, t_lsi, offs, ints, None,
                                      *tile)
        return self.output_proj(out), None


class TemporalMSDeformAttnDecoder(TemporalMSDeformAttnBase):
    def __init__(self, n_frames=36, d_model=256, n_levels=4, t_window=2, n_heads=8, n_curr_points=4,
                 n_temporal_points=2, dec_instance_aware_att=True):
        super().__init__(n_frames=n_frames, d_model=d_model, n_levels=n_levels, t_window=t_window, n_heads=n_heads,
                         n_curr_points=n_curr_points, n_temporal_points=n_temporal_points)
        self.dec_instance_aware_att = dec_instance_aware_att

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                temporal_offsets):
        """query (1,T*q,C); reference_points (1,T*q,L,2|4) or (T,q,L,2|4); input_flatten (T,S,C).  Returns the
        reference's 5-tuple (ms_deform_attn.py:414): out (1,T*q,C), T current location tensors
        (1,q,M,L,Pc,2), T temporal location tensors (1,q,M,Wt*L,Pt,2), current and temporal weights."""
        cur_shapes, t_shapes = _pair_halves(input_spatial_shapes)
        cur_lsi, t_lsi = _pair_halves(input_level_start_index)
        offs, ints = _offset_args(temporal_offsets)
        n_frames = input_flatten.shape[0]
        q = query.shape[1] // n_frames
        query = query.reshape(n_frames, q, query.shape[-1])
        if reference_points.shape[0] != n_frames:
            reference_points = reference_points.reshape((n_frames, q) + tuple(reference_points.shape[-2:]))
        m, nl, wt, pc, pt = self.n_heads, self.n_levels, self.t_window, self.n_curr_points, self.n_temporal_points
        value = self.value_proj(input_flatten).view(n_frames, input_flatten.shape[1], m, self.d_model // m)
        if reference_points.shape[-1] not in (2, 4):
            raise ValueError("Last dim of reference_points must be 2 or 4, but get {} instead.".format(
                reference_points.shape[-1]))

        if self.fuse_prologue and TemporalMSDeformAttnFusedFunction.supported(value, reference_points, pc, pt):
            # one launch each way: softmax, `ref + off / (W, H)` or the box form, the instance-aware reference lookup and
            # the 5-tuple's locations / weights (by-products, not differentiable) all happen in the kernels
            out, loc_c, aw_c, loc_t, aw_t = temporal_func._fused_op(
                value, reference_points,
                self.sampling_offsets(query).view(n_frames, q, m, nl, pc, 2),
                self.attention_weights(query).view(n_frames, q, m, nl * pc),
                self.temporal_sampling_offsets(query).view(n_frames, q, m, wt * nl, pt, 2),
                self.temporal_attention_weights(query).view(n_frames, q, m, wt * nl * pt), cur_shapes, cur_lsi,
                t_shapes, t_lsi, offs, ints, None, 0, 0, _lib.TREF_SAMPLED if self.dec_instance_aware_att else _lib.TREF_OWN,
                True, None, False)
            out = self.output_proj(out.flatten(0, 1)[None])
            return (out, [loc_c[t][None] for t in range(n_frames)], [loc_t[t][None] for t in range(n_frames)],
                    aw_c, aw_t)

        _, off_c, off_t, aw_c, aw_t = self._compute_deformable_attention(query, None)

        # reference point each temporal (slot, level) starts from: the same query's own reference in the
        # sampled frame when instance-aware (:342-344), else its frame-t reference repeated (:346-347)
        if self.dec_instance_aware_att:
            table = _frame_index(temporal_offsets, n_frames, query.device)                     # (T, Wt)
            ref_t = reference_points[table].permute(0, 2, 1, 3, 4).flatten(2, 3)                 # (T,q,Wt*L,.)
        else:
            ref_t = reference_points.repeat(1, 1, self.t_window, 1)

        if reference_points.shape[-1] == 2:
            wh = _wh(cur_shapes, off_c.dtype)
            loc_c = reference_points[:, :, None, :, None, :] + off_c / wh[None, None, None, :, None, :]
            loc_t = ref_t[:, :, None, :, None, :] + off_t / wh.repeat(self.t_window, 1)[None, None, None, :, None, :]
        else:
            loc_c = reference_points[:, :, None, :, None, :2] \
                + (off_c / self.n_curr_points) * reference_points[:, :, None, :, None, 2:] * 0.5
            loc_t = ref_t[:, :, None, :, None, :2] + (off_t / self.n_temporal_points) * ref_t[:, :, None, :, None, 2:] * 0.5

        out = temporal_func._tmsda_op(value, loc_c, aw_c, loc_t, aw_t, cur_shapes, cur_lsi, t_shapes, t_lsi, offs, ints, None,
                                      0, 0)
        out = self.output_proj(out.flatten(0, 1)[None])
        return (out, [loc_c[t][None] for t in range(n_frames)], [loc_t[t][None] for t in range(n_frames)],
                aw_c, aw_t)
