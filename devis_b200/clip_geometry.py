"""Host-side description of a clip's value pyramid for the whole-clip temporal op.

The reference keeps ``spatial_shapes`` / ``level_start_index`` / ``temporal_offsets`` as device
tensors that its kernels dereference (cuda/ms_deform_attn_cuda.cu:67-68) and rebuilds repeated
"temporal" copies of them for every forward (devis_transformer.py:94-118,147-154).  The whole-clip
kernels take the per-frame level table and the (T, t_window) frame table as kernel parameters
instead, so they are needed on the host.  ``ClipGeometry`` is that host copy; ``from_reference_args``
derives it from the reference's module arguments with one device->host read that is cached per
tensor (all 12 attention layers of a forward share the same tensors).
"""
import ctypes
import weakref

import numpy as np
import torch


def all_frames_table(n_frames):
    """devis_transformer.py:96-100,147-151: every other frame in frame order -> (T, T-1) frame indices."""
    return [[f for f in range(n_frames) if f != t] for t in range(n_frames)]


def window_table(n_frames, t_window):
    """devis_transformer.py:102-112: +-t_window/2 neighbours, reflected at the clip ends (a frame can
    then appear twice in a row of the table)."""
    deltas = [d for d in range(-t_window // 2, t_window // 2 + 1) if d != 0]
    return [[t + (-d if (t + d < 0 or t + d > n_frames - 1) else d) for d in deltas] for t in range(n_frames)]


class ClipGeometry:
    def __init__(self, shapes, n_frames, frame_table, level_start_index=None):
        shapes = [(int(h), int(w)) for h, w in shapes]
        self.shapes = shapes
        self.n_levels = len(shapes)
        self.n_frames = int(n_frames)
        areas = [h * w for h, w in shapes]
        if level_start_index is None:
            level_start_index = [int(x) for x in np.concatenate([[0], np.cumsum(areas)[:-1]])]
        self.level_start_index = [int(x) for x in level_start_index]
        self.spatial_size = max(st + a for st, a in zip(self.level_start_index, areas))
        table = [[int(f) for f in row] for row in frame_table] if frame_table is not None else [[] for _ in range(n_frames)]
        if len(table) != self.n_frames or any(len(r) != len(table[0]) for r in table):
            raise ValueError("frame_table must have one equally long row per frame")
        if any(f < 0 or f >= self.n_frames for r in table for f in r):
            raise ValueError("frame_table entry outside [0, n_frames)")
        self.frame_table = table
        self.t_window = len(table[0]) if table else 0
        # C-ABI views (kept alive by self)
        self._shapes_np = np.ascontiguousarray(np.array(shapes, dtype=np.int64).reshape(-1, 2))
        self._lsi_np = np.ascontiguousarray(np.array(self.level_start_index, dtype=np.int64))
        self._frames_np = np.ascontiguousarray(np.array(table, dtype=np.int32).reshape(self.n_frames, -1))
        self.shapes_ptr = self._shapes_np.ctypes.data_as(ctypes.c_void_p)
        self.lsi_ptr = self._lsi_np.ctypes.data_as(ctypes.c_void_p)
        self.frames_ptr = self._frames_np.ctypes.data_as(ctypes.c_void_p) if self.t_window else None
        self._orders = {}
        self._op_args = None

    # ------------------------------------------------------------------------------------------
    def op_args(self):
        """(spatial_shapes (L,2), level_start_index (L,) as int64 CPU tensors with their host copies attached, the
        frame offsets as a row-major (T, t_window) list of ints): how the ops (devis::tmsda*) receive this geometry.
        The op body rebuilds the geometry from them (memoised by value) without a device read."""
        if self._op_args is None:
            shapes = attach_host_copy(torch.as_tensor(self._shapes_np), [list(r) for r in self.shapes])
            lsi = attach_host_copy(torch.as_tensor(self._lsi_np), list(self.level_start_index))
            offs = [f - t for t, row in enumerate(self.frame_table) for f in row] if self.t_window else []
            self._op_args = (shapes, lsi, offs)
            _geom_cache.setdefault((self.n_frames, tuple(tuple(r) for r in self.shapes), tuple(self.level_start_index),
                                    tuple(tuple(r) for r in self.frame_table) if self.t_window else None), self)
        return self._op_args

    def frame_table_tensor(self, device):
        """(T, t_window) int64 frame indices on `device`, uploaded once (the decoder's instance-aware gather of
        reference points indexes with it every layer; a fresh upload per call would also break CUDA-graph capture)"""
        key = ("frames", str(device))
        if key not in self._orders:
            self._orders[key] = torch.as_tensor(self.frame_table, dtype=torch.long).reshape(self.n_frames, -1).to(device)
        return self._orders[key]

    def tile_order(self, device, tile_h=8, tile_w=8):
        """Permutation of the S pixel-queries of one frame (encoder self-attention: query i is pixel i,
        deformable_transformer.py:184-198) that walks every level in tile_h x tile_w tiles.  Only
        meaningful when num_query == spatial_size and levels are stored back to back: returns None otherwise (the
        caller then visits the queries in index order -- the order only affects cache locality)."""
        key = (str(device), tile_h, tile_w)
        if key not in self._orders:
            areas = [h * w for h, w in self.shapes]
            packed = all(st == sum(areas[:i]) for i, st in enumerate(self.level_start_index))
            if not packed or sum(areas) != self.spatial_size:
                self._orders[key] = None
                return None
            order = []
            for (h, w), start in zip(self.shapes, self.level_start_index):
                idx = np.arange(h * w, dtype=np.int64).reshape(h, w) + start
                for y0 in range(0, h, tile_h):
                    for x0 in range(0, w, tile_w):
                        order.append(idx[y0:y0 + tile_h, x0:x0 + tile_w].reshape(-1))
            perm = np.concatenate(order).astype(np.int32)
            self._orders[key] = torch.from_numpy(perm).to(device)
        return self._orders[key]


# ------------------------------------------------------------------------------------------------
# Host copies of the small integer tensors the reference passes around.  The copy is memoised ON THE TENSOR OBJECT
# (attribute + version counter), never by address: a later forward with other image sizes allocates new tensors, and
# the caching allocator may well hand them the same address again.
# ------------------------------------------------------------------------------------------------
_ATTR = "_devis_b200_host_copy"


def _host_list(t):
    """device int tensor -> nested python list; one synchronising read per tensor object and version."""
    if not isinstance(t, torch.Tensor):
        return [list(r) if hasattr(r, "__len__") else int(r) for r in t]
    hit = getattr(t, _ATTR, None)
    if hit is not None and hit[0] == t._version:
        return hit[1]
    host = t.tolist()
    try:
        setattr(t, _ATTR, (t._version, host))
    except AttributeError:      # exotic tensor subclasses without a __dict__: just do not memoise
        pass
    return host


host_list = _host_list


def attach_host_copy(t, host):
    """Record the host value of a freshly built device tensor (shapes, start indices) so that `host_list` never has
    to read it back: the producer knew the numbers before it uploaded them."""
    try:
        setattr(t, _ATTR, (t._version, host))
    except AttributeError:
        pass
    return t


_pyramid_cache = {}


def pyramid_tensors(shapes, device):
    """(spatial_shapes (L,2), level_start_index (L,)) int64 device tensors for a pyramid given as host numbers, with
    their host copies attached; uploaded once per (shapes, device) and reused by every later forward."""
    shapes = tuple((int(h), int(w)) for h, w in shapes)
    key = (shapes, str(device))
    hit = _pyramid_cache.get(key)
    if hit is None:
        if len(_pyramid_cache) > 64:
            _pyramid_cache.clear()
        starts, acc = [], 0
        for h, w in shapes:
            starts.append(acc)
            acc += h * w
        hit = (attach_host_copy(torch.as_tensor(shapes, dtype=torch.long).to(device), [list(s) for s in shapes]),
               attach_host_copy(torch.as_tensor(starts, dtype=torch.long).to(device), starts))
        _pyramid_cache[key] = hit
    return hit


def _offsets_table(temporal_offsets):
    """list of T per-frame offset tensors (or one (T, Wt) tensor) -> list of lists, with a single device read"""
    if isinstance(temporal_offsets, torch.Tensor):
        return _host_list(temporal_offsets)
    tensors = [o for o in temporal_offsets if isinstance(o, torch.Tensor)]
    if len(tensors) != len(temporal_offsets) or not tensors:
        return [_host_list(o) for o in temporal_offsets]
    first = tensors[0]
    key = tuple((weakref.ref(o), o._version) for o in tensors)
    hit = getattr(first, _ATTR + "_table", None)
    if hit is not None and len(hit[0]) == len(key) and all(a[0]() is b[0]() and a[1] == b[1] for a, b in zip(hit[0], key)):
        return hit[1]
    if len({o.numel() for o in tensors}) == 1:
        table = torch.stack([o.reshape(-1) for o in tensors]).tolist()      # one kernel, one read
    else:
        table = [o.tolist() for o in tensors]
    try:
        setattr(first, _ATTR + "_table", (key, table))
    except AttributeError:
        pass
    return table


_geom_cache = {}


def from_reference_args(n_frames, input_spatial_shapes, input_level_start_index, temporal_offsets):
    """Build (and memoise by VALUE) the geometry from the arguments the reference modules receive
    (ms_deform_attn.py:268-284): the (current, temporal) shape / start-index pairs and the list of
    per-frame temporal offset tensors."""
    cur_shapes = input_spatial_shapes[0] if isinstance(input_spatial_shapes, (tuple, list)) else input_spatial_shapes
    cur_lsi = input_level_start_index[0] if isinstance(input_level_start_index, (tuple, list)) else input_level_start_index
    shapes = tuple(tuple(r) for r in _host_list(cur_shapes))
    lsi = tuple(_host_list(cur_lsi))
    offs = _offsets_table(temporal_offsets)
    table = tuple(tuple(int(o) + t for o in row) for t, row in enumerate(offs))
    # The whole-clip op derives the temporal halves of the pairs itself (every sampled frame has the query frame's
    # pyramid, laid out like it: what devis_transformer.py:97,118,153-154 builds).  The reference honours whatever it is
    # handed, so anything else must be refused, not silently mis-evaluated.  Read once per tensor object (memoised).
    wt = len(table[0]) if table else 0
    if isinstance(input_spatial_shapes, (tuple, list)) and len(input_spatial_shapes) > 1 and wt \
            and input_spatial_shapes[1] is not None:
        tshapes = tuple(tuple(r) for r in _host_list(input_spatial_shapes[1]))
        if tshapes != shapes * wt:
            raise RuntimeError("temporal spatial shapes must be the current shapes repeated t_window times "
                               f"(got {tshapes}, current {shapes}, t_window {wt})")
    if isinstance(input_level_start_index, (tuple, list)) and len(input_level_start_index) > 1 and wt \
            and input_level_start_index[1] is not None:
        tlsi = tuple(_host_list(input_level_start_index[1]))
        frame_rows = max(st + h * w for st, (h, w) in zip(lsi, shapes))
        if tlsi != tuple(j * frame_rows + st for j in range(wt) for st in lsi):
            raise RuntimeError("temporal level_start_index must be the per-frame start indices offset by one frame's rows "
                               "per temporal slot")
    return _memoised(n_frames, shapes, lsi, table)


def _memoised(n_frames, shapes, lsi, table):
    key = (n_frames, shapes, lsi, table)
    geom = _geom_cache.get(key)
    if geom is None:
        if len(_geom_cache) > 64:
            _geom_cache.clear()
        geom = ClipGeometry(shapes, n_frames, table, lsi)
        _geom_cache[key] = geom
    return geom


def batch_geometry(batch, input_spatial_shapes, input_level_start_index):
    """Geometry of MSDeformAttn's batched op for the whole-clip kernels: the batch of images is the frame axis and
    there are no temporal slots (no frame table).  Host values read as in from_reference_args (memoised per tensor
    object and version); the geometry is memoised by value."""
    shapes = tuple(tuple(int(x) for x in r) for r in _host_list(input_spatial_shapes))
    lsi = tuple(int(x) for x in _host_list(input_level_start_index))
    return _memoised(int(batch), shapes, lsi, None)


def op_geometry(n_frames, spatial_shapes, level_start_index, temporal_spatial_shapes, temporal_level_start_index,
                temporal_offsets, frame_offsets):
    """The geometry inside the ops: from the current pyramid tensors, the optional temporal halves of the reference's
    (current, temporal) pairs (validated as in from_reference_args) and the frame offsets -- T per-frame tensors of
    t_window offsets or one (T, t_window) tensor (`temporal_offsets`), or the same numbers as a row-major list of ints
    (`frame_offsets`); both empty for a clip without temporal slots (MSDeformAttn's batch)."""
    if frame_offsets:
        wt = len(frame_offsets) // n_frames
        offs = [list(frame_offsets[t * wt:(t + 1) * wt]) for t in range(n_frames)]
    elif temporal_offsets:
        offs = temporal_offsets[0] if len(temporal_offsets) == 1 and temporal_offsets[0].dim() == 2 else temporal_offsets
    else:
        return batch_geometry(n_frames, spatial_shapes, level_start_index)
    return from_reference_args(n_frames, (spatial_shapes, temporal_spatial_shapes),
                               (level_start_index, temporal_level_start_index), offs)
