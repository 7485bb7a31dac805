"""torch.compile / torch.export of the modules built on the custom ops (torch.ops.devis.*), on the GPU.

  * torch.library.opcheck of every op (schema, fake tensors, autograd registration, AOT dispatch) at small shapes;
  * torch.compile(fullgraph=True): aot_eager bit-identical to eager (outputs and every gradient, with the backward in
    deterministic mode so that both runs sum in the same order), inductor within the fp32 tolerances of the other
    module tests; no graph break, no recompilation on a second call with the same shapes;
  * flags toggled after compilation are obeyed (read inside the op bodies at run time);
  * torch.export at fixed shapes, run after run_decompositions();
  * CUDA-graph capture (GraphedLayer) of the ops; the launch counters prove which kernels served a compiled call.
"""
import copy
import os

import pytest
import torch

from conftest import load_golden, nmax

pytestmark = pytest.mark.gpu

DEV = "cuda"
SHAPES_L = ((12, 20), (6, 10))
S = sum(h * w for h, w in SHAPES_L)


def _t(x):
    return x.detach().float().cpu().numpy()


@pytest.fixture
def fresh_dynamo():
    import torch._dynamo
    torch._dynamo.reset()
    torch._dynamo.utils.counters.clear()
    yield torch._dynamo.utils.counters
    torch._dynamo.reset()


@pytest.fixture
def deterministic():
    """deterministic backward for the library (fixed-point grad_value / grad_input) and for ATen"""
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    old = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
           os.environ.get("CUBLAS_WORKSPACE_CONFIG"))
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
    torch.use_deterministic_algorithms(True, warn_only=True)
    MSDA.set_deterministic(True)
    yield
    MSDA.set_deterministic(False)
    torch.use_deterministic_algorithms(old[0], warn_only=old[1])
    if old[2] is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = old[2]


def _pyramid(n_slots=0):
    from devis_b200 import clip_geometry
    shapes, lsi = clip_geometry.pyramid_tensors(SHAPES_L, DEV)
    if not n_slots:
        return shapes, lsi
    tshapes = shapes.repeat(n_slots, 1)
    tlsi = torch.cat([tshapes.new_zeros(1), tshapes.prod(1).cumsum(0)[:-1]])
    return (shapes, tshapes), (lsi, tlsi)


def _randomize(mod, std=0.02):
    torch.manual_seed(1)
    with torch.no_grad():
        for name, p in mod.named_parameters():
            if "sampling_offsets" in name or "attention_weights" in name:
                p.normal_(0, std)


def _flat_tensors(out):
    if isinstance(out, torch.Tensor):
        return [out]
    res = []
    for o in out:
        res.extend(_flat_tensors(o) if isinstance(o, (list, tuple)) else ([o] if isinstance(o, torch.Tensor) else []))
    return res


def _fwd_bwd(fn, mod, args, kwargs=None, seed=0):
    """outputs, and the gradients of every floating input requiring grad and of every parameter, for a fixed cotangent"""
    for p in mod.parameters():
        p.grad = None
    leaves = [a.detach().clone().requires_grad_(a.requires_grad) if isinstance(a, torch.Tensor) and a.is_floating_point()
              else a for a in args]
    out = fn(*leaves, **(kwargs or {}))
    outs = _flat_tensors(out)
    g = torch.Generator(device=DEV).manual_seed(seed)
    diff = [o for o in outs if o.requires_grad]
    if diff:
        torch.autograd.backward(diff, [torch.randn(o.shape, device=DEV, generator=g, dtype=o.dtype) for o in diff])
    grads = [x.grad for x in leaves if isinstance(x, torch.Tensor) and x.requires_grad]
    grads += [p.grad for p in mod.parameters() if p.grad is not None]
    return [o.detach() for o in outs], grads


def _compare(a, b, exact, tol_out=2e-5, tol_grad=2e-4):
    (oa, ga), (ob, gb) = a, b
    assert len(oa) == len(ob) and len(ga) == len(gb) and ga
    for i, (x, y) in enumerate(zip(oa, ob)):
        assert x.shape == y.shape and x.dtype == y.dtype, i
        if exact:
            assert torch.equal(x, y), ("output", i)
        else:
            assert nmax(_t(x), _t(y)) < tol_out, ("output", i)
    for i, (x, y) in enumerate(zip(ga, gb)):
        if exact:
            assert torch.equal(x, y), ("grad", i)
        else:
            assert nmax(_t(x), _t(y)) < tol_grad, ("grad", i)


# ---- the module cases of the compile tests -----------------------------------------------------------------------------
def _msdeformattn(fused, ref_dim, mask, lq=40):
    from devis_b200 import MSDeformAttn
    torch.manual_seed(0)
    mod = MSDeformAttn(256, 2, 8, 4).to(DEV)
    mod.fuse_prologue = fused
    _randomize(mod)
    n = 2
    query = torch.randn(n, lq, 256, device=DEV, requires_grad=True)
    ref = torch.rand(n, lq, 2, ref_dim, device=DEV) * 0.6 + 0.2
    if ref_dim == 4:
        ref[..., 2:] *= 0.3
    x = torch.randn(n, S, 256, device=DEV, requires_grad=True)
    shapes, lsi = _pyramid()
    pm = None
    if mask:
        pm = torch.zeros(n, S, dtype=torch.bool, device=DEV)
        pm[1, -37:] = True
    return mod, (query, ref, x, shapes, lsi, pm), {}


def _encoder(fused, T=3):
    from devis_b200 import TemporalMSDeformAttnEncoder, synthetic
    torch.manual_seed(0)
    mod = TemporalMSDeformAttnEncoder(T, 256, 2, T - 1, 8, 4, 4).to(DEV)
    mod.fuse_prologue = fused
    _randomize(mod)
    shp, lsi = _pyramid(T - 1)
    offsets = [torch.tensor([d for d in range(-t, T - t) if d != 0], device=DEV) for t in range(T)]
    ref = synthetic.pixel_reference_points(SHAPES_L, T, DEV)
    args = (torch.randn(T, S, 256, device=DEV, requires_grad=True), ref,
            torch.randn(T, S, 256, device=DEV, requires_grad=True), shp, lsi, offsets)
    return mod, args, {}


def _decoder(fused, ref_dim, T=3, q=7):
    from devis_b200 import TemporalMSDeformAttnDecoder
    torch.manual_seed(0)
    mod = TemporalMSDeformAttnDecoder(T, 256, 2, T - 1, 8, 4, 4).to(DEV)
    mod.fuse_prologue = fused
    _randomize(mod)
    shp, lsi = _pyramid(T - 1)
    offsets = [[d for d in range(-t, T - t) if d != 0] for t in range(T)]       # python lists, as the trunk passes them
    ref = torch.rand(1, T * q, 2, ref_dim, device=DEV) * 0.6 + 0.2
    if ref_dim == 4:
        ref[..., 2:] *= 0.3
    args = (torch.randn(1, T * q, 256, device=DEV, requires_grad=True), ref,
            torch.randn(T, S, 256, device=DEV, requires_grad=True), shp, lsi, offsets)
    return mod, args, {}


class _Conv(torch.nn.Module):
    """deform_conv2d as a module (weight, bias as parameters) so the cases share one driver"""

    def __init__(self, cin, cout):
        super().__init__()
        torch.manual_seed(0)
        self.weight = torch.nn.Parameter(torch.randn(cout, cin, 3, 3, device=DEV) * 0.1)
        self.bias = torch.nn.Parameter(torch.randn(cout, device=DEV) * 0.1)

    def forward(self, x, offset, mask):
        from devis_b200.deform_conv import deform_conv2d
        return deform_conv2d(x, offset, self.weight, self.bias, padding=(1, 1), mask=mask)


def _conv_case(cin, cout, n=3, h=12, w=20):
    torch.manual_seed(0)
    x = torch.randn(n, cin, h, w, device=DEV, requires_grad=True)
    off = (torch.randn(n, 18, h, w, device=DEV) * 2).requires_grad_(True)
    m = torch.rand(n, 9, h, w, device=DEV).requires_grad_(True)
    return _Conv(cin, cout), (x, off, m), {}


@pytest.fixture
def dcn_form():
    from devis_b200 import deform_conv
    old = deform_conv.set_fused(True), deform_conv.set_tensor_core(True)
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False

    def select(form):
        deform_conv.set_fused(form == "fused")
        deform_conv.set_tensor_core(form == "igemm")
    yield select
    deform_conv.set_fused(old[0])
    deform_conv.set_tensor_core(old[1])
    torch.backends.cuda.matmul.allow_tf32 = old_tf32


# the fused form serves 32 -> 16 (forward and data backward); 64 -> 64 is a tensor-core layer; with both switched off
# every layer takes the im2col form
CONV_SHAPES = {"fused": (32, 16), "im2col": (32, 16), "igemm": (64, 64)}


def _mdc():
    from devis_b200.deformable_segmentation import ModulatedDeformableConv2d
    torch.manual_seed(0)
    mod = ModulatedDeformableConv2d(32, 16, 3, padding=1, bias=True).to(DEV)
    with torch.no_grad():
        mod.offset_conv.weight.normal_(0, 0.05)
        mod.modulator_conv.weight.normal_(0, 0.05)
    return mod, (torch.randn(3, 32, 12, 20, device=DEV, requires_grad=True),), {}


class _Head(torch.nn.Module):
    """MaskHeadConv with its call's non-tensor arguments bound (instances per batch, the expand function)"""

    def __init__(self, head, n_inst):
        super().__init__()
        self.head, self.n_inst = head, n_inst

    def forward(self, f0, f1, f2, a0, a1):
        expand = lambda t, n: t.unsqueeze(1).repeat(1, n, 1, 1, 1).flatten(0, 1)
        return self.head([f0, f1, f2], [a0, a1], self.n_inst, expand)


def _mask_head():
    import devis_b200.deformable_segmentation as seg
    g = load_golden("dcn_mask_head")
    dim, nheads, n_inst, *fpn_dims = [int(v) for v in g["cfg"]]
    sd = {k[3:]: torch.from_numpy(v).float() for k, v in g.items() if k.startswith("sd.")}
    head = seg.MaskHeadConv(dim, fpn_dims, nheads, True, ["/32", "/16"], 2).float()
    head.load_state_dict(sd, strict=True)
    feats = tuple(torch.from_numpy(g[f"feat{i}"]).to(DEV).float().requires_grad_(True) for i in range(3))
    att = tuple(torch.from_numpy(g[f"att{i}"]).to(DEV).float() for i in range(2))
    return _Head(head, n_inst).to(DEV), feats + att, {}


def _encoder_layer():
    from devis_b200 import DeVISTransformerEncoderLayer, synthetic
    from devis_b200.devis_transformer import DeVISTransformerEncoder
    torch.manual_seed(0)
    T = 3
    layer = DeVISTransformerEncoderLayer(256, 512, 0.0, "relu", T, T - 1, 2, 8, 4, 4).to(DEV)
    _randomize(layer)
    shp, lsi = _pyramid(T - 1)
    enc = DeVISTransformerEncoder(layer, 1, T - 1, True)
    offsets = enc.frame_offsets(T)
    ref = synthetic.pixel_reference_points(SHAPES_L, T, DEV)
    args = (torch.randn(T, S, 256, device=DEV, requires_grad=True), torch.randn(T, S, 256, device=DEV), ref, shp, lsi)
    return layer, args, {"temporal_offsets": offsets}


def _decoder_layer():
    from devis_b200 import DeVISTransformerDecoderLayer
    torch.manual_seed(0)
    T, q = 3, 7
    layer = DeVISTransformerDecoderLayer(256, 512, 0.0, "relu", T, T - 1, True, 2, 8, 4, 4).to(DEV)
    _randomize(layer)
    shp, lsi = _pyramid(T - 1)
    offsets = [[f - t for f in row] for t, row in enumerate([[f for f in range(T) if f != t] for t in range(T)])]
    ref = (torch.rand(1, T * q, 2, 4, device=DEV) * 0.6 + 0.2) * torch.tensor([1, 1, 0.3, 0.3], device=DEV)
    args = (torch.randn(1, T * q, 256, device=DEV, requires_grad=True), torch.randn(1, T * q, 256, device=DEV), ref,
            torch.randn(T, S, 256, device=DEV, requires_grad=True), shp, lsi)
    return layer, args, {"temporal_offsets": offsets}


MODULES = {
    **{f"msdeformattn_{'fused' if f else 'unfused'}_{'boxes' if r == 4 else 'points'}{'_mask' if m else ''}":
       (lambda f=f, r=r, m=m: _msdeformattn(f, r, m)) for f in (True, False) for r in (2, 4) for m in (False, True)},
    "msdeformattn_fused_pixel_queries": lambda: _msdeformattn(True, 2, True, lq=S),
    "encoder_fused": lambda: _encoder(True),
    "encoder_unfused": lambda: _encoder(False),
    **{f"decoder_{'fused' if f else 'unfused'}_{'boxes' if r == 4 else 'points'}": (lambda f=f, r=r: _decoder(f, r))
       for f in (True, False) for r in (2, 4)},
    "modulated_deformable_conv2d": _mdc,
    "mask_head_conv": _mask_head,
    "devis_encoder_layer": _encoder_layer,
    "devis_decoder_layer": _decoder_layer,
}
INDUCTOR = ["msdeformattn_fused_points_mask", "msdeformattn_unfused_boxes", "encoder_fused", "decoder_fused_boxes",
            "decoder_unfused_points", "modulated_deformable_conv2d", "mask_head_conv", "devis_decoder_layer"]


def _check_compiled(case, backend, counters, exact, tol_out=2e-5, tol_grad=2e-4):
    import torch._dynamo
    mod, args, kwargs = case()
    want = _fwd_bwd(mod, mod, args, kwargs)
    compiled = torch.compile(mod, fullgraph=True, backend=backend)
    got = _fwd_bwd(compiled, mod, args, kwargs)
    assert not counters["graph_break"], dict(counters["graph_break"])
    _compare(got, want, exact, tol_out, tol_grad)
    with torch._dynamo.config.patch(error_on_recompile=True):
        again = _fwd_bwd(compiled, mod, args, kwargs)
    _compare(again, want, exact, tol_out, tol_grad)


@pytest.mark.parametrize("name", list(MODULES))
def test_aot_eager_fullgraph_bit_identical(name, fresh_dynamo, deterministic):
    _check_compiled(MODULES[name], "aot_eager", fresh_dynamo, exact=True)


@pytest.mark.parametrize("form", ["fused", "im2col", "igemm"])
def test_deform_conv2d_forms_aot_eager_bit_identical(form, fresh_dynamo, deterministic, dcn_form):
    from devis_b200 import _lib
    dcn_form(form)
    fam = _lib.KERNEL_DCN_IGEMM
    before = _lib.kernel_launches(fam)
    _check_compiled(lambda: _conv_case(*CONV_SHAPES[form]), "aot_eager", fresh_dynamo, exact=True)
    # (no_grad calls take the tensor-core forward; with gradients the igemm layer keeps it, the others never do)
    assert (_lib.kernel_launches(fam) > before) == (form == "igemm")


@pytest.mark.parametrize("name", INDUCTOR)
def test_inductor_fullgraph_within_tolerance(name, fresh_dynamo, deterministic):
    # inductor fuses the GroupNorm / LayerNorm / softmax reductions around the ops and reorders their sums: through the
    # five GroupNorm layers of the mask head that moves the output by up to 1e-4 and the feature gradients by up to 1e-3
    # of their range (2e-5 / 2e-4 for the attention modules, as in the eager module tests)
    head = name == "mask_head_conv"
    _check_compiled(MODULES[name], "inductor", fresh_dynamo, exact=False, tol_out=1e-4 if head else 2e-5,
                    tol_grad=1e-3 if head else 2e-4)


@pytest.mark.parametrize("form", ["fused", "im2col", "igemm"])
def test_deform_conv2d_forms_inductor(form, fresh_dynamo, dcn_form):
    dcn_form(form)
    _check_compiled(lambda: _conv_case(*CONV_SHAPES[form]), "inductor", fresh_dynamo, exact=False)


def test_deform_conv2d_inference_forms_under_compile(fresh_dynamo, dcn_form):
    """no gradients: the fused forward serves 32 -> 16 and the tensor cores 64 -> 64, inside the compiled graph"""
    from devis_b200 import _lib
    dcn_form("igemm")
    from devis_b200 import deform_conv
    deform_conv.set_fused(True)
    for (cin, cout), fam in (((32, 16), _lib.KERNEL_DCN), ((64, 64), _lib.KERNEL_DCN_IGEMM)):
        mod, args, _ = _conv_case(cin, cout)
        with torch.no_grad():
            want = mod(*args)
            compiled = torch.compile(mod, fullgraph=True, backend="aot_eager")
            before = _lib.kernel_launches(fam)
            got = compiled(*args)
        assert _lib.kernel_launches(fam) > before
        assert torch.equal(got, want) and got.stride() == want.stride()
    assert not fresh_dynamo["graph_break"]


def test_whole_devis_encoder_and_decoder_match_eager(fresh_dynamo, deterministic):
    """DeVISTransformerEncoder / Decoder called as DeVISTransformer calls them (pyramid tensors with host copies
    attached): compiled without fullgraph -- their own host reads may split the graph -- and bit-identical to eager"""
    from devis_b200 import DeVISTransformer
    torch.manual_seed(0)
    T = 3
    tr = DeVISTransformer(d_model=256, num_frames=T, nhead=8, num_encoder_layers=2, num_decoder_layers=2,
                          dim_feedforward=512, dropout=0.0, num_feature_levels=2, enc_n_temporal_points=4,
                          dec_n_temporal_points=4).to(DEV)
    srcs = [torch.randn(T, 256, h, w, device=DEV) for h, w in SHAPES_L]
    masks = [torch.zeros(T, h, w, dtype=torch.bool, device=DEV) for h, w in SHAPES_L]
    pos = [torch.randn(T, 256, h, w, device=DEV) for h, w in SHAPES_L]
    src, _, posf, shapes, lsi, ratios = tr.prepare_data(srcs, masks, pos)
    src.requires_grad_(True)
    qe = torch.randn(1, 15, 256, device=DEV)
    tgt = torch.randn(1, 15, 256, device=DEV, requires_grad=True)
    ref = torch.rand(1, 15, 2, device=DEV) * 0.6 + 0.2

    class Trunk(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.encoder, self.decoder = tr.encoder, tr.decoder

        def forward(self, src, tgt):
            memory = self.encoder(src, shapes, lsi, ratios, posf)
            return self.decoder(tgt, ref, memory, shapes, lsi, ratios, qe)

    trunk = Trunk()
    want = _fwd_bwd(trunk, trunk, (src, tgt))
    got = _fwd_bwd(torch.compile(trunk, backend="aot_eager"), trunk, (src, tgt))
    _compare(got, want, exact=True)


def test_flags_toggled_after_compilation_are_obeyed(fresh_dynamo):
    """deterministic mode switched on after compiling: grad_value bit-identical run to run and equal to eager's, and
    the op reads the flag at run time (no recompilation needed)"""
    import torch._dynamo
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    from devis_b200 import clip_geometry, synthetic
    clip = synthetic.make_clip(n_frames=3, shapes=SHAPES_L, heads=8, channels=32, queries=60, dist="local", seed=0,
                               device=DEV)
    geom = clip_geometry.ClipGeometry(SHAPES_L, 3, clip["frame_table"])
    shapes, lsi, offs = geom.op_args()
    names = ("value", "loc_curr", "aw_curr", "loc_temporal", "aw_temporal")

    def op(v, lc, ac, lt, at):
        return torch.ops.devis.tmsda(v, lc, ac, lt, at, shapes, lsi, None, None, [], offs, None, 0, 0)

    def grad_value(fn):
        leaves = [clip[k].clone().requires_grad_(True) for k in names]
        fn(*leaves).backward(clip["grad_out"])
        return leaves[0].grad

    compiled = torch.compile(op, fullgraph=True, backend="aot_eager")
    grad_value(compiled)
    MSDA.set_deterministic(True)
    try:
        with torch._dynamo.config.patch(error_on_recompile=True):
            a, b = grad_value(compiled), grad_value(compiled)
        eager = grad_value(op)
    finally:
        MSDA.set_deterministic(False)
    assert torch.equal(a, b) and torch.equal(a, eager)


def test_fused_kernels_serve_the_compiled_module(fresh_dynamo):
    """launch counters: the compiled MSDeformAttn / encoder run the fused-prologue kernels forward and backward and
    nothing of the unfused op"""
    from devis_b200 import _lib
    fams = ("KERNEL_FUSED_FWD", "KERNEL_FUSED_BWD", "KERNEL_FWD_GROUPED", "KERNEL_FWD_GENERIC", "KERNEL_BWD_GROUPED",
            "KERNEL_BWD_GENERIC")
    for case in (lambda: _msdeformattn(True, 2, True), lambda: _encoder(True)):
        mod, args, kwargs = case()
        compiled = torch.compile(mod, fullgraph=True, backend="inductor")
        _fwd_bwd(compiled, mod, args, kwargs)
        before = {f: _lib.kernel_launches(getattr(_lib, f)) for f in fams}
        _fwd_bwd(compiled, mod, args, kwargs)
        delta = {f: _lib.kernel_launches(getattr(_lib, f)) - before[f] for f in fams}
        assert delta["KERNEL_FUSED_FWD"] >= 1 and delta["KERNEL_FUSED_BWD"] >= 1, delta
        assert all(delta[f] == 0 for f in fams[2:]), delta


EXPORT = {"msdeformattn_batched_mask": lambda: _msdeformattn(True, 2, True),
          "temporal_encoder": lambda: _encoder(True),
          "mask_head_conv": _mask_head}


@pytest.mark.parametrize("name", list(EXPORT))
def test_export_runs_after_decompositions(name):
    mod, args, kwargs = EXPORT[name]()
    mod.eval()
    with torch.no_grad():
        want = _flat_tensors(mod(*args, **kwargs))
        ep = torch.export.export(mod, args, kwargs)
        assert any("devis" in str(n.target) for n in ep.graph.nodes), "the custom op is not in the exported graph"
        got = _flat_tensors(ep.run_decompositions().module()(*args, **kwargs))
    assert len(got) == len(want)
    for x, y in zip(got, want):
        assert x.shape == y.shape and nmax(_t(x), _t(y)) < 2e-5


def test_graphed_layer_captures_the_ops():
    """GraphedLayer around the encoder attention with python-list frame offsets (the CPU frame-offset tensor path):
    replays of new values equal eager"""
    from devis_b200 import GraphedLayer
    T = 3
    mod, args, _ = _encoder(True, T)
    offsets = [[d for d in range(-t, T - t) if d != 0] for t in range(T)]
    q0, r0, x0, shp, lsi, _ = args
    fast = GraphedLayer(copy.deepcopy(mod), q0, r0, x0, shp, lsi, offsets)
    for seed in (3, 4):
        g = torch.Generator(device=DEV).manual_seed(seed)
        q = torch.randn(q0.shape, device=DEV, generator=g).requires_grad_(True)
        x = torch.randn(x0.shape, device=DEV, generator=g).requires_grad_(True)
        gout = torch.randn(T, S, 256, device=DEV, generator=g)
        out = mod(q, r0, x, shp, lsi, offsets)[0]
        out.backward(gout)
        q2, x2 = q.detach().clone().requires_grad_(True), x.detach().clone().requires_grad_(True)
        out2 = fast(q2, r0, x2, shp, lsi, offsets)[0]
        out2.backward(gout)
        torch.cuda.synchronize()
        assert nmax(_t(out2), _t(out)) < 1e-6
        assert nmax(_t(q2.grad), _t(q.grad)) < 1e-5 and nmax(_t(x2.grad), _t(x.grad)) < 1e-5


# ---- opcheck ------------------------------------------------------------------------------------------------------------
def _opcheck(op, args):
    res = torch.library.opcheck(op, args)
    assert all(v == "SUCCESS" for v in res.values()), res


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float64])
def test_opcheck_ms_deform_attn(dtype):
    from devis_b200 import synthetic
    torch.manual_seed(0)
    shapes, lsi = _pyramid()
    v = torch.randn(2, S, 4, 32, device=DEV, dtype=dtype)
    loc = (torch.rand(2, 9, 4, 2, 4, 2, device=DEV) * 0.8 + 0.1).to(torch.float64 if dtype == torch.float64 else torch.float32)
    aw = torch.softmax(torch.randn(2, 9, 4, 8, device=DEV), -1).view(2, 9, 4, 2, 4).to(loc.dtype)
    g = torch.randn(2, 9, 128, device=DEV, dtype=dtype)
    _opcheck(torch.ops.devis.ms_deform_attn.default, (v.requires_grad_(True), shapes, lsi, loc.requires_grad_(True),
                                                      aw.requires_grad_(True), 64, True))
    for need in (True, False):
        _opcheck(torch.ops.devis.ms_deform_attn_backward.default, (g, v.detach(), shapes, lsi, loc.detach(), aw.detach(),
                                                                   64, need))
    assert synthetic is not None


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16, torch.float64])
@pytest.mark.parametrize("temporal", [True, False])
def test_opcheck_tmsda(dtype, temporal):
    from devis_b200 import clip_geometry, synthetic
    clip = synthetic.make_clip(n_frames=3, shapes=SHAPES_L, heads=8, channels=32, queries=20, dist="local", seed=0,
                               device=DEV)
    geom = clip_geometry.ClipGeometry(SHAPES_L, 3, clip["frame_table"] if temporal else None)
    shapes, lsi, offs = geom.op_args()
    v = clip["value"].to(dtype)
    aux = lambda k: clip[k].to(torch.float64 if dtype == torch.float64 else torch.float32)
    lt, at = (aux("loc_temporal"), aux("aw_temporal")) if temporal else (None, None)
    req = lambda t: None if t is None else t.clone().requires_grad_(True)
    _opcheck(torch.ops.devis.tmsda.default, (req(v), req(aux("loc_curr")), req(aux("aw_curr")), req(lt), req(at), shapes,
                                             lsi, None, None, [], offs, None, 8, 8))
    g = clip["grad_out"].to(dtype)
    for need in (True, False):
        _opcheck(torch.ops.devis.tmsda_backward.default, (g, v, aux("loc_curr"), aux("aw_curr"), lt, at, shapes, lsi, [],
                                                          offs, None, 8, 8, need))


def _fused_operands(dtype, ref_dim, temporal, T=3, lq=20):
    from devis_b200 import clip_geometry
    torch.manual_seed(0)
    table = [[f for f in range(T) if f != t] for t in range(T)] if temporal else None
    geom = clip_geometry.ClipGeometry(SHAPES_L, T, table)
    shapes, lsi, offs = geom.op_args()
    v = torch.randn(T, S, 8, 32, device=DEV).to(dtype)
    ref = torch.rand(T, lq, 2, ref_dim, device=DEV) * 0.6 + 0.2
    if ref_dim == 4:
        ref[..., 2:] *= 0.3
    oc, lc = torch.randn(T, lq, 8, 2, 4, 2, device=DEV), torch.randn(T, lq, 8, 8, device=DEV)
    ot = torch.randn(T, lq, 8, (T - 1) * 2, 4, 2, device=DEV) if temporal else None
    lt = torch.randn(T, lq, 8, (T - 1) * 8, device=DEV) if temporal else None
    return v, ref, oc, lc, ot, lt, shapes, lsi, offs


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("variant", ["encoder", "decoder_boxes_sampling", "batch_mask"])
def test_opcheck_tmsda_fused(dtype, variant):
    temporal = variant != "batch_mask"
    ref_dim = 4 if "boxes" in variant else 2
    v, ref, oc, lc, ot, lt, shapes, lsi, offs = _fused_operands(dtype, ref_dim, temporal)
    mask = None
    if variant == "batch_mask":
        mask = torch.zeros(v.shape[0], S, dtype=torch.bool, device=DEV)
        mask[1, -40:] = True
    tref = 2 if variant.startswith("decoder") else 0
    want = variant == "decoder_boxes_sampling"
    req = lambda t: None if t is None else t.clone().requires_grad_(True)
    # (reference points without grad: d/d ref is a float-atomic sum whose last bits vary from run to run, which the
    # AOT check compares exactly enough to notice)
    _opcheck(torch.ops.devis.tmsda_fused.default, (req(v), ref, req(oc), req(lc), req(ot), req(lt), shapes, lsi, None,
                                                   None, [], offs, None, 0 if want else 8, 0 if want else 8, tref, want, mask,
                                                   not temporal))
    g = torch.randn(v.shape[0], ref.shape[1], 256, device=DEV).to(dtype)
    for need_gv, need_gref in ((True, False), (False, False)):
        _opcheck(torch.ops.devis.tmsda_fused_backward.default,
                 (g, v, ref, oc, lc, ot, lt, shapes, lsi, [], offs, None, 8, 8, tref, mask, need_gv, need_gref))


@pytest.mark.parametrize("form", ["fused", "im2col", "igemm"])
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_opcheck_deform_conv2d(form, channels_last, dtype, dcn_form):
    from devis_b200 import deform_conv
    if dtype == torch.float64 and form != "im2col":
        pytest.skip("the fused and tensor-core forms are float32 only")
    cin, cout = CONV_SHAPES[form]
    mod, (x, off, m), _ = _conv_case(cin, cout, n=2, h=6, w=10)
    x = x.detach().to(dtype)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    off, m, wt, b = off.detach().to(dtype), m.detach().to(dtype), mod.weight.detach().to(dtype), mod.bias.detach().to(dtype)
    geo = (1, 1, 1, 1, 1, 1)
    req = lambda t: t.clone().requires_grad_(True)
    if form == "fused":
        elems = deform_conv._packed_weight_elems(cin, cout, 3, 3, 1)
        op, extra, bwd = torch.ops.devis.deform_conv2d_fused.default, (elems,), torch.ops.devis.deform_conv2d_fused_backward
    elif form == "im2col":
        op, extra, bwd = torch.ops.devis.deform_conv2d_im2col.default, (), torch.ops.devis.deform_conv2d_im2col_backward
    else:
        op, extra, bwd = torch.ops.devis.deform_conv2d_igemm.default, (), torch.ops.devis.deform_conv2d_igemm_backward
    x_req = req(x) if not channels_last else x.clone(memory_format=torch.channels_last).requires_grad_(True)
    _opcheck(op, (x_req, req(off), req(wt), req(b), req(m)) + geo + extra)
    res = op(x, off, wt, b, m, *geo, *extra)
    g = torch.randn(res[0].shape, device=DEV, dtype=dtype)
    saved = res[2:] if form != "igemm" else ()
    form_arg = (deform_conv._fused_form(cin, cout, 3, 3, dtype),) if form == "fused" else ()
    for need in ((True, True, True, True, True), (False, False, True, False, False)):
        _opcheck(bwd.default, (g, x, res[1], off, wt, b, m, *saved, *geo, *form_arg, *need))
