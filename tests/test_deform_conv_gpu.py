"""GPU parity of the modulated deformable convolution (devis_b200.deform_conv, C ABI devis_dcn_im2col / devis_dcn_col2im)
against fixtures produced by torchvision.ops.deform_conv2d on CPU (the operator the reference's mask head calls,
deformable_segmentation.py:265) and by the reference's own ModulatedDeformableConv2d / MaskHeadConv modules.

Tolerances (normalised max error): float64 1e-12; float32 forward 1e-5, gradients 1e-4 (the north-star's op tolerances;
the float32 figures include the cuBLAS GEMM with the weights, run with TF32 off).
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, nmax

pytestmark = pytest.mark.gpu

FUSED_CASES = ["dcn_fused_c32_o16", "dcn_fused_c72_o32", "dcn_fused_c16_o1", "dcn_fused_c8_o4_s2", "dcn_fused_c40_o64",
               "dcn_fused_c20_o2", "dcn_fused_c136_o8_k1", "dcn_fused_c16_o16_s2"]
DCN_CASES = ["dcn_k3_mask", "dcn_k3_c24", "dcn_k3_c40", "dcn_stride2_dil2_nomask", "dcn_k1", "dcn_c33",
             "dcn_fused_c32_o16", "dcn_fused_c72_o32", "dcn_fused_c16_o1", "dcn_fused_c8_o4_s2", "dcn_fused_c40_o64",
             "dcn_fused_c20_o2", "dcn_fused_c136_o8_k1", "dcn_fused_c16_o16_s2"]
GRAD_KEYS = (("x", "gx"), ("offset", "goffset"), ("weight", "gweight"), ("bias", "gbias"), ("mask", "gmask"))


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _run(g, dtype, channels_last=False):
    from devis_b200.deform_conv import deform_conv2d
    t = lambda k: torch.from_numpy(g[k]).to("cuda", dtype)
    st, pd, dl, use_mask = [int(v) for v in g["cfg"]]
    names = ["x", "offset", "weight", "bias"] + (["mask"] if use_mask else [])
    leaves = [t(k).clone() for k in names]
    if channels_last:
        leaves[0] = leaves[0].contiguous(memory_format=torch.channels_last)
    leaves = [x.requires_grad_(True) for x in leaves]
    out = deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], stride=st, padding=pd, dilation=dl,
                        mask=leaves[4] if use_mask else None)
    out.backward(t("gout"))
    return out.detach(), dict(zip(names, [x.grad for x in leaves]))


@pytest.mark.parametrize("name", DCN_CASES)
def test_fp64_matches_torchvision_fixture(name):
    from devis_b200 import _lib
    g = load_golden(name)
    before = _lib.launch_count()
    out, grads = _run(g, torch.float64)
    assert _lib.launch_count() >= before + 2, "the CUDA kernels were not launched"
    assert out.shape == g["out"].shape
    assert nmax(out.cpu().numpy(), g["out"]) < 1e-12
    for k, key in GRAD_KEYS:
        if k in grads:
            assert nmax(grads[k].cpu().numpy(), g[key]) < 1e-12, k


@pytest.mark.parametrize("name", DCN_CASES)
@pytest.mark.parametrize("channels_last", [False, True])
def test_fp32_within_tolerance(name, channels_last):
    from devis_b200 import _lib, deform_conv
    g = load_golden(name)
    before = _lib.launch_count()
    out, grads = _run(g, torch.float32, channels_last)
    if name in FUSED_CASES:      # weight packing, forward, data gradients, im2col for the weight gradient
        cout, cin, kh, kw = g["weight"].shape
        assert deform_conv._fused_form(cin, cout, kh, kw, torch.float32) & 1
        assert _lib.launch_count() - before >= 2, "the CUDA kernels were not launched"
    assert nmax(out.cpu().numpy(), g["out"]) < 1e-5
    for k, key in GRAD_KEYS:
        if k in grads:
            assert nmax(grads[k].cpu().numpy(), g[key]) < 1e-4, k


@pytest.mark.parametrize("name", FUSED_CASES)
def test_fused_and_im2col_forms_agree(name):
    """the two kernel families of this library on the same layer (float32), and both against the fixture"""
    from devis_b200 import deform_conv
    g = load_golden(name)
    tc = deform_conv.set_tensor_core(False)        # the two CUDA-core families; the tensor-core form has its own tests
    try:
        out_f, grads_f = _run(g, torch.float32)
        old = deform_conv.set_fused(False)
        try:
            out_u, grads_u = _run(g, torch.float32)
        finally:
            deform_conv.set_fused(old)
    finally:
        deform_conv.set_tensor_core(tc)
    assert nmax(out_f.cpu().numpy(), out_u.cpu().numpy()) < 1e-5
    for k in grads_f:
        assert nmax(grads_f[k].cpu().numpy(), grads_u[k].cpu().numpy()) < 1e-4, k
        assert nmax(grads_u[k].cpu().numpy(), g[dict(GRAD_KEYS)[k]]) < 1e-4, k


@pytest.mark.parametrize("name", FUSED_CASES)
def test_fused_forward_inference_mode(name):
    """no autograd graph: every served layer takes the fused forward kernels (lane-group or constant-bank, the latter
    with several 16/32-channel tiles and kernel-position chunks where the weights exceed the bank)"""
    from devis_b200 import _lib, deform_conv
    from devis_b200.deform_conv import deform_conv2d
    g = load_golden(name)
    t = lambda k: torch.from_numpy(g[k]).to("cuda", torch.float32)
    st, pd, dl, use_mask = [int(v) for v in g["cfg"]]
    cout, cin, kh, kw = g["weight"].shape
    assert deform_conv._fused_form(cin, cout, kh, kw, torch.float32) & 1
    w = t("weight")
    assert int(_lib.load().devis_dcn_packed_weight_elems(cin, cout, kh, kw)) > 0
    calls = []
    real_pack = deform_conv._packed_weight
    deform_conv._packed_weight = lambda weight: (calls.append(1), real_pack(weight))[1]
    tc = deform_conv.set_tensor_core(False)        # (72 -> 32 would otherwise take the tensor-core forward)
    try:
        with torch.no_grad():
            out = deform_conv2d(t("x"), t("offset"), w, t("bias"), stride=st, padding=pd, dilation=dl,
                                mask=t("mask") if use_mask else None)
    finally:
        deform_conv._packed_weight = real_pack
        deform_conv.set_tensor_core(tc)
    assert calls                                                                # went through the fused function
    with torch.no_grad():
        again = deform_conv2d(t("x"), t("offset"), w, None, stride=st, padding=pd, dilation=dl,
                              mask=t("mask") if use_mask else None)
    assert nmax(out.cpu().numpy(), g["out"]) < 1e-5
    assert nmax((again + t("bias")[None, :, None, None]).cpu().numpy(), g["out"]) < 1e-5


def test_fused_forward_without_grad_and_partial_grads():
    """inference call (no autograd graph) and a call where only the offsets need gradients"""
    from devis_b200 import _lib
    from devis_b200.deform_conv import deform_conv2d
    g = load_golden("dcn_fused_c32_o16")
    t = lambda k: torch.from_numpy(g[k]).to("cuda", torch.float32)
    with torch.no_grad():
        out = deform_conv2d(t("x"), t("offset"), t("weight"), t("bias"), padding=1, mask=t("mask"))
    assert nmax(out.cpu().numpy(), g["out"]) < 1e-5
    off = t("offset").requires_grad_(True)
    before = _lib.launch_count()
    out = deform_conv2d(t("x"), off, t("weight"), None, padding=1, mask=t("mask"))
    out.backward(t("gout"))
    assert _lib.launch_count() - before <= 4          # pack (2 layouts), forward, one data-gradient kernel; no weight gradient
    assert nmax(off.grad.cpu().numpy(), g["goffset"]) < 1e-4


def test_fused_path_sees_weight_changes_made_through_parameter_data():
    """ADVICE round 1 (medium): writes through ``Parameter.data`` (nn.Module.to, EMA / weight-swap code) do not bump
    ``_version``; the fused path must still read the CURRENT weight -- it repacks on every call"""
    from devis_b200.deform_conv import deform_conv2d
    g = load_golden("dcn_fused_c32_o16")
    t = lambda k: torch.from_numpy(g[k]).to("cuda", torch.float32)
    w = torch.nn.Parameter(t("weight"))
    args = (t("x"), t("offset"))
    with torch.no_grad():
        first = deform_conv2d(*args, w, t("bias"), padding=1, mask=t("mask"))
        version = w._version
        w.data.mul_(2.0)                                   # in place through .data: _version unchanged
        assert w._version == version
        second = deform_conv2d(*args, w, None, padding=1, mask=t("mask"))
        w.data = t("weight") * 3.0                         # set_data: what Module.to() / .cuda() do
        third = deform_conv2d(*args, w, None, padding=1, mask=t("mask"))
    base = first - t("bias").view(1, -1, 1, 1)
    assert nmax(second.cpu().numpy(), (2.0 * base).cpu().numpy()) < 1e-6
    assert nmax(third.cpu().numpy(), (3.0 * base).cpu().numpy()) < 1e-6


def test_half_inputs_are_computed_in_float32_and_cast_back():
    g = load_golden("dcn_k3_c24")
    from devis_b200.deform_conv import deform_conv2d
    t = lambda k: torch.from_numpy(g[k]).to("cuda", torch.bfloat16)
    out = deform_conv2d(t("x"), t("offset"), t("weight"), t("bias"), padding=1, mask=t("mask"))
    assert out.dtype == torch.bfloat16
    want = deform_conv2d(t("x").float(), t("offset").float(), t("weight").float(), t("bias").float(), padding=1,
                         mask=t("mask").float())
    assert nmax(out.float().cpu().numpy(), want.cpu().numpy()) < 1e-2


def test_matches_installed_torchvision_cuda_op_at_mask_head_shape():
    """same inputs through torchvision's CUDA operator (third-party baseline) at one real mask-head layer shape:
    136 -> 64 channels at 23x40 (SURVEY.md appendix A, config 4), a handful of instances"""
    tv = pytest.importorskip("torchvision.ops")
    from devis_b200.deform_conv import deform_conv2d
    gen = torch.Generator(device="cuda").manual_seed(5)
    rn = lambda *s: torch.randn(*s, generator=gen, device="cuda")
    n, cin, cout, h, w = 6, 136, 64, 23, 40
    x, wt, b = rn(n, cin, h, w), rn(cout, cin, 3, 3) / 35, rn(cout)
    off, m = 2 * rn(n, 18, h, w), 2 * torch.sigmoid(rn(n, 9, h, w))
    gout = rn(n, cout, h, w)
    res = []
    for fn in (deform_conv2d, tv.deform_conv2d):
        leaves = [t.clone().requires_grad_(True) for t in (x, off, wt, b, m)]
        try:
            out = fn(leaves[0], leaves[1], leaves[2], leaves[3], padding=1, mask=leaves[4])
        except (RuntimeError, NotImplementedError) as exc:      # torchvision built without its CUDA ops
            pytest.skip(f"torchvision CUDA deform_conv2d unavailable: {exc}")
        out.backward(gout)
        res.append([out.detach()] + [t.grad for t in leaves])
    for name, a, c in zip(("out", "gx", "goffset", "gweight", "gbias", "gmask"), *res):
        assert nmax(a.cpu().numpy(), c.cpu().numpy()) < (1e-5 if name == "out" else 1e-4), name


def _load_sd(module, g, dtype):
    module = module.to(dtype)          # before loading: the fixtures are float64
    sd = {k[3:]: torch.from_numpy(v).to(dtype) for k, v in g.items() if k.startswith("sd.")}
    module.load_state_dict(sd, strict=True)
    return module.to("cuda")


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-11), (torch.float32, 1e-4)])
def test_modulated_layer_matches_reference_module(dtype, tol):
    """reference ModulatedDeformableConv2d (deformable_segmentation.py:244-267): its state dict loads unchanged;
    output, input gradient and every parameter gradient"""
    from devis_b200.deformable_segmentation import ModulatedDeformableConv2d
    g = load_golden("dcn_mod_layer")
    layer = _load_sd(ModulatedDeformableConv2d(12, 8, 3, padding=1, bias=True), g, dtype)
    x = torch.from_numpy(g["x"]).to("cuda", dtype).requires_grad_(True)
    with torch.backends.cudnn.flags(enabled=dtype != torch.float64):   # cuDNN's double convolutions are not double-accurate
        y = layer(x)
        y.backward(torch.from_numpy(g["gout"]).to("cuda", dtype))
    assert nmax(y.detach().cpu().numpy(), g["out"]) < tol
    assert nmax(x.grad.cpu().numpy(), g["gx"]) < tol
    for k, p in layer.named_parameters():
        assert nmax(p.grad.cpu().numpy(), g["pg." + k]) < tol, k


def _run_mask_head(dtype, layer_check=None):
    import devis_b200.deformable_segmentation as seg
    g = load_golden("dcn_mask_head")
    dim, nheads, n_inst, *fpn_dims = [int(v) for v in g["cfg"]]
    head = _load_sd(seg.MaskHeadConv(dim, fpn_dims, nheads, True, ["/32", "/16"], 2), g, dtype)
    feats = [torch.from_numpy(g[f"feat{i}"]).to("cuda", dtype).requires_grad_(True) for i in range(3)]
    att = [torch.from_numpy(g[f"att{i}"]).to("cuda", dtype) for i in range(2)]
    expand = lambda t, n: t.unsqueeze(1).repeat(1, int(n), 1, 1, 1).flatten(0, 1)
    orig = seg.deform_conv2d
    if layer_check is not None:
        def checked(input, offset, weight, bias=None, stride=(1, 1), padding=(0, 0), dilation=(1, 1), mask=None):
            out = orig(input, offset, weight, bias, stride, padding, dilation, mask)
            layer_check(input, offset, weight, bias, padding, mask, out)
            return out
        seg.deform_conv2d = checked
    try:
        with torch.backends.cudnn.flags(enabled=dtype != torch.float64):
            y = head(feats, att, n_inst, expand)
            y.backward(torch.from_numpy(g["gout"]).to("cuda", dtype))
    finally:
        seg.deform_conv2d = orig
    return g, y.detach(), feats


def test_mask_head_matches_reference_module_fp64():
    """reference MaskHeadConv (deformable_segmentation.py:323-380) with deformable layers: five stacked modulated
    deformable convolutions + GroupNorm + the FPN adapters; output and feature gradients"""
    g, y, feats = _run_mask_head(torch.float64)
    assert nmax(y.cpu().numpy(), g["out"]) < 1e-10
    for i, f in enumerate(feats):
        assert nmax(f.grad.cpu().numpy(), g[f"gfeat{i}"]) < 1e-10, i


def test_mask_head_fp32_every_layer_matches_oracle_on_identical_inputs():
    """float32: rounding differences are amplified from layer to layer through the offset branches (a 1e-7 change of an
    offset moves every sample of the next layer), so the end-to-end error of ANY float32 implementation against the
    float64 fixture is ~1e-2.  The meaningful float32 statement is per layer: each of the five deformable convolutions
    (im2col, lane-group and constant-bank kernels all occur) agrees with the float64 oracle evaluated on the very inputs
    it received -- its output, and the gradients of its input, offset, weight, bias and mask for the grad_out it
    received in the backward."""
    import devis_b200.deformable_segmentation as seg
    from oracle.deform_conv_torch import deform_conv2d_torch
    layers = []
    orig = seg.deform_conv2d

    def capturing(input, offset, weight, bias=None, stride=(1, 1), padding=(0, 0), dilation=(1, 1), mask=None):
        # fresh graph nodes in front of the layer: the gradients hooked on them are this call's alone (the input also
        # feeds the offset and mask branches, the weight is a Parameter)
        rec = {"args": [input, offset, weight, bias, mask], "padding": padding, "grads": {}}
        ins = []
        for i, t in enumerate(rec["args"]):
            if t is not None and t.requires_grad:
                t = t.view_as(t)
                t.register_hook(lambda gr, i=i: rec["grads"].__setitem__(i, gr.detach().clone()))
            ins.append(t)
        out = orig(ins[0], ins[1], ins[2], ins[3], stride, padding, dilation, ins[4])
        out.register_hook(lambda gr: rec.__setitem__("gout", gr.detach().clone()))
        rec["out"] = out.detach()
        layers.append(rec)
        return out

    seg.deform_conv2d = capturing
    try:
        g, y, feats = _run_mask_head(torch.float32)
    finally:
        seg.deform_conv2d = orig
    assert len(layers) == 5
    for li, rec in enumerate(layers):
        pad = (rec["padding"],) * 2 if isinstance(rec["padding"], int) else rec["padding"]
        leaves = [None if t is None else t.detach().double().requires_grad_(i in rec["grads"])
                  for i, t in enumerate(rec["args"])]
        ref = deform_conv2d_torch(leaves[0], leaves[1], leaves[2], leaves[3], (1, 1), pad, (1, 1), leaves[4])
        assert nmax(rec["out"].cpu().numpy(), ref.detach().cpu().numpy()) < 1e-5, li
        ref.backward(rec["gout"].double())
        assert set(rec["grads"]) >= {0, 1, 2}, (li, sorted(rec["grads"]))
        for i, got in rec["grads"].items():
            e = nmax(got.cpu().numpy(), leaves[i].grad.cpu().numpy())
            assert e < 1e-4, (li, ("input", "offset", "weight", "bias", "mask")[i], e)
    assert nmax(y.cpu().numpy(), g["out"]) < 0.2            # sanity only, see above
    assert all(torch.isfinite(f.grad).all() for f in feats)


def test_error_behaviour_and_empty_batch():
    from devis_b200.deform_conv import deform_conv2d
    x = torch.randn(1, 8, 5, 5, device="cuda")
    w = torch.randn(4, 8, 3, 3, device="cuda")
    off = torch.zeros(1, 18, 5, 5, device="cuda")
    with pytest.raises(RuntimeError):
        deform_conv2d(x.cpu(), off.cpu(), w.cpu(), padding=1)                    # no CPU path
    with pytest.raises(RuntimeError):
        deform_conv2d(x, off[:, :10], w, padding=1)                              # wrong offset channels
    with pytest.raises(RuntimeError):
        deform_conv2d(x, off, w[:, :4], padding=1)                               # groups = 2
    with pytest.raises(RuntimeError):
        deform_conv2d(x, off, w, padding=1, mask=torch.ones(1, 9, 4, 5, device="cuda"))
    # zero offsets and no mask: a plain convolution
    out = deform_conv2d(x, off, w, padding=1)
    assert nmax(out.cpu().numpy(), torch.nn.functional.conv2d(x, w, padding=1).cpu().numpy()) < 1e-5
    empty = deform_conv2d(x[:0], off[:0], w, padding=1)
    assert empty.shape == (0, 4, 5, 5)
