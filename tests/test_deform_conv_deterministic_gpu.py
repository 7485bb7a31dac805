"""Deterministic backward of the modulated deformable convolution under torch.use_deterministic_algorithms(True).

grad_input goes through 64-bit fixed point (DEVIS_MSDA_FLAG_DETERMINISTIC of devis_dcn_col2im_ex /
devis_dcn_fused_backward_ex): every gradient must be bit-identical from run to run and stay within the float32 bars of
the default mode.  grad_offset / grad_mask (fixed shuffle trees, written once) and the weight gradient (GEMM route under
the flag) are checked for the same property rather than assumed.  The last tests need no GPU: host-side validation of
the _ex entry points and the chunking rule."""
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import load_golden, nmax

DCN_CASES = ["dcn_k3_mask", "dcn_k3_c24", "dcn_k3_c40", "dcn_stride2_dil2_nomask", "dcn_k1", "dcn_c33",
             "dcn_fused_c32_o16", "dcn_fused_c72_o32", "dcn_fused_c16_o1", "dcn_fused_c8_o4_s2", "dcn_fused_c40_o64",
             "dcn_fused_c20_o2", "dcn_fused_c136_o8_k1", "dcn_fused_c16_o16_s2"]
GRAD_KEYS = (("x", "gx"), ("offset", "goffset"), ("weight", "gweight"), ("bias", "gbias"), ("mask", "gmask"))


@pytest.fixture
def no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _set_cublas_config(value):
    """CUBLAS_WORKSPACE_CONFIG = value (None: unset).  torch allocates a cuBLAS workspace once per handle and stream, at
    the size the variable names at that moment, but reads the variable again whenever it binds the workspace to a
    handle: changing it in a running process without dropping the cached workspaces lets cuBLAS write past the end of
    a smaller one (into whatever tensor follows it).  So the workspaces are released around every change."""
    if os.environ.get("CUBLAS_WORKSPACE_CONFIG") == value:
        return
    torch.cuda.synchronize()
    torch._C._cuda_clearCublasWorkspaces()
    if value is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = value


def _set_deterministic(on, warn_only=False):
    """torch.use_deterministic_algorithms with the cuBLAS workspace setting its own cuBLAS check asks for"""
    old = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
           os.environ.get("CUBLAS_WORKSPACE_CONFIG"))
    if on:
        _set_cublas_config(":4096:8")
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    return old


def _restore(old):
    torch.use_deterministic_algorithms(old[0], warn_only=old[1])
    _set_cublas_config(old[2])


@pytest.fixture
def deterministic(no_tf32):
    old = _set_deterministic(True)
    yield
    _restore(old)


def _run_golden(g, dtype):
    from devis_b200.deform_conv import deform_conv2d
    t = lambda k: torch.from_numpy(g[k]).to("cuda", dtype)
    st, pd, dl, use_mask = [int(v) for v in g["cfg"]]
    names = ["x", "offset", "weight", "bias"] + (["mask"] if use_mask else [])
    leaves = [t(k).clone().requires_grad_(True) for k in names]
    out = deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], stride=st, padding=pd, dilation=dl,
                        mask=leaves[4] if use_mask else None)
    out.backward(t("gout"))
    return out.detach(), {k: x.grad for k, x in zip(names, leaves)}


def _run_layer(fn, x, offset, weight, bias, mask, gout):
    """forward + backward of one layer through ``fn`` (deform_conv2d, or an autograd Function's apply);
    returns (out, [grad x, grad offset, grad weight, grad bias, grad mask])"""
    leaves = [t.clone().requires_grad_(True) for t in (x, offset, weight, bias, mask)]
    out = fn(*leaves)
    out.backward(gout)
    return out.detach(), [t.grad for t in leaves]


def _aux_launches():
    from devis_b200 import _lib
    return _lib.kernel_launches(_lib.KERNEL_AUX)


def _assert_equal_runs(a, b):
    assert torch.equal(a[0], b[0]), "out"
    for i, (p, q) in enumerate(zip(a[1], b[1])):
        assert torch.equal(p, q), f"gradient {i}"


def _assert_close(a, b, tol):
    for i, (p, q) in enumerate(zip([a[0]] + list(a[1]), [b[0]] + list(b[1]))):
        assert nmax(p.cpu().numpy(), q.cpu().numpy()) < tol, i


@pytest.mark.gpu
@pytest.mark.parametrize("name", DCN_CASES)
def test_every_form_is_bit_reproducible_and_accurate(deterministic, name):
    """im2col, lane-group fused, constant-bank fused and tensor-core forward forms: three runs give the same bits for
    the output and all five gradients, and every one of them is within the float32 bars of the float64 fixture"""
    g = load_golden(name)
    aux = _aux_launches()
    runs = [_run_golden(g, torch.float32) for _ in range(3)]
    assert _aux_launches() > aux, "the fixed-point scatter did not run"
    out, grads = runs[0]
    for other_out, other in runs[1:]:
        assert torch.equal(out, other_out)
        for k in grads:
            assert torch.equal(grads[k], other[k]), k
    assert nmax(out.cpu().numpy(), g["out"]) < 1e-5
    for k, key in GRAD_KEYS:
        if k in grads:
            assert nmax(grads[k].cpu().numpy(), g[key]) < 1e-4, k


def _layer_inputs(n, cin, cout, h, w, seed, collide=0):
    """random layer operands (3x3, padding 1, with mask).  collide > 0: 90 % of the taps of every plane are steered
    into ``collide`` pixels (plus a fixed fractional part), so thousands of grad_input contributions meet per element"""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(n, cin, h, w, generator=gen)
    off = torch.randn(n, 18, h, w, generator=gen) * 0.7
    if collide:
        ys = torch.randint(1, h - 1, (collide,), generator=gen).double() + 0.3
        xs = torch.randint(1, w - 1, (collide,), generator=gen).double() + 0.6
        pick = torch.randint(0, collide, (n, 9, h, w), generator=gen)
        steer = torch.rand(n, 9, h, w, generator=gen) < 0.9
        ho = torch.arange(h).double().view(1, 1, h, 1)
        wo = torch.arange(w).double().view(1, 1, 1, w)
        ky = torch.arange(9).double().div(3, rounding_mode="floor").view(1, 9, 1, 1)
        kx = torch.arange(9).double().remainder(3).view(1, 9, 1, 1)
        oh = (ys[pick] - (ho - 1 + ky)).float()
        ow = (xs[pick] - (wo - 1 + kx)).float()
        off[:, 0::2] = torch.where(steer, oh, off[:, 0::2])
        off[:, 1::2] = torch.where(steer, ow, off[:, 1::2])
    weight = torch.randn(cout, cin, 3, 3, generator=gen) / (3 * cin ** 0.5)
    bias = torch.randn(cout, generator=gen)
    mask = torch.rand(n, 9, h, w, generator=gen)
    gout = torch.randn(n, cout, h, w, generator=gen)
    return [t.cuda() for t in (x, off, weight, bias, mask, gout)]


def _dcn(x, offset, weight, bias, mask):
    from devis_b200.deform_conv import deform_conv2d
    return deform_conv2d(x, offset, weight, bias, padding=1, mask=mask)


@pytest.mark.gpu
def test_tensor_core_route(no_tf32):
    """the wide 264 -> 128 layer (60 instances at 12 x 20) through the tcgen05 forward and the col2im backward"""
    from devis_b200 import deform_conv
    x, off, weight, bias, mask, gout = _layer_inputs(60, 264, 128, 12, 20, seed=1)
    fn = lambda *t: deform_conv.IGemmDeformConv2dFunction.apply(*t, (1, 1), (1, 1), (1, 1))
    default = _run_layer(fn, x, off, weight, bias, mask, gout)
    old = _set_deterministic(True)
    try:
        a = _run_layer(fn, x, off, weight, bias, mask, gout)
        b = _run_layer(fn, x, off, weight, bias, mask, gout)
    finally:
        _restore(old)
    _assert_equal_runs(a, b)
    _assert_close(a, default, 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,h,w,n", [(32, 16, 90, 160, 2), (136, 64, 23, 40, 8)])
def test_collision_stress(no_tf32, cin, cout, h, w, n):
    """fused backward (32 -> 16 @ 90 x 160) and col2im (136 -> 64 @ 23 x 40) with most taps of a plane steered into
    a few pixels: bit-identical runs, within 1e-5 of the float scatter, and the fixed-point path demonstrably ran"""
    args = _layer_inputs(n, cin, cout, h, w, seed=2, collide=48 if h > 50 else 8)
    aux = _aux_launches()
    default = _run_layer(_dcn, *args)
    assert _aux_launches() == aux, "the default mode launched fixed-point helpers"
    old = _set_deterministic(True)
    try:
        a = _run_layer(_dcn, *args)
        assert _aux_launches() > aux, "the fixed-point scatter did not run"
        b = _run_layer(_dcn, *args)
    finally:
        _restore(old)
    _assert_equal_runs(a, b)
    _assert_close(a, default, 1e-5)


@pytest.mark.gpu
def test_mask_head_parameter_and_feature_gradients_repeat(deterministic):
    """MaskHeadConv (five stacked modulated deformable convolutions, GroupNorm, FPN adapters): two forward + backward
    passes give the same bits for every parameter gradient and every feature gradient"""
    import devis_b200.deformable_segmentation as seg
    g = load_golden("dcn_mask_head")
    dim, nheads, n_inst, *fpn_dims = [int(v) for v in g["cfg"]]
    sd = {k[3:]: torch.from_numpy(v).float() for k, v in g.items() if k.startswith("sd.")}
    expand = lambda t, n: t.unsqueeze(1).repeat(1, int(n), 1, 1, 1).flatten(0, 1)
    results = []
    for _ in range(2):
        head = seg.MaskHeadConv(dim, fpn_dims, nheads, True, ["/32", "/16"], 2).float()
        head.load_state_dict(sd, strict=True)
        head = head.cuda()
        feats = [torch.from_numpy(g[f"feat{i}"]).cuda().float().requires_grad_(True) for i in range(3)]
        att = [torch.from_numpy(g[f"att{i}"]).cuda().float() for i in range(2)]
        y = head(feats, att, n_inst, expand)
        y.backward(torch.from_numpy(g["gout"]).cuda().float())
        results.append((y.detach(), [f.grad for f in feats], {k: p.grad for k, p in head.named_parameters()}))
    (y0, f0, p0), (y1, f1, p1) = results
    assert torch.equal(y0, y1)
    for i, (a, b) in enumerate(zip(f0, f1)):
        assert torch.equal(a, b), i
    assert p0.keys() == p1.keys()
    for k in p0:
        assert torch.equal(p0[k], p1[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout", [(32, 16), (136, 64)])
def test_batch_chunks(deterministic, monkeypatch, cin, cout):
    """a small accumulator budget splits the data backward into several calls (each with its own fixed-point scale):
    within 1e-6 of the single call, and bit-identical from run to run"""
    from devis_b200 import deform_conv
    args = _layer_inputs(6, cin, cout, 24, 40, seed=3)
    whole = _run_layer(_dcn, *args)
    per_image = 24 * 40 * cin * 8
    monkeypatch.setattr(deform_conv, "_DET_ACC_CHUNK_BYTES", 2 * per_image)
    assert deform_conv._data_chunk(6, 24, 40, cin, 1, 6) == 2
    a = _run_layer(_dcn, *args)
    b = _run_layer(_dcn, *args)
    _assert_equal_runs(a, b)
    _assert_close(a, whole, 1e-6)


@pytest.mark.gpu
def test_warn_only_and_float64(no_tf32):
    """warn_only: float32 backward emits no devis_b200.deform_conv2d warning; float64 under the strict flag keeps
    raising torch's non-determinism alert (there is no fixed-point float64 form)"""
    args = _layer_inputs(2, 16, 8, 10, 12, seed=4)
    old = _set_deterministic(True, warn_only=True)
    try:
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            _run_layer(_dcn, *args)
        assert not [w for w in caught if "devis_b200.deform_conv2d" in str(w.message)]
    finally:
        _restore(old)
    old = _set_deterministic(True)
    try:
        with pytest.raises(RuntimeError, match="deterministic"):
            _run_layer(_dcn, *[t.double() for t in args])
    finally:
        _restore(old)


# ---- no GPU needed --------------------------------------------------------------------------------------------------

ERR_NULL, ERR_TOO_LARGE, ERR_WORKSPACE, ERR_UNSUPPORTED = -1, -5, -6, -8


def test_ex_entry_points_validate_on_the_host():
    """_ex validation codes, the workspace size, and that empty batches launch nothing -- no device involved"""
    from devis_b200 import _lib
    lib = _lib.load()
    det = _lib.FLAG_DETERMINISTIC
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below returns before any CUDA call
    dims = (2, 5, 7, 8, 5, 7, 3, 3, 1, 1, 1, 1, 1, 1)
    need = 2 * 5 * 7 * 8 * 8 + 16
    assert lib.devis_dcn_backward_workspace_bytes(2, 5, 7, 8, det) == need
    assert lib.devis_dcn_backward_workspace_bytes(2, 5, 7, 8, 0) == 0
    assert lib.devis_dcn_backward_workspace_bytes(0, 5, 7, 8, det) == 16

    def col2im(dims, gi, dtype, flags, ws, nbytes):
        return lib.devis_dcn_col2im_ex(None, None, None, None, gi, None, None, *dims, dtype, flags, ws, nbytes, None)

    def fused(dims, gi, flags, ws, nbytes):
        return lib.devis_dcn_fused_backward_ex(None, None, None, None, None, gi, None, None, *dims, 16, flags, ws,
                                               nbytes, None)

    for call in (lambda *a: col2im(a[0], a[1], _lib.F32, *a[2:]), fused):
        assert call(dims, fake, det, None, 0) == ERR_WORKSPACE                 # missing workspace
        assert call(dims, fake, det, fake, need - 1) == ERR_WORKSPACE          # short workspace
        assert call(dims, fake, det, fake, need) == ERR_NULL                   # valid: the operands are checked next
        assert call(dims, None, det, None, 0) == ERR_NULL                      # no grad_input: flag ignored
        assert call(dims, fake, 0, None, 0) == ERR_NULL                        # default mode needs no workspace
        # headroom: Ho * Wo * kh * kw contributions per element and image must stay below 2^26
        big = (1, 5, 7, 8, 1 << 13, 1 << 13, 1, 1, 1, 1, 0, 0, 1, 1)
        ok = big[:5] + ((1 << 13) - 1,) + big[6:]
        assert call(big, fake, det, fake, need) == ERR_TOO_LARGE
        assert call(ok, fake, det, fake, need) == ERR_NULL
    assert col2im(dims, fake, _lib.F64, det, fake, need) == ERR_UNSUPPORTED   # float64 has no fixed-point form
    before = lib.devis_msda_launch_count()
    empty = (0,) + dims[1:]
    assert col2im(empty, fake, _lib.F32, det, fake, 16) == 0
    assert fused(empty, fake, det, fake, 16) == 0
    assert col2im(empty, fake, _lib.F32, 0, None, 0) == 0
    assert lib.devis_msda_launch_count() == before


def test_chunk_rule():
    """deterministic data backward: at most _DET_ACC_CHUNK_BYTES of 8-byte accumulators per call; default mode keeps
    the caller's bound"""
    from devis_b200 import deform_conv
    assert deform_conv._DET_ACC_CHUNK_BYTES == 256 << 20
    per_image = 90 * 160 * 32 * 8
    assert deform_conv._data_chunk(1800, 90, 160, 32, 1, 1800) == (256 << 20) // per_image
    assert deform_conv._data_chunk(1800, 90, 160, 32, 0, 1800) == 1800
    assert deform_conv._data_chunk(1800, 90, 160, 32, 1, 10) == 10
    assert deform_conv._data_chunk(3, 4096, 4096, 64, 1, 3) == 1
    assert np.ceil(1800 / deform_conv._data_chunk(1800, 90, 160, 32, 1, 1800)) == 25
