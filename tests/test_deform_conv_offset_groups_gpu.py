"""Offset groups of the modulated deformable convolution on the GPU (offset of 2 * G * kh * kw channels, mask of
G * kh * kw; torchvision's offset_groups): the dcn_og_*.npz fixtures from torchvision's CPU operator, which form serves
a layer, the decomposition into G one-group convolutions at the mask head's layer sizes, torchvision's CUDA operator,
the _og entry points at G = 1 against the old ones, and the deterministic backward.

Tolerances (normalised max error) as in test_deform_conv_gpu.py: float64 1e-12; float32 forward 1e-5, gradients 1e-4
with TF32 off."""
import glob
import os

import pytest
import torch

from conftest import GOLDEN, load_golden, nmax

pytestmark = pytest.mark.gpu

OG_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "dcn_og_*.npz")))
FUSED_OG_CASES = [n for n in OG_CASES if n.startswith("dcn_og_fused_")]
GRAD_KEYS = (("x", "gx"), ("offset", "goffset"), ("weight", "gweight"), ("bias", "gbias"), ("mask", "gmask"))
# (name, Cin, Cout, H, W) of benchmarks/dcn_bench.py
LAYERS = [("lay1", 264, 264, 12, 20), ("lay2", 264, 128, 12, 20), ("lay3", 136, 64, 23, 40), ("lay4", 72, 32, 45, 80),
          ("lay5", 32, 16, 90, 160), ("out_lay", 16, 1, 90, 160)]


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _set_cublas_config(value):
    """CUBLAS_WORKSPACE_CONFIG = value (None: unset), releasing torch's cached cuBLAS workspaces around the change: torch
    sizes a workspace when it allocates it but reads the variable again when it binds it, so changing the variable in a
    running process without dropping the cached workspaces lets cuBLAS write past the end of a smaller one."""
    if os.environ.get("CUBLAS_WORKSPACE_CONFIG") == value:
        return
    torch.cuda.synchronize()
    torch._C._cuda_clearCublasWorkspaces()
    if value is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = value


@pytest.fixture
def deterministic():
    old = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
           os.environ.get("CUBLAS_WORKSPACE_CONFIG"))
    _set_cublas_config(":4096:8")
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(old[0], warn_only=old[1])
    _set_cublas_config(old[2])


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


def _check_fixture(g, out, grads, tol_out, tol_grad):
    assert out.shape == g["out"].shape
    assert nmax(out.cpu().numpy(), g["out"]) <= tol_out
    for k, key in GRAD_KEYS:
        if k in grads:
            assert nmax(grads[k].cpu().numpy(), g[key]) <= tol_grad, k


def test_fixture_list():
    assert len(OG_CASES) >= 12 and len(FUSED_OG_CASES) >= 3


@pytest.mark.parametrize("name", OG_CASES)
def test_fp64_matches_torchvision_fixture(name):
    from devis_b200 import _lib
    g = load_golden(name)
    before = _lib.launch_count()
    out, grads = _run(g, torch.float64)
    assert _lib.launch_count() >= before + 2, "the CUDA kernels were not launched"
    _check_fixture(g, out, grads, 1e-12, 1e-12)


@pytest.mark.parametrize("name", OG_CASES)
@pytest.mark.parametrize("channels_last", [False, True])
def test_fp32_within_tolerance_and_form(name, channels_last, monkeypatch):
    """float32 against the fixture; the lane-group fused form serves the fused cases (the weights are packed), every
    other case takes the im2col form, and the tensor-core forward never runs at G > 1"""
    from devis_b200 import _lib, deform_conv
    g = load_golden(name)
    cout, cin, kh, kw = g["weight"].shape
    og = g["offset"].shape[1] // (2 * kh * kw)
    assert og > 1
    fused = name in FUSED_OG_CASES
    assert (deform_conv._fused_form(cin, cout, kh, kw, torch.float32, og) == 3) == fused
    calls = []
    real_pack = deform_conv._packed_weight
    monkeypatch.setattr(deform_conv, "_packed_weight", lambda weight, *a: (calls.append(a), real_pack(weight, *a))[1])
    igemm = _lib.kernel_launches(_lib.KERNEL_DCN_IGEMM)
    out, grads = _run(g, torch.float32, channels_last)
    assert _lib.kernel_launches(_lib.KERNEL_DCN_IGEMM) == igemm
    assert calls == ([(og,)] if fused else [])
    _check_fixture(g, out, grads, 1e-5, 1e-4)


@pytest.mark.parametrize("name", FUSED_OG_CASES)
def test_fused_and_im2col_forms_agree(name):
    from devis_b200 import deform_conv
    g = load_golden(name)
    out_f, grads_f = _run(g, torch.float32)
    old = deform_conv.set_fused(False)
    try:
        out_u, grads_u = _run(g, torch.float32)
    finally:
        deform_conv.set_fused(old)
    assert nmax(out_f.cpu().numpy(), out_u.cpu().numpy()) < 1e-5
    for k in grads_f:
        assert nmax(grads_f[k].cpu().numpy(), grads_u[k].cpu().numpy()) < 1e-4, k


def _layer_operands(n, cin, cout, h, w, og, seed, dtype=torch.float64, collide=0):
    """random 3x3 / padding 1 operands with og offset groups.  collide > 0: 90 % of the taps of every plane and group
    are steered into ``collide`` pixels (plus a fixed fractional part), so many grad_input contributions meet per
    element"""
    gen = torch.Generator().manual_seed(seed)
    k = 9
    x = torch.randn(n, cin, h, w, generator=gen, dtype=torch.float64)
    off = torch.randn(n, 2 * og * k, h, w, generator=gen, dtype=torch.float64) * 1.5
    if collide:
        ys = torch.randint(1, h - 1, (collide,), generator=gen).double() + 0.3
        xs = torch.randint(1, w - 1, (collide,), generator=gen).double() + 0.6
        pick = torch.randint(0, collide, (n, og * k, h, w), generator=gen)
        steer = torch.rand(n, og * k, h, w, generator=gen) < 0.9
        ho = torch.arange(h).double().view(1, 1, h, 1)
        wo = torch.arange(w).double().view(1, 1, 1, w)
        kk = torch.arange(og * k) % k
        ky = kk.div(3, rounding_mode="floor").double().view(1, -1, 1, 1)
        kx = kk.remainder(3).double().view(1, -1, 1, 1)
        off[:, 0::2] = torch.where(steer, ys[pick] - (ho - 1 + ky), off[:, 0::2])
        off[:, 1::2] = torch.where(steer, xs[pick] - (wo - 1 + kx), off[:, 1::2])
    weight = torch.randn(cout, cin, 3, 3, generator=gen, dtype=torch.float64) / (3 * cin ** 0.5)
    bias = torch.randn(cout, generator=gen, dtype=torch.float64)
    mask = 2 * torch.rand(n, og * k, h, w, generator=gen, dtype=torch.float64)
    gout = torch.randn(n, cout, h, w, generator=gen, dtype=torch.float64)
    return [t.to("cuda", dtype) for t in (x, off, weight, bias, mask, gout)]


def _fwd_bwd(x, off, weight, bias, mask, gout):
    """deform_conv2d (padding 1) forward + backward: (out, [grad x, offset, weight, bias, mask])"""
    from devis_b200.deform_conv import deform_conv2d
    leaves = [t.clone().requires_grad_(True) for t in (x, off, weight, bias, mask)]
    out = deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], padding=1, mask=leaves[4])
    out.backward(gout)
    return out.detach(), [t.grad for t in leaves]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("layer", LAYERS, ids=[lay[0] for lay in LAYERS])
def test_decomposition_into_one_group_convolutions(layer, dtype):
    """at the mask head's layer sizes (6 instances) a G = 4 call equals the sum of four G = 1 calls on the channel
    slices (bias once), and its gradients are the concatenations of theirs"""
    _, cin, cout, h, w = layer
    og, k = 4, 9
    x, off, weight, bias, mask, gout = _layer_operands(6, cin, cout, h, w, og, seed=7, dtype=dtype)
    out, grads = _fwd_bwd(x, off, weight, bias, mask, gout)
    cg = cin // og
    parts = [_fwd_bwd(x[:, g * cg:(g + 1) * cg], off[:, 2 * g * k:2 * (g + 1) * k], weight[:, g * cg:(g + 1) * cg],
                      bias * (g == 0), mask[:, g * k:(g + 1) * k], gout) for g in range(og)]
    want_out = sum(p[0] for p in parts)
    want = [torch.cat([p[1][i] for p in parts], dim=1) for i in (0, 1, 2)]
    want.insert(3, parts[0][1][3])
    want.append(torch.cat([p[1][4] for p in parts], dim=1))
    tol_out, tol_grad = (1e-12, 1e-12) if dtype == torch.float64 else (1e-5, 1e-4)
    assert nmax(out.cpu().numpy(), want_out.cpu().numpy()) <= tol_out
    for i, (a, b) in enumerate(zip(grads, want)):
        assert nmax(a.cpu().numpy(), b.cpu().numpy()) <= tol_grad, i


def test_matches_installed_torchvision_cuda_op_with_offset_groups():
    """torchvision's CUDA operator at one real mask-head shape with G = 4: 136 -> 64 channels at 23 x 40, 6 instances"""
    tv = pytest.importorskip("torchvision.ops")
    from devis_b200.deform_conv import deform_conv2d
    x, off, wt, b, m, gout = _layer_operands(6, 136, 64, 23, 40, 4, seed=5, dtype=torch.float32)
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


def test_og_entry_points_at_one_group_equal_the_old_ones():
    """same operands through devis_dcn_*_og with offset_groups = 1 and through the entry points without the suffix:
    bit-identical results (grad_input through the fixed-point form, the float scatter's sum order varies run to run)"""
    from devis_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    p = lambda t: t.data_ptr() if t is not None else None
    det = _lib.FLAG_DETERMINISTIC
    for cin, cout, dtype in ((32, 16, torch.float32), (16, 1, torch.float32), (33, 3, torch.float32),
                             (24, 6, torch.float64)):
        n, h, w = 3, 20, 28
        x, off, weight, _, mask, gout = _layer_operands(n, cin, cout, h, w, 1, seed=11, dtype=dtype)
        xl = x.permute(0, 2, 3, 1).contiguous()
        dims = (n, h, w, cin, h, w, 3, 3, 1, 1, 1, 1, 1, 1)
        dt = _lib.F32 if dtype == torch.float32 else _lib.F64
        cols = [torch.empty(n * h * w, 9 * cin, device="cuda", dtype=dtype) for _ in range(2)]
        _lib.check(lib.devis_dcn_im2col(p(xl), p(off), p(mask), p(cols[0]), *dims, dt, st))
        _lib.check(lib.devis_dcn_im2col_og(p(xl), p(off), p(mask), p(cols[1]), *dims, 1, dt, st))
        assert torch.equal(cols[0], cols[1])
        gcols = torch.randn_like(cols[0])
        flags = det if dtype == torch.float32 else 0
        nbytes = int(lib.devis_dcn_backward_workspace_bytes(n, h, w, cin, flags))
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
        res = []
        for og_call in (False, True):
            gx, goff, gm = torch.empty_like(xl), torch.empty_like(off), torch.empty_like(mask)
            args = (p(xl), p(off), p(mask), p(gcols), p(gx), p(goff), p(gm), *dims)
            if og_call:
                _lib.check(lib.devis_dcn_col2im_og(*args, 1, dt, flags, p(ws), nbytes, st))
            else:
                _lib.check(lib.devis_dcn_col2im_ex(*args, dt, flags, p(ws), nbytes, st))
            res.append((gx, goff, gm))
        for i, (a, b) in enumerate(zip(*res)):
            if i == 0 and not flags:       # float64 grad_input: float atomics
                assert nmax(a.cpu().numpy(), b.cpu().numpy()) < 1e-12
            else:
                assert torch.equal(a, b), i
        if dtype != torch.float32 or cin % 4 or cout not in (1, 2, 4, 8, 16):
            continue
        assert lib.devis_dcn_fused_form_og(cin, cout, 3, 3, 1, dt) == lib.devis_dcn_fused_form(cin, cout, 3, 3, dt) == 3
        elems = int(lib.devis_dcn_packed_weight_elems(cin, cout, 3, 3))
        packed = [torch.empty(elems, device="cuda") for _ in range(2)]
        _lib.check(lib.devis_dcn_pack_weight(p(weight), p(packed[0]), cin, cout, 3, 3, st))
        _lib.check(lib.devis_dcn_pack_weight_og(p(weight), p(packed[1]), cin, cout, 3, 3, 1, st))
        assert torch.equal(packed[0], packed[1])
        outs = [torch.empty(n, h, w, cout, device="cuda") for _ in range(2)]
        _lib.check(lib.devis_dcn_fused_forward(p(xl), p(off), p(mask), p(packed[0]), None, p(outs[0]), *dims, cout, st))
        _lib.check(lib.devis_dcn_fused_forward_og(p(xl), p(off), p(mask), p(packed[0]), None, p(outs[1]), *dims, 1, cout,
                                                  st))
        assert torch.equal(outs[0], outs[1])
        gl = gout.permute(0, 2, 3, 1).contiguous()
        res = []
        for og_call in (False, True):
            gx, goff, gm = torch.empty_like(xl), torch.empty_like(off), torch.empty_like(mask)
            args = (p(xl), p(off), p(mask), p(packed[0]), p(gl), p(gx), p(goff), p(gm), *dims)
            if og_call:
                _lib.check(lib.devis_dcn_fused_backward_og(*args, 1, cout, det, p(ws), nbytes, st))
            else:
                _lib.check(lib.devis_dcn_fused_backward_ex(*args, cout, det, p(ws), nbytes, st))
            res.append((gx, goff, gm))
        for a, b in zip(*res):
            assert torch.equal(a, b)


def _aux_launches():
    from devis_b200 import _lib
    return _lib.kernel_launches(_lib.KERNEL_AUX)


@pytest.mark.parametrize("name", ["dcn_og_fused_c32_o16_g2", "dcn_og_fused_c16_o1_g4", "dcn_og_g4_c32",
                                  "dcn_og_c72_o32_g2", "dcn_og_g2_c66"])
def test_deterministic_fixtures(deterministic, name):
    """fused and im2col forms at G > 1 under torch.use_deterministic_algorithms(True): two runs give the same bits for
    the output and every gradient, within the float32 bars of the float64 fixture"""
    g = load_golden(name)
    aux = _aux_launches()
    (out, grads), (out2, grads2) = _run(g, torch.float32), _run(g, torch.float32)
    assert _aux_launches() > aux, "the fixed-point scatter did not run"
    assert torch.equal(out, out2)
    for k in grads:
        assert torch.equal(grads[k], grads2[k]), k
    _check_fixture(g, out, grads, 1e-5, 1e-4)


@pytest.mark.parametrize("cin,cout,h,w,n,og", [(32, 16, 90, 160, 2, 2), (72, 32, 45, 80, 4, 2), (16, 1, 45, 80, 4, 4)])
@pytest.mark.parametrize("collide", [0, 24])
def test_deterministic_collisions(cin, cout, h, w, n, og, collide):
    """zero offsets (every input element is reached by nine taps of each pixel neighbourhood) and taps steered into a
    few pixels, fused (32 -> 16, 16 -> 1) and im2col (72 -> 32) at G > 1: bit-identical deterministic runs, within 1e-5
    of the float scatter"""
    x, off, weight, bias, mask, gout = _layer_operands(n, cin, cout, h, w, og, seed=3, dtype=torch.float32,
                                                       collide=collide)
    if not collide:
        off = torch.zeros_like(off)
    args = (x, off, weight, bias, mask, gout)
    default = _fwd_bwd(*args)
    old = (torch.are_deterministic_algorithms_enabled(), os.environ.get("CUBLAS_WORKSPACE_CONFIG"))
    _set_cublas_config(":4096:8")
    torch.use_deterministic_algorithms(True)
    try:
        aux = _aux_launches()
        a = _fwd_bwd(*args)
        assert _aux_launches() > aux, "the fixed-point scatter did not run"
        b = _fwd_bwd(*args)
    finally:
        torch.use_deterministic_algorithms(old[0])
        _set_cublas_config(old[1])
    assert torch.equal(a[0], b[0])
    for i, (p, q) in enumerate(zip(a[1], b[1])):
        assert torch.equal(p, q), i
    for i, (p, q) in enumerate(zip([a[0]] + a[1], [default[0]] + default[1])):
        assert nmax(p.cpu().numpy(), q.cpu().numpy()) < 1e-5, i


def test_errors_empty_batch_and_no_mask():
    from devis_b200.deform_conv import deform_conv2d
    x = torch.randn(2, 8, 5, 5, device="cuda")
    w = torch.randn(4, 8, 3, 3, device="cuda")
    with pytest.raises(RuntimeError, match="divisible"):
        deform_conv2d(x[:, :6], torch.zeros(2, 72, 5, 5, device="cuda"), w[:, :6], padding=1)      # C % G != 0
    with pytest.raises(RuntimeError, match="multiple"):
        deform_conv2d(x, torch.zeros(2, 27, 5, 5, device="cuda"), w, padding=1)                   # not 2 * K * G
    with pytest.raises(RuntimeError, match="mask"):
        deform_conv2d(x, torch.zeros(2, 36, 5, 5, device="cuda"), w, padding=1,
                      mask=torch.ones(2, 9, 5, 5, device="cuda"))                                  # mask of G = 1
    off = torch.zeros(2, 36, 5, 5, device="cuda")
    empty = deform_conv2d(x[:0], off[:0], w, padding=1, mask=torch.ones(0, 18, 5, 5, device="cuda"))
    assert empty.shape == (0, 4, 5, 5)
    # zero offsets, no mask: every group samples the plain 3 x 3 neighbourhood -- an ordinary convolution
    out = deform_conv2d(x, off, w, padding=1)
    assert nmax(out.cpu().numpy(), torch.nn.functional.conv2d(x, w, padding=1).cpu().numpy()) < 1e-5
