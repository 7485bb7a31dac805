"""Every deformable-convolution kernel instantiation and launch shape against the float64 oracle.

The case table (dcn_cases.CASES; test_dcn_kernels_host.py checks that it reaches every instantiation) runs each form of
the library -- im2col / col2im, lane-group fused forward and backward, constant-bank forward, the weight-gradient kernel,
the tcgen05 implicit-GEMM forward -- at unequal kernel sizes, strides, paddings and dilations, partial tiles, more than
65535 batch items, and the mask head's real layers.  Offsets lie on a 2^-10 grid (every sampling coordinate is exact in
float32, so the float64 reference samples the same points) and a quarter of the coordinates are steered onto the edges
of the map: integers, H - 1, (-1, 0), exactly -1 and exactly H.

Reference: oracle/deform_conv_torch.py in float64 on the GPU (offset groups: the sum over groups of one-group calls on
the channel slices), evaluated on the very float32 values the kernels read, in batch slices.  Bounds:
  * float64 forms: normalised max error <= 1e-12;
  * float32: forward <= 1e-5 (tensor-core 3xTF32 forward 2e-5), gradients <= 1e-4, and element-wise
    |got - ref| <= tau * S for the output and the gradients of input, weight, bias and mask, where S is the oracle on
    |x|, |W|, |bias|, |mask| and |grad_out| with the same offsets (each of these quantities is multilinear in those
    operands, so S bounds the magnitude of its terms; where S = 0 the result must be exactly 0).  tau = 2^-16 for the
    CUDA-core kernels and 3xTF32, 2^-9 for a single-pass TF32 forward.  grad_offset: normalised max error <= 1e-4.
  * each float32 case runs twice more under torch.use_deterministic_algorithms(True): the two runs are bit-identical,
    meet the same bounds, and take the fixed-point grad_input forms and the GEMM route for grad_weight.  The fixed-point
    grad_input rounds every contribution to a quantum set by the largest possible contribution, so its element-wise
    bound is tau * S plus half a quantum per contribution the element receives (fixed_point_slack).
Every case also asserts which C entry points the Python layer called and how many kernels of each family were launched.
The largest |got - ref| / (tau * S) per kernel family is printed at the end of the module (and written as JSON to the
file named by DEVIS_DCN_HEADROOM_JSON, if set)."""
import json
import math
import os

import pytest
import torch

import dcn_cases as dc
from conftest import nmax

pytestmark = pytest.mark.gpu

TAU_FP32, TAU_TF32 = 2.0 ** -16, 2.0 ** -9
REF_SLICE_ELEMS = 4e7          # N * C * K * Ho * Wo per oracle slice (float64, a few GB of autograd state)
LAUNCHING = {"devis_dcn_im2col", "devis_dcn_im2col_og", "devis_dcn_col2im", "devis_dcn_col2im_ex", "devis_dcn_col2im_og",
             "devis_dcn_pack_weight", "devis_dcn_pack_weight_og", "devis_dcn_fused_forward", "devis_dcn_fused_forward_og",
             "devis_dcn_fused_backward", "devis_dcn_fused_backward_ex", "devis_dcn_fused_backward_og",
             "devis_dcn_weight_grad", "devis_dcn_igemm_pack_weight", "devis_dcn_igemm_forward"}
KEYS = ("gx", "goff", "gw", "gb", "gm")
F32_CASES = [c for c in dc.CASES if c.dtype == "float32"]
HEADROOM = {}
_REF = {}


def _set_cublas_config(value):
    """as in test_deform_conv_offset_groups_gpu.py: drop torch's cached cuBLAS workspaces around a change of
    CUBLAS_WORKSPACE_CONFIG (torch sizes a workspace when it allocates it but reads the variable when it binds it)"""
    if os.environ.get("CUBLAS_WORKSPACE_CONFIG") == value:
        return
    torch.cuda.synchronize()
    torch._C._cuda_clearCublasWorkspaces()
    if value is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = value


@pytest.fixture
def state():
    """restores the form switches, the TF32 flags and the deterministic state"""
    from devis_b200 import deform_conv
    old_fused, old_tc = deform_conv.set_fused(True), deform_conv.set_tensor_core(True)
    old_tf32 = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    old_det = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
               os.environ.get("CUBLAS_WORKSPACE_CONFIG"))
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    deform_conv.set_fused(old_fused)
    deform_conv.set_tensor_core(old_tc)
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old_tf32
    torch.use_deterministic_algorithms(old_det[0], warn_only=old_det[1])
    _set_cublas_config(old_det[2])


@pytest.fixture(scope="module", autouse=True)
def _report_headroom():
    yield
    if HEADROOM:
        print("\nlargest |got - ref| / (tau * S) per kernel family:")
        for fam in sorted(HEADROOM):
            print(f"  {fam:28s} {HEADROOM[fam]:.3e}")
        path = os.environ.get("DEVIS_DCN_HEADROOM_JSON")
        if path:
            with open(path, "w") as f:
                json.dump(HEADROOM, f, indent=1, sort_keys=True)


def _deterministic(on):
    _set_cublas_config(":4096:8" if on else None)
    torch.use_deterministic_algorithms(on)


def _recorder(monkeypatch):
    """C entry points the Python layer calls: _lib.load() returns a proxy that records the launching ones"""
    from devis_b200 import _lib
    real, calls = _lib.load(), []

    class Proxy:
        def __getattr__(self, name):
            fn = getattr(real, name)
            if name not in LAUNCHING:
                return fn
            return lambda *a: (calls.append(name), fn(*a))[1]

    monkeypatch.setattr(_lib, "load", lambda: Proxy())
    return calls


def _cuda(ops, dtype):
    return [None if t is None else t.to("cuda", dtype) for t in ops]


def run(case, ops):
    """the library on the case's operands (float64 CPU tensors, cast to the case's dtype): {'out', 'gx', ...}"""
    from devis_b200 import deform_conv
    x, off, wt, b, m, gout = _cuda(ops, getattr(torch, case.dtype))
    deform_conv.set_fused(case.form in ("fused", "auto"))
    deform_conv.set_tensor_core(case.form == "auto")
    leaves = [None if t is None else t.clone().requires_grad_(case.train) for t in (x, off, wt, b, m)]
    with torch.set_grad_enabled(case.train):
        if case.form == "igemm":
            # the forward's precision follows allow_tf32; the backward's cuBLAS GEMMs run in float32 either way here
            torch.backends.cuda.matmul.allow_tf32 = case.tf32
            try:
                out = deform_conv.IGemmDeformConv2dFunction.apply(*leaves, case.stride, case.pad, case.dil)
            finally:
                torch.backends.cuda.matmul.allow_tf32 = False
        else:
            out = deform_conv.deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], case.stride, case.pad, case.dil,
                                            leaves[4])
    res = {"out": out.detach()}
    if case.train:
        out.backward(gout)
        res.update({k: t.grad for k, t in zip(KEYS, leaves) if t is not None})
    return res


def _oracle(case, x, off, wt, b, m):
    from oracle.deform_conv_torch import deform_conv2d_torch
    geo = dict(stride=case.stride, padding=case.pad, dilation=case.dil)
    if case.og == 1:
        return deform_conv2d_torch(x, off, wt, b, mask=m, **geo)
    k, cg = case.k, case.cin // case.og
    return sum(deform_conv2d_torch(x[:, g * cg:(g + 1) * cg], off[:, 2 * g * k:2 * (g + 1) * k], wt[:, g * cg:(g + 1) * cg],
                                   b if g == 0 else None, mask=None if m is None else m[:, g * k:(g + 1) * k], **geo)
               for g in range(case.og))


def _oracle_run(case, vals, magnitude):
    """float64 oracle, forward (+ gradients), in batch slices; ``magnitude``: on |operands| (the bound S), no offset
    gradient"""
    if magnitude:
        vals = [t if t is None or i == 1 else t.abs() for i, t in enumerate(vals)]      # offsets unchanged
    x, off, wt, b, m, gout = vals
    wt = wt.clone().requires_grad_(case.train)
    b = None if b is None else b.clone().requires_grad_(case.train)
    per = max(1, int(REF_SLICE_ELEMS // (case.cin * case.k * case.ho * case.wo)))
    parts = {k: [] for k in ("out", "gx", "goff", "gm")}
    for n0 in range(0, case.n, per):
        sl = lambda t: None if t is None else t[n0:n0 + per].clone().requires_grad_(case.train)
        xs, os_, ms = sl(x), sl(off), sl(m)
        if magnitude:
            os_.requires_grad_(False)
        with torch.set_grad_enabled(case.train):
            out = _oracle(case, xs, os_, wt, b, ms)
        parts["out"].append(out.detach())
        if case.train:
            out.backward(gout[n0:n0 + per])
            parts["gx"].append(xs.grad)
            if not magnitude:
                parts["goff"].append(os_.grad)
            if ms is not None:
                parts["gm"].append(ms.grad)
    res = {k: torch.cat(v) for k, v in parts.items() if v}
    if case.train:
        res["gw"] = wt.grad
        if b is not None:
            res["gb"] = b.grad
    return res


def reference(case, ops):
    """(oracle, bound S) on the values the kernels read, cached per case"""
    if case.name not in _REF:
        vals = [None if t is None else t.to(getattr(torch, case.dtype)).to("cuda", torch.float64) for t in ops]
        ref = _oracle_run(case, vals, False)
        mag = _oracle_run(case, vals, True) if case.dtype == "float32" else None
        _REF[case.name] = {"ref": ref, "mag": mag}
    return _REF[case.name]["ref"], _REF[case.name]["mag"]


def fixed_point_slack(case, ops, route):
    """per grad_input element, the rounding the fixed-point form adds on top of float arithmetic: half a quantum
    2^(e - 36) per contribution (deform_conv.cuh "Deterministic form": 2^e > 2 * the bound of any contribution, from the
    maxima of grad_out, mask, weight and Cout for the fused kernel, of grad_cols and mask for col2im; one bit more here,
    the library takes its maxima over float32 values).  Contributions = live corners landing on the element."""
    x, off, wt, b, m, gout = [None if t is None else t.to(getattr(torch, case.dtype)).to("cuda", torch.float64)
                              for t in ops]
    n, og, k, h, w = case.n, case.og, case.k, case.h, case.w
    by, bx = [t.cuda() for t in dc._base(case)]
    o = off.view(n, og * k, 2, case.ho, case.wo)
    py, px = by + o[:, :, 0], bx + o[:, :, 1]
    inside = (py > -1) & (px > -1) & (py < h) & (px < w)
    y0, x0 = torch.floor(py), torch.floor(px)
    grp = (torch.arange(og * k, device="cuda") // k).view(1, -1, 1, 1)
    img = torch.arange(n, device="cuda").view(-1, 1, 1, 1)
    cnt = torch.zeros(n * og * h * w, dtype=torch.float64, device="cuda")
    for yy, xx in ((y0, x0), (y0, x0 + 1), (y0 + 1, x0), (y0 + 1, x0 + 1)):
        live = inside & (yy >= 0) & (yy <= h - 1) & (xx >= 0) & (xx <= w - 1)
        at = ((img * og + grp) * h + yy.clamp(0, h - 1).long()) * w + xx.clamp(0, w - 1).long()
        cnt.index_add_(0, at[live], torch.ones_like(at[live], dtype=torch.float64))
    cnt = cnt.view(n, og, 1, h, w).expand(n, og, case.cin // og, h, w).reshape(n, case.cin, h, w)
    m_max = float(m.abs().max()) if m is not None else 1.0
    if route == "fused":
        bound = float(gout.abs().max()) * m_max * float(wt.abs().max()) * case.cout
    else:
        gc = gout.permute(0, 2, 3, 1).reshape(-1, case.cout) @ wt.permute(0, 2, 3, 1).reshape(case.cout, -1)
        bound = float(gc.abs().max()) * m_max
    e = math.frexp(bound)[1] + 1
    return cnt * 2.0 ** (e + 1 - 36) / 2


def _family(case, key, pl):
    """kernel family that computed ``key`` of a case"""
    r = pl["route"]
    if key == "out":
        if r == "igemm":
            return "out:igemm_tf32" if case.tf32 else "out:igemm_3xtf32"
        if r == "fused":
            return "out:const_bank" if any(i[0] == "const_fwd" for i in pl["inst"]) else "out:lane_fwd"
        return "out:im2col+gemm"
    if key == "gw":
        return "gw:wgrad_kernel" if "devis_dcn_weight_grad" in pl["calls"] else "gw:im2col+gemm"
    if key == "gb":
        return "gb:sum"
    return f"{key}:{'lane_bwd' if r == 'fused' else 'col2im'}"


def check(case, got, ref, mag, pl, slack=None, tag=""):
    """``slack``: absolute per-element allowance of grad_input on top of tau * S (the fixed-point form's rounding)"""
    assert set(got) == set(ref), (sorted(got), sorted(ref))
    for key in got:
        a, r = got[key].double(), ref[key]
        assert a.shape == r.shape, key
        assert torch.isfinite(a).all(), key
        e = nmax(a.cpu().numpy(), r.cpu().numpy())
        if case.dtype == "float64":
            assert e <= 1e-12, (key, e)
            continue
        if key == "goff":
            assert e <= 1e-4, (key, e)
            continue
        if key == "out":
            bar = None if case.tf32 else (2e-5 if pl["route"] == "igemm" else 1e-5)
        else:
            bar = 1e-4
        if bar is not None:
            assert e <= bar, (key, e)
        tau = TAU_TF32 if key == "out" and case.tf32 else TAU_FP32
        bound = tau * mag[key]
        if key == "gx" and slack is not None:
            bound = bound + slack
        err = (a - r).abs()
        zero = bound == 0
        assert (a[zero] == 0).all(), f"{key}: nonzero where no term reaches"
        ratio = float((err[~zero] / bound[~zero]).max()) if (~zero).any() else 0.0
        fam = tag + _family(case, key, pl)
        HEADROOM[fam] = max(HEADROOM.get(fam, 0.0), ratio)
        assert ratio <= 1.0, (key, ratio)


def _counters():
    from devis_b200 import _lib
    return [_lib.kernel_launches(f) for f in (_lib.KERNEL_DCN, _lib.KERNEL_DCN_IGEMM, _lib.KERNEL_AUX)]


def _run_and_check_path(case, ops, monkeypatch, det):
    calls = _recorder(monkeypatch)
    before = _counters()
    got = run(case, ops)
    torch.cuda.synchronize()
    after = _counters()
    monkeypatch.undo()
    helper = torch.cuda.get_device_properties(0).multi_processor_count * 8
    pl = dc.plan(case, det=det, helper_blocks=helper)
    assert calls == pl["calls"]
    assert after[0] - before[0] == pl["dcn"], ("KERNEL_DCN", after[0] - before[0], pl["dcn"])
    assert after[1] - before[1] == pl["igemm"], ("KERNEL_DCN_IGEMM", after[1] - before[1], pl["igemm"])
    fixed_point = det and case.train and case.dtype == "float32"
    assert (after[2] > before[2]) == fixed_point, "fixed-point grad_input forms"
    return got, pl


@pytest.mark.parametrize("case", dc.CASES, ids=dc.CASE_IDS)
def test_kernels_match_float64_oracle(case, state, monkeypatch):
    ops = dc.operands(case, seed=1000 + dc.CASE_IDS.index(case.name))
    got, pl = _run_and_check_path(case, ops, monkeypatch, det=False)
    ref, mag = reference(case, ops)
    check(case, got, ref, mag, pl)


@pytest.mark.parametrize("case", F32_CASES, ids=[c.name for c in F32_CASES])
def test_deterministic_runs_bit_identical_and_within_bounds(case, state, monkeypatch):
    ops = dc.operands(case, seed=1000 + dc.CASE_IDS.index(case.name))
    _deterministic(True)
    a, pl = _run_and_check_path(case, ops, monkeypatch, det=True)
    b, _ = _run_and_check_path(case, ops, monkeypatch, det=True)
    if case.train:
        assert "devis_dcn_weight_grad" not in pl["calls"]
    for key in a:
        assert torch.equal(a[key], b[key]), key
    ref, mag = reference(case, ops)
    slack = fixed_point_slack(case, ops, pl["route"]) if case.train else None
    check(case, a, ref, mag, pl, slack, tag="det ")


# ---- out-of-map taps never read the input ---------------------------------------------------------------------------
POISON_CASES = ["i2c_f32_v4g4_asym", "i2c_f32_v1g8_nobias", "i2c_f64_v1g8_asym", "i2c_f32_og2", "lane_o4_g4",
                "lane_o8_g8", "lane_og2_o4_g4", "lane_fwd_infer_o4_g4", "wg_c16_o4_asym", "wg_c32_o8_asym",
                "cb_c32_ct16_asym", "cb_c72_ct32_2chunks", "cb_c40_o48", "ig3_o44_mb2_s2", "igt_o80_mb2_s3_asym",
                "ig3_o304_mb1_s2_2mma"]


@pytest.mark.parametrize("name", POISON_CASES)
def test_out_of_map_taps_do_not_read_the_input(name, state, monkeypatch):
    """pixels (0..1, 0..1) hold Inf / -Inf / NaN and are reached only as corners outside the map (a tap outside the map
    clamps its four dead corners onto exactly these pixels): every output and gradient equals, bit for bit, the run with
    those pixels finite.  grad_input and grad_weight through the deterministic forms (fixed-point scatter, GEMM on
    recomputed columns); the weight-gradient kernel's atomics are compared by normalised error."""
    case = dc.CASES[dc.CASE_IDS.index(name)]
    x, off, wt, b, m, gout = dc.operands(case, seed=77)
    bad, good, off = dc.poison(case, x, off)
    det = case.dtype == "float32"
    _deterministic(det)
    res = [run(case, (xx, off, wt, b, m, gout)) for xx in (bad, good)]
    for key in res[1]:
        assert torch.isfinite(res[0][key]).all(), key
        if key == "gx" and not det:          # float64: float atomics
            assert nmax(res[0][key].cpu().numpy(), res[1][key].cpu().numpy()) <= 1e-12
        else:
            assert torch.equal(res[0][key], res[1][key]), key
    if case.train and case.form == "fused" and case.dtype == "float32":
        _deterministic(False)
        calls = _recorder(monkeypatch)
        res = [run(case, (xx, off, wt, b, m, gout)) for xx in (bad, good)]
        monkeypatch.undo()
        if "devis_dcn_weight_grad" in calls:
            assert torch.isfinite(res[0]["gw"]).all()
            assert nmax(res[0]["gw"].cpu().numpy(), res[1]["gw"].cpu().numpy()) <= 1e-6
        for key in ("out", "goff", "gm", "gb"):
            if key in res[1]:
                assert torch.equal(res[0][key], res[1][key]), key
