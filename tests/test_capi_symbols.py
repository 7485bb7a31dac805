"""CPU-side checks of the drop-in boundary: libdevis_msda.so loads without a GPU, exports every function that
include/devis_msda.h declares, and the Python binding types exactly those.  No compute calls."""
import ctypes
import os
import re

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "devis_msda.h")
HEADERS = [HEADER, os.path.join(ROOT, "include", "devis_deform_conv.h")]


def _declared_functions():
    names = []
    for path in HEADERS:
        text = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
        names += re.findall(r"\b(devis_(?:t?msda|dcn)_\w+)\s*\(", text)
    return sorted(set(names))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from devis_b200 import _lib, build
    build.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_functions()
    assert len(declared) >= 13 and "devis_dcn_im2col" in declared
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/*.h but not exported"
    assert sorted(_lib.SIGNATURES) == declared, "python binding and header disagree on the function list"


def test_abi_version_and_error_strings_without_gpu():
    from devis_b200 import _lib
    lib = _lib.load()
    assert lib.devis_msda_abi_version() == _lib.ABI_VERSION
    header = open(HEADER).read()
    assert f"#define DEVIS_MSDA_ABI_VERSION {_lib.ABI_VERSION}" in header
    codes = {name: int(val) for name, val in re.findall(r"#define (DEVIS_MSDA_ERR_\w+) \((-\d+)\)", header)}
    assert len(codes) == 9
    for name, code in codes.items():
        msg = lib.devis_msda_error_string(code).decode()
        assert msg and "unknown" not in msg, name
    assert "unknown" in lib.devis_msda_error_string(-99).decode()
    for flag, val in (("DEVIS_MSDA_F32", _lib.F32), ("DEVIS_MSDA_F64", _lib.F64), ("DEVIS_MSDA_BF16", _lib.BF16)):
        assert re.search(rf"#define {flag} {val}\b", header)


def test_argument_validation_happens_before_any_cuda_call():
    """bad dtype / shape / batch-step are rejected on the host (no device needed)"""
    from devis_b200 import _lib
    lib = _lib.load()
    null = None
    # per-family launch counters before the calls below: GPU tests earlier in the same process may have launched kernels
    launched = [lib.devis_msda_kernel_launches(f) for f in range(64)]
    assert lib.devis_msda_forward(null, null, null, null, null, null, 1, 4, 2, 32, 1, 1, 1, 64, 7, null) == -3
    assert lib.devis_msda_forward(null, null, null, null, null, null, 1, 4, 0, 32, 1, 1, 1, 64, 0, null) == -2
    assert lib.devis_msda_forward(null, null, null, null, null, null, 3, 4, 2, 32, 1, 1, 1, 2, 0, null) == -4
    assert lib.devis_msda_forward(null, null, null, null, null, null, 1, 4, 2, 32, 1, 1, 1, 64, 0, null) == -1
    assert lib.devis_msda_backward(null, null, null, null, null, null, null, null, null, 1, 4, 2, 32, 1, 1, 1, 64, 0,
                                   0, null, 0, null) == -1
    # deformable-convolution entry points: dtype (bf16 is not served), shape, null pointers
    dims = (1, 4, 4, 8, 4, 4, 3, 3, 1, 1, 1, 1, 1, 1)
    assert lib.devis_dcn_im2col(null, null, null, null, *dims, 2, null) == -3
    assert lib.devis_dcn_im2col(null, null, null, null, *((1, 0) + dims[2:]), 0, null) == -2
    assert lib.devis_dcn_im2col(null, null, null, null, *dims, 0, null) == -1
    assert lib.devis_dcn_col2im(null, null, null, null, null, null, null, *dims, 0, null) == -1
    assert lib.devis_dcn_im2col(null, null, null, null, *((0,) + dims[1:]), 0, null) == 0
    # fused form: which layers it serves, packed-weight size, validation order
    assert lib.devis_dcn_fused_form(32, 16, 3, 3, 0) == 3 and lib.devis_dcn_fused_form(16, 1, 3, 3, 0) == 3
    assert lib.devis_dcn_fused_form(72, 32, 3, 3, 0) == 1 and lib.devis_dcn_fused_form(264, 128, 3, 3, 0) == 0
    assert lib.devis_dcn_fused_form(136, 64, 3, 3, 0) == 0 and lib.devis_dcn_fused_form(136, 8, 3, 3, 0) == 3
    assert lib.devis_dcn_fused_form(30, 16, 3, 3, 0) == 0 and lib.devis_dcn_fused_form(32, 16, 3, 3, 1) == 0
    assert lib.devis_dcn_packed_weight_elems(72, 32, 3, 3) == 9 * 72 * 32                       # constant layout only
    assert lib.devis_dcn_packed_weight_elems(32, 16, 3, 3) == 9 * 1 * 16 * 8 * 4 + 9 * 32 * 16   # both layouts
    assert lib.devis_dcn_packed_weight_elems(72, 5, 3, 3) == 0
    assert lib.devis_dcn_pack_weight(null, null, 72, 5, 3, 3, null) == -8
    assert lib.devis_dcn_pack_weight(null, null, 72, 32, 3, 3, null) == -1
    assert lib.devis_dcn_fused_forward(null, null, null, null, null, null, *dims, 16, null) == -1
    assert lib.devis_dcn_fused_forward(null, null, null, null, null, null, *dims, 5, null) == -8
    assert lib.devis_dcn_fused_backward(null, null, null, null, null, null, null, null, *dims, 16, null) == -1
    assert lib.devis_dcn_fused_forward(null, null, null, null, null, null, *((0,) + dims[1:]), 16, null) == 0
    # empty problems are fine with null pointers and launch nothing
    before = lib.devis_msda_launch_count()
    assert lib.devis_msda_forward(null, null, null, null, null, null, 0, 4, 2, 32, 1, 0, 1, 64, 0, null) == 0
    assert lib.devis_msda_launch_count() == before
    assert lib.devis_msda_set_tuning(99, 1) == -2 and lib.devis_msda_set_tuning(0, 0) == 0   # conftest enables the knobs
    # fused-prologue entry points: reference-point width and temporal reference mode are validated on the host
    fused = lambda ref_dim, tref, d=32: lib.devis_tmsda_fused_forward(
        *([null] * 15), 2, 8, 8, d, 1, 3, 4, 4, 1, ref_dim, tref, 0, null)
    assert fused(3, 0) == -2 and fused(2, 3) == -2 and fused(2, 0, 16) == -8 and fused(4, 2) == -1
    # per-family launch counters exist for every family the header names and none of the calls above launched anything
    header = open(HEADER).read()
    n_fam = int(re.search(r"#define DEVIS_MSDA_KERNEL_FAMILIES (\d+)", header).group(1))
    assert n_fam == 10 and [lib.devis_msda_kernel_launches(f) for f in range(64)] == launched
    assert all(v == 0 for v in launched[n_fam:])
    assert lib.devis_msda_kernel_launches(-1) == 0 and lib.devis_msda_kernel_launches(n_fam) == 0
    for name in ("TREF_LEVEL0", "TREF_OWN", "TREF_SAMPLED"):
        assert re.search(rf"#define DEVIS_TMSDA_{name} {getattr(_lib, name)}\b", header)
    for name in re.findall(r"#define DEVIS_MSDA_(KERNEL_[A-Z_]+) (\d+)", header):
        if name[0] != "KERNEL_FAMILIES":
            assert getattr(_lib, name[0]) == int(name[1]), name


def test_tuning_knobs_are_inert_in_a_product_process():
    """devis_msda_set_tuning only works when the process was started with DEVIS_MSDA_TUNING=1 (developer benchmarks,
    this test suite); a product process gets DEVIS_MSDA_ERR_UNSUPPORTED and keeps the built-in kernel selection"""
    import subprocess
    import sys
    code = ("import sys\nsys.path.insert(0, %r)\nfrom devis_b200 import _lib\n"
            "print('RC', _lib.load().devis_msda_set_tuning(0, 128))\n" % ROOT)
    env = {k: v for k, v in os.environ.items() if k != "DEVIS_MSDA_TUNING"}
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300).stdout
    assert "RC -8" in out, out
    out = subprocess.run([sys.executable, "-c", code], env=dict(env, DEVIS_MSDA_TUNING="1"), capture_output=True,
                         text=True, timeout=300).stdout
    assert "RC 0" in out, out


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "devis_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "/root/reference" not in src.replace("(/root/reference/", "("), f


def test_missing_library_fails_loudly():
    """no fallback: with the library absent every op raises (checked in a subprocess so this process keeps its library)"""
    import subprocess
    import sys
    code = (
        "import os, sys, torch\n"
        "sys.path.insert(0, %r)\n"
        "import devis_b200\n"
        "from devis_b200 import _lib\n"
        "try:\n"
        "    _lib.load()\n"
        "    print('LOADED')\n"
        "except _lib.MSDAError as e:\n"
        "    print('RAISED', 'no CPU or PyTorch fallback' in str(e))\n" % ROOT)
    env = dict(os.environ, DEVIS_MSDA_LIB="/nonexistent/libdevis_msda.so")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300).stdout
    assert "RAISED True" in out, out
