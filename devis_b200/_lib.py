"""ctypes binding of the C-ABI library (include/devis_msda.h).

There is NO fallback: if libdevis_msda.so is missing or does not export the ABI this package was
written against, importing the ops raises.  (The reference behaves the same way: its Python op
imports the compiled module unconditionally, functions/ms_deform_attn_func.py:18, and its CPU
entry points raise "Not implemented on the CPU", src/cpu/ms_deform_attn_cpu.cpp:26,39.)
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEVIS_MSDA_LIB selects another build of the same ABI (kernel A/B experiments); the default is the in-tree library
LIB_PATH = os.environ.get("DEVIS_MSDA_LIB") or os.path.join(_HERE, "libdevis_msda.so")

ABI_VERSION = 5
F32, F64, BF16, F16 = 0, 1, 2, 3
FLAG_DETERMINISTIC, FLAG_NO_GRAD_VALUE, FLAG_BF16_GRAD_VALUE = 1, 2, 4
# temporal_ref_mode of the fused-prologue entry points (DEVIS_TMSDA_TREF_*)
TREF_LEVEL0, TREF_OWN, TREF_SAMPLED = 0, 1, 2
# kernel families of devis_msda_kernel_launches (DEVIS_MSDA_KERNEL_*)
KERNEL_FWD_GROUPED, KERNEL_FWD_GENERIC, KERNEL_BWD_GROUPED, KERNEL_BWD_GENERIC = 0, 1, 2, 3
KERNEL_FUSED_FWD, KERNEL_FUSED_BWD, KERNEL_BWD_SORTED, KERNEL_AUX, KERNEL_DCN, KERNEL_DCN_IGEMM = 4, 5, 6, 7, 8, 9
DCN_PRECISION_3XTF32, DCN_PRECISION_TF32 = 0, 1

_vp, _i, _u, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/devis_msda.h declaration by declaration
SIGNATURES = {
    "devis_msda_abi_version": (_i, []),
    "devis_msda_error_string": (ctypes.c_char_p, [_i]),
    "devis_msda_last_cuda_error": (_i, []),
    "devis_msda_launch_count": (ctypes.c_uint64, []),
    "devis_msda_kernel_launches": (ctypes.c_uint64, [_i]),
    "devis_msda_set_tuning": (_i, [_i, _i]),
    "devis_msda_forward": (_i, [_vp] * 6 + [_i] * 9 + [_vp]),
    "devis_msda_backward_workspace_bytes": (_sz, [_i] * 8 + [_u]),
    "devis_msda_backward": (_i, [_vp] * 9 + [_i] * 9 + [_u, _vp, _sz, _vp]),
    "devis_tmsda_forward": (_i, [_vp] * 10 + [_i] * 10 + [_vp]),
    "devis_tmsda_backward_workspace_bytes": (_sz, [_i] * 10 + [_u]),
    "devis_tmsda_backward": (_i, [_vp] * 15 + [_i] * 10 + [_u, _vp, _sz, _vp]),
    "devis_tmsda_fused_forward": (_i, [_vp] * 15 + [_i] * 12 + [_vp]),
    "devis_tmsda_fused_backward_workspace_bytes": (_sz, [_i] * 4 + [_u]),
    "devis_tmsda_fused_backward": (_i, [_vp] * 17 + [_i] * 12 + [_u, _vp, _sz, _vp]),
    # include/devis_deform_conv.h
    "devis_dcn_im2col": (_i, [_vp] * 4 + [_i] * 15 + [_vp]),
    "devis_dcn_im2col_og": (_i, [_vp] * 4 + [_i] * 16 + [_vp]),
    "devis_dcn_col2im": (_i, [_vp] * 7 + [_i] * 15 + [_vp]),
    "devis_dcn_backward_workspace_bytes": (_sz, [_i] * 4 + [_u]),
    "devis_dcn_col2im_ex": (_i, [_vp] * 7 + [_i] * 15 + [_u, _vp, _sz, _vp]),
    "devis_dcn_col2im_og": (_i, [_vp] * 7 + [_i] * 16 + [_u, _vp, _sz, _vp]),
    "devis_dcn_fused_form": (_i, [_i] * 5),
    "devis_dcn_fused_form_og": (_i, [_i] * 6),
    "devis_dcn_packed_weight_elems": (_sz, [_i] * 4),
    "devis_dcn_packed_weight_elems_og": (_sz, [_i] * 5),
    "devis_dcn_pack_weight": (_i, [_vp] * 2 + [_i] * 4 + [_vp]),
    "devis_dcn_pack_weight_og": (_i, [_vp] * 2 + [_i] * 5 + [_vp]),
    "devis_dcn_fused_forward": (_i, [_vp] * 6 + [_i] * 15 + [_vp]),
    "devis_dcn_fused_forward_og": (_i, [_vp] * 6 + [_i] * 16 + [_vp]),
    "devis_dcn_fused_backward": (_i, [_vp] * 8 + [_i] * 15 + [_vp]),
    "devis_dcn_fused_backward_ex": (_i, [_vp] * 8 + [_i] * 15 + [_u, _vp, _sz, _vp]),
    "devis_dcn_fused_backward_og": (_i, [_vp] * 8 + [_i] * 16 + [_u, _vp, _sz, _vp]),
    "devis_dcn_wgrad_supported": (_i, [_i] * 5),
    "devis_dcn_weight_grad": (_i, [_vp] * 5 + [_i] * 15 + [_vp]),
    "devis_dcn_igemm_supported": (_i, [_i] * 5),
    "devis_dcn_igemm_packed_weight_elems": (_sz, [_i] * 4),
    "devis_dcn_igemm_pack_weight": (_i, [_vp] * 2 + [_i] * 4 + [_vp]),
    "devis_dcn_igemm_forward": (_i, [_vp] * 6 + [_i] * 16 + [_vp]),
}

_lib = None


class MSDAError(RuntimeError):
    pass


def load():
    """Load (once) and type the library.  Raises if it is absent -- build it with
    ``python -m devis_b200.build`` (nvcc, sm_100a)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MSDAError(f"{LIB_PATH} not found: the CUDA library is not built "
                        "(python -m devis_b200.build); there is no CPU or PyTorch fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    got = lib.devis_msda_abi_version()
    if got != ABI_VERSION:
        raise MSDAError(f"libdevis_msda.so has ABI {got}, this package needs {ABI_VERSION}")
    _lib = lib
    return lib


def check(code):
    if code != 0:
        lib = load()
        msg = lib.devis_msda_error_string(code).decode()
        if code == -7:
            msg += f" [cudaError {lib.devis_msda_last_cuda_error()}]"
        raise MSDAError(f"devis_msda: {msg} (code {code})")


def launch_count():
    return int(load().devis_msda_launch_count())


def kernel_launches(family):
    """launches of one kernel family (KERNEL_*) so far: which kernel served a call, not just that one ran"""
    return int(load().devis_msda_kernel_launches(int(family)))


def set_tuning(key, value):
    """developer knob of the benchmarks; the library refuses it unless the process runs with DEVIS_MSDA_TUNING=1"""
    check(load().devis_msda_set_tuning(int(key), int(value)))
