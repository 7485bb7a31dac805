"""CPU-side checks of the float16 value type (DEVIS_MSDA_F16): every attention entry point accepts the code and gets as
far as its pointer checks, the bf16-only grad_value accumulation flag is refused for it, the workspace sizes equal the
bf16 ones, the deformable-convolution entry points keep refusing it, and the reference's dispatch (the compiled-module
mirror) keeps refusing float16.  No device, no compute calls."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "devis_msda.h")
OK, ERR_NULL, ERR_BAD_DTYPE, ERR_UNSUPPORTED = 0, -1, -3, -8
null = None
# a non-null DEVICE address that is never dereferenced: the calls below return before any CUDA call
FAKE = ctypes.c_void_p(1 << 20)


@pytest.fixture(scope="module")
def lib():
    from devis_b200 import _lib
    return _lib.load()


def _host_tables(n_frames=2, t_window=1):
    shapes = np.array([[4, 6], [2, 3]], dtype=np.int64)
    lsi = np.array([0, 24], dtype=np.int64)
    frames = np.array([[1 - t] for t in range(n_frames)], dtype=np.int32)
    assert frames.shape == (n_frames, t_window)
    return shapes, lsi, frames


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_header_and_binding_define_f16(lib):
    from devis_b200 import _lib
    header = open(HEADER).read()
    assert _lib.F16 == 3 and re.search(r"#define DEVIS_MSDA_F16 3\b", header)
    assert _lib.ABI_VERSION == 5 and lib.devis_msda_abi_version() == 5


@pytest.mark.parametrize("dtype,want", [(3, ERR_NULL), (4, ERR_BAD_DTYPE)])
def test_f16_passes_dtype_validation_in_every_attention_entry_point(lib, dtype, want):
    """code 3 is accepted and the call stops at the null pointers; code 4 still is a bad dtype"""
    launched = lib.devis_msda_launch_count()
    # devis_msda_forward / backward: batch 1, 30 rows, 2 heads, 32 channels, 2 levels, 3 queries, 4 points
    dims = (1, 30, 2, 32, 2, 3, 4, 64)
    assert lib.devis_msda_forward(*([null] * 6), *dims, dtype, null) == want
    assert lib.devis_msda_backward(*([null] * 9), *dims, dtype, 0, null, 0, null) == want
    # whole-clip op: 2 frames, 30 rows, 2 heads, 32 channels, 2 levels, 3 queries, 4 + 4 points, window 1
    cdims = (2, 30, 2, 32, 2, 3, 4, 4, 1)
    assert lib.devis_tmsda_forward(*([null] * 10), *cdims, dtype, null) == want
    assert lib.devis_tmsda_backward(*([null] * 15), *cdims, dtype, 0, null, 0, null) == want
    # fused op (channels 32, points multiples of 4): ref_dim 2, TREF_LEVEL0
    fdims = cdims + (2, 0)
    assert lib.devis_tmsda_fused_forward(*([null] * 15), *fdims, dtype, null) == want
    assert lib.devis_tmsda_fused_backward(*([null] * 17), *fdims, dtype, 0, null, 0, null) == want
    assert lib.devis_msda_launch_count() == launched


def test_bf16_grad_value_flag_is_refused_for_f16(lib):
    """DEVIS_MSDA_FLAG_BF16_GRAD_VALUE: bf16 only -- fp16's range makes rounding every partial sum unsafe"""
    from devis_b200 import _lib
    flag, f16 = _lib.FLAG_BF16_GRAD_VALUE, _lib.F16
    launched = lib.devis_msda_launch_count()
    dims = (1, 30, 2, 32, 2, 3, 4, 64)
    assert lib.devis_msda_backward(*([FAKE] * 9), *dims, f16, flag, null, 0, null) == ERR_UNSUPPORTED
    shapes, lsi, frames = _host_tables()
    cdims = (2, 30, 2, 32, 2, 3, 4, 4, 1)
    dev = [FAKE] * 10          # loc_curr .. grad_aw_temporal; query_order stays NULL
    assert lib.devis_tmsda_backward(FAKE, _p(shapes), _p(lsi), _p(frames), *dev, null, *cdims, f16, flag, null, 0,
                                    null) == ERR_UNSUPPORTED
    dev = [FAKE] * 11          # ref .. grad_logit_temporal; grad_ref and query_order stay NULL
    assert lib.devis_tmsda_fused_backward(FAKE, _p(shapes), _p(lsi), _p(frames), *dev, null, null, *cdims, 2, 0, f16,
                                          flag, null, 0, null) == ERR_UNSUPPORTED
    assert lib.devis_msda_launch_count() == launched


@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_workspace_bytes_for_f16_equal_bf16(lib, flags):
    from devis_b200 import _lib
    for t, s, m, d in ((1, 30, 2, 32), (6, 4820, 8, 32), (3, 100, 4, 30)):
        per = [lib.devis_msda_backward_workspace_bytes(t, s, m, d, 4, 7, 4, code, flags) for code in (_lib.BF16, _lib.F16)]
        clip = [lib.devis_tmsda_backward_workspace_bytes(t, s, m, d, 4, 7, 4, 4, 2, code, flags)
                for code in (_lib.BF16, _lib.F16)]
        assert per[0] == per[1] and clip[0] == clip[1]
        if flags == _lib.FLAG_DETERMINISTIC:
            assert per[1] == t * s * m * d * 8 + 16 and clip[1] == per[1]
    # the fused op's workspace does not depend on the dtype at all (no dtype argument)
    assert lib.devis_tmsda_fused_backward_workspace_bytes(6, 4820, 8, 32, flags) == \
        (6 * 4820 * 8 * 32 * 8 + 16 if flags == _lib.FLAG_DETERMINISTIC else 0)


def test_deformable_convolution_keeps_refusing_f16(lib):
    dims = (1, 4, 4, 8, 4, 4, 3, 3, 1, 1, 1, 1, 1, 1)
    for code in (2, 3):
        assert lib.devis_dcn_im2col(null, null, null, null, *dims, code, null) == ERR_BAD_DTYPE
        assert lib.devis_dcn_col2im(null, null, null, null, null, null, null, *dims, code, null) == ERR_BAD_DTYPE
        assert lib.devis_dcn_im2col_og(null, null, null, null, *dims, 1, code, null) == ERR_BAD_DTYPE
        assert lib.devis_dcn_col2im_og(*([null] * 7), *dims, 1, code, 0, null, 0, null) == ERR_BAD_DTYPE
        assert lib.devis_dcn_col2im_ex(*([null] * 7), *dims, code, 0, null, 0, null) == ERR_BAD_DTYPE
    assert lib.devis_dcn_im2col(null, null, null, null, *dims, 0, null) == ERR_NULL


def test_reference_dispatch_keeps_refusing_float16():
    """the compiled-module mirror (and so MSDeformAttnFunction / MSDeformAttn) keeps the reference's dtype dispatch;
    only the temporal ops take float16"""
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    from devis_b200.functions import temporal_func
    assert torch.float16 not in MSDA._DTYPES
    with pytest.raises(RuntimeError, match="not implemented for"):
        MSDA._dtype_code(torch.empty(1, dtype=torch.float16))
    assert temporal_func._DTYPES[torch.float16] == 3
    # supported() is a host-side decision: a CPU value is never supported, whatever its dtype
    v = torch.empty(1, 4, 8, 32, dtype=torch.float16)
    assert not temporal_func.TemporalMSDeformAttnFusedFunction.supported(v, torch.empty(1, 2, 1, 2))
