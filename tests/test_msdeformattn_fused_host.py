"""CPU-side checks of MSDeformAttn's fused path: argument validation of the padding-mask entry points
(devis_tmsda_fused_forward_ex / _backward_ex) before any CUDA call, and the module's decision of which path to take.
No device, no compute calls."""
import ctypes

import pytest
import torch

ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_UNSUPPORTED = -1, -2, -3, -8


@pytest.fixture(scope="module")
def lib():
    from devis_b200 import _lib, build
    build.build()
    return _lib.load()


def _fwd(lib, *, mask=None, value=None, ref=None, off=None, logit=None, out=None, n=2, d=32, pc=4, ref_dim=2, tref=0,
         dtype=0, shapes=None, lsi=None):
    return lib.devis_tmsda_fused_forward_ex(value, shapes, lsi, None, ref, off, logit, None, None, out,
                                            None, None, None, None, None, mask, n, 8, 8, d, 1, 3, pc, 0, 0, ref_dim,
                                            tref, dtype, None)


def _bwd(lib, *, mask=None, n=2, d=32, dtype=0, flags=0, shapes=None, lsi=None):
    return lib.devis_tmsda_fused_backward_ex(None, shapes, lsi, None, None, None, None, None, None, None, None, None,
                                             None, None, None, None, None, mask, n, 8, 8, d, 1, 3, 4, 0, 0, 2, 0, dtype,
                                             flags, None, 0, None)


def test_ex_entries_validate_before_any_cuda_call(lib):
    launched = [lib.devis_msda_kernel_launches(f) for f in range(16)]
    fake = ctypes.c_void_p(0x1000)          # never dereferenced: every call below stops in validation
    shapes = (ctypes.c_int64 * 2)(2, 4)
    lsi = (ctypes.c_int64 * 1)(0)
    host = dict(shapes=ctypes.cast(shapes, ctypes.c_void_p), lsi=ctypes.cast(lsi, ctypes.c_void_p))
    for mask in (None, fake):
        assert _fwd(lib, mask=mask, dtype=7, **host) == ERR_DTYPE
        assert _fwd(lib, mask=mask, ref_dim=3, **host) == ERR_SHAPE
        assert _fwd(lib, mask=mask, tref=3, **host) == ERR_SHAPE
        assert _fwd(lib, mask=mask, d=16, **host) == ERR_UNSUPPORTED
        assert _fwd(lib, mask=mask, pc=3, **host) == ERR_UNSUPPORTED
        assert _fwd(lib, mask=mask, dtype=1, **host) == ERR_UNSUPPORTED      # fp64 has no fused kernel
        assert _fwd(lib, mask=mask) == ERR_NULL                             # host level tables missing
        assert _fwd(lib, mask=mask, **host) == ERR_NULL                     # a mask does not stand in for value
        assert _fwd(lib, mask=mask, value=fake, ref=fake, off=fake, logit=fake, **host) == ERR_NULL   # no output
        assert _bwd(lib, mask=mask, dtype=7, **host) == ERR_DTYPE
        assert _bwd(lib, mask=mask, d=16, **host) == ERR_UNSUPPORTED
        assert _bwd(lib, mask=mask, **host) == ERR_NULL
        # empty problems are fine with null tensors, mask or not, and launch nothing
        assert _fwd(lib, mask=mask, n=0, **host) == 0
    assert [lib.devis_msda_kernel_launches(f) for f in range(16)] == launched


def test_ex_entries_agree_with_the_plain_entries_on_errors(lib):
    """the plain entries are the _ex entries with padding_mask = NULL"""
    shapes = (ctypes.c_int64 * 2)(2, 4)
    lsi = (ctypes.c_int64 * 1)(0)
    for dtype, d, ref_dim in ((7, 32, 2), (0, 16, 2), (0, 32, 3), (1, 32, 2), (0, 32, 2)):
        plain = lib.devis_tmsda_fused_forward(None, shapes, lsi, None, None, None, None, None, None, None, None, None,
                                              None, None, None, 2, 8, 8, d, 1, 3, 4, 0, 0, ref_dim, 0, dtype, None)
        ex = lib.devis_tmsda_fused_forward_ex(None, shapes, lsi, None, None, None, None, None, None, None, None, None,
                                              None, None, None, None, 2, 8, 8, d, 1, 3, 4, 0, 0, ref_dim, 0, dtype,
                                              None)
        assert plain == ex != 0


def _decide(monkeypatch, dtype, fuse=True, d_model=256, n_points=4):
    """MSDeformAttn._fused_path on a CPU tensor of `dtype`, with the device-side capability check standing in as
    `supported` (the kernels' own shape rules) -- this is the module's part of the decision"""
    from devis_b200.functions import TemporalMSDeformAttnFusedFunction as Fused
    from devis_b200.modules import MSDeformAttn
    monkeypatch.setattr(Fused, "supported", staticmethod(
        lambda value, ref, pc=4, pt=4: value.shape[-1] == 32 and pc % 4 == 0 and pt % 4 == 0))
    mod = MSDeformAttn(d_model, 4, 8, n_points)
    mod.fuse_prologue = fuse
    value = torch.zeros(2, 10, 8, d_model // 8, dtype=dtype)
    return mod._fused_path(value, torch.zeros(2, 5, 4, 2))


def test_module_decision(monkeypatch):
    assert _decide(monkeypatch, torch.float32) and _decide(monkeypatch, torch.bfloat16)
    assert not _decide(monkeypatch, torch.float16)          # MSDeformAttn keeps the reference's dtype dispatch
    assert not _decide(monkeypatch, torch.float64)
    assert not _decide(monkeypatch, torch.float32, fuse=False)
    assert not _decide(monkeypatch, torch.float32, d_model=64)      # D = 8
    assert not _decide(monkeypatch, torch.float32, n_points=3)


def test_module_float16_still_refused_by_the_op():
    from devis_b200 import MultiScaleDeformableAttention as MSDA
    with pytest.raises(RuntimeError, match="not implemented for"):
        MSDA._dtype_code(torch.empty(1, dtype=torch.float16))


def test_supported_is_false_off_device():
    from devis_b200.functions import TemporalMSDeformAttnFusedFunction as Fused
    assert not Fused.supported(torch.zeros(2, 10, 8, 32), torch.zeros(2, 5, 4, 2))
