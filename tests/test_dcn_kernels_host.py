"""Without a GPU: the case table of test_dcn_kernels_gpu.py reaches every kernel instantiation and launch shape of the
deformable convolution.  The host rules of dcn_cases.py are first pinned against the library's own host queries
(devis_dcn_fused_form_og, devis_dcn_packed_weight_elems_og, devis_dcn_igemm_supported, devis_dcn_wgrad_supported);
adding an instantiation to the library without a case for it fails here."""
import dcn_cases as dc

F32 = 0


def _lib():
    from devis_b200 import _lib
    return _lib.load()


def _shapes():
    """every (Cin, Cout, kh, kw, og) of the table plus a grid around the rules' boundaries"""
    seen = {(c.cin, c.cout, c.kh, c.kw, c.og) for c in dc.CASES}
    for cin in (4, 6, 8, 12, 16, 20, 24, 32, 33, 36, 40, 48, 64, 72, 136, 264):
        for cout in (1, 2, 3, 4, 8, 12, 16, 20, 32, 44, 48, 64, 80, 128, 264, 300, 304, 320, 512, 528):
            for og in (1, 2, 4):
                if cin % og == 0:
                    seen.add((cin, cout, 3, 3, og))
    return sorted(seen)


def test_rules_match_the_library_host_queries():
    lib = _lib()
    for cin, cout, kh, kw, og in _shapes():
        assert lib.devis_dcn_fused_form_og(cin, cout, kh, kw, og, F32) == dc.fused_form(cin, cout, kh, kw, og)
        p = dc.fused_plan(cin, cout, kh, kw, og)
        # the lane-group and constant-bank layouts differ in size: the sum pins both parts of the plan
        assert lib.devis_dcn_packed_weight_elems_og(cin, cout, kh, kw, og) == p["lanes_elems"] + p["const_elems"]
        if og == 1:
            assert bool(lib.devis_dcn_igemm_supported(cin, cout, kh, kw, F32)) == (dc.igemm_plan(cin, cout, kh, kw) is not None)
            assert bool(lib.devis_dcn_wgrad_supported(cin, cout, kh, kw, F32)) == dc.wgrad_supported(cin, cout, kh, kw)


def test_igemm_refuses_npad_beyond_304():
    lib = _lib()
    assert lib.devis_dcn_igemm_supported(64, 304, 3, 3, F32) == 1
    assert lib.devis_dcn_igemm_supported(64, 320, 3, 3, F32) == 0
    assert dc.igemm_plan(64, 320, 3, 3) is None


def test_case_table_reaches_every_instantiation():
    reached = set()
    for case in dc.CASES:
        reached |= dc.plan(case)["inst"]
        if case.dtype == "float32":
            reached |= dc.plan(case, det=True)["inst"]
    want = dc.all_instantiations()
    assert reached == want, (sorted(want - reached, key=str), sorted(reached - want, key=str))


def test_case_table_covers_geometry_and_batch_slicing():
    """unequal kh / kw, stride, padding and dilation in every form; more than 65535 batch items for every CUDA-core
    launcher (im2col / col2im, lane-group forward and backward, constant bank, weight-gradient kernel)"""
    asym = lambda c: c.kh != c.kw and c.stride[0] != c.stride[1] and c.pad[0] != c.pad[1] and c.dil[0] != c.dil[1]
    for route in ("im2col", "fused", "igemm"):
        assert any(asym(c) and dc.route(c) == route for c in dc.CASES), route
    assert any(asym(c) and ("const_fwd", c.cin, 16) in dc.plan(c)["inst"] for c in dc.CASES)
    assert any(asym(c) and any(i[0] == "wgrad" for i in dc.plan(c)["inst"]) for c in dc.CASES)
    big = set()
    for case in dc.CASES:
        if case.n > dc.MAX_GRID_Z:
            big |= {i[0] for i in dc.plan(case)["inst"]}
            big |= {i[0] for i in dc.plan(case, det=True)["inst"]}
    assert {"im2col", "col2im", "col2im_det", "lane_fwd", "lane_bwd", "lane_bwd_det", "const_fwd", "wgrad"} <= big
