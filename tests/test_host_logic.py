"""CPU tests of the host-side mirror: frame tables and temporal level tables against what the reference's
DeVISTransformerEncoder/Decoder build (golden book_* fixtures), query tile orders, module parameter layout and
initial values, the projection stage against the oracle port, and the no-CPU-fallback contract."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from devis_b200 import clip_geometry, synthetic
from devis_b200.modules import MSDeformAttn, TemporalMSDeformAttnDecoder, TemporalMSDeformAttnEncoder


def test_frame_tables_match_reference_transformer_bookkeeping():
    g = load_golden("book_enc_all")
    t = g["temporal_offsets"].shape[0]
    assert clip_geometry.all_frames_table(t) == (g["temporal_offsets"] + np.arange(t)[:, None]).tolist()
    g = load_golden("book_enc_window")
    t = g["temporal_offsets"].shape[0]
    assert clip_geometry.window_table(t, int(g["t_window"])) == (g["temporal_offsets"] + np.arange(t)[:, None]).tolist()
    g = load_golden("book_dec_2d")
    assert clip_geometry.all_frames_table(3) == (g["temporal_offsets"] + np.arange(3)[:, None]).tolist()


def test_geometry_from_reference_arguments():
    g = load_golden("book_enc_window")
    offs = [torch.from_numpy(r) for r in g["temporal_offsets"]]
    geom = clip_geometry.from_reference_args(4, (torch.from_numpy(g["shapes"]), torch.from_numpy(g["tshapes"])),
                                             (torch.from_numpy(g["lsi"]), torch.from_numpy(g["tlsi"])), offs)
    assert geom.shapes == [tuple(r) for r in g["shapes"].tolist()]
    assert geom.level_start_index == g["lsi"].tolist()
    assert geom.spatial_size == int(g["shapes"].prod(1).sum()) and geom.t_window == 2
    assert geom.frame_table[0] == [1, 1]                 # reflection lists a frame twice (devis_transformer.py:102-112)
    # the temporal tables the reference rebuilds per forward are implied by (shapes, t_window)
    assert np.array_equal(np.tile(g["shapes"], (geom.t_window, 1)), g["tshapes"])
    again = clip_geometry.from_reference_args(4, (torch.from_numpy(g["shapes"]), None), (torch.from_numpy(g["lsi"]), None), offs)
    assert again is geom                                  # memoised
    with pytest.raises(ValueError):
        clip_geometry.ClipGeometry([(2, 2)], 2, [[5], [0]])


def test_tile_order_is_a_permutation_that_keeps_levels_apart():
    geom = clip_geometry.ClipGeometry(synthetic.DEVIS_SHAPES, 6, clip_geometry.all_frames_table(6))
    assert geom.spatial_size == 4820 and geom.level_start_index == [0, 3600, 4520, 4760]
    for th, tw in ((8, 8), (4, 8), (16, 16)):
        order = geom.tile_order("cpu", th, tw).numpy()
        assert np.array_equal(np.sort(order), np.arange(4820))
        assert order[:3600].max() < 3600 and order[3600:4520].min() >= 3600
    first = geom.tile_order("cpu", 8, 8).numpy()[:64]
    ys, xs = first // 80, first % 80
    assert ys.max() == 7 and xs.max() == 7               # first 64 queries are the top-left 8x8 pixel tile of level 0


def test_modules_have_reference_parameter_names_shapes_and_initial_values():
    for cls, fixture, kw in ((MSDeformAttn, "mod_msda_2d", dict(d_model=32, n_levels=2, n_heads=4, n_points=3)),
                             (TemporalMSDeformAttnEncoder, "mod_tenc_all",
                              dict(n_frames=3, d_model=32, n_levels=2, t_window=2, n_heads=4, n_curr_points=2, n_temporal_points=2)),
                             (TemporalMSDeformAttnDecoder, "mod_tdec_2d_ia",
                              dict(n_frames=3, d_model=32, n_levels=2, t_window=2, n_heads=4, n_curr_points=2, n_temporal_points=2))):
        g = load_golden(fixture)
        mod = cls(**kw)
        ref = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
        assert set(mod.state_dict()) == set(ref)
        for k, v in mod.state_dict().items():
            assert tuple(v.shape) == ref[k].shape, k
    # initial pattern (ms_deform_attn.py:184-221): zero offset weights, head rays (i+1) steps long, zero logits
    enc = TemporalMSDeformAttnEncoder(n_frames=6, d_model=256, n_levels=4, t_window=5, n_heads=8, n_curr_points=4,
                                      n_temporal_points=4)
    assert not enc.sampling_offsets.weight.any() and not enc.temporal_sampling_offsets.weight.any()
    assert not enc.attention_weights.bias.any() and not enc.temporal_attention_weights.weight.any()
    b = enc.sampling_offsets.bias.view(8, 4, 4, 2)
    assert torch.allclose(b[0, :, :, 0], torch.arange(1., 5.).expand(4, 4)) and not b[0, :, :, 1].abs().max() > 1e-6
    assert torch.allclose(b[2, 1, 3], torch.tensor([0., 4.]), atol=1e-6)
    bt = enc.temporal_sampling_offsets.bias.view(8, 20, 4, 2)
    assert torch.allclose(bt[:, 0], b[:, 0]) and torch.allclose(bt[:, 19], b[:, 0])
    assert enc.im2col_step == 64 and MSDeformAttn().im2col_step == 64
    with pytest.raises(ValueError):
        MSDeformAttn(d_model=30, n_heads=4)


def test_projection_stage_matches_oracle_port():
    """_compute_deformable_attention is pure PyTorch (cuBLAS/ATen on GPU): check it on CPU against the oracle port,
    which is pinned to the reference module by tests/test_oracle_golden.py"""
    from oracle import temporal_torch
    g = load_golden("mod_tenc_all")
    t_frames, c, nl, t_window, heads, pc, pt = [int(x) for x in g["cfg"]]
    mod = TemporalMSDeformAttnEncoder(t_frames, c, nl, t_window, heads, pc, pt).double()
    sd = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}
    mod.load_state_dict(sd)
    q, x = torch.from_numpy(g["query"]), torch.from_numpy(g["inp"])
    got = mod._compute_deformable_attention(q, x)
    want = temporal_torch.temporal_projections(sd, q, x, heads, nl, t_window, pc, pt)
    for a, b in zip(got, want):
        assert a.shape == b.shape and torch.allclose(a, b, rtol=0, atol=1e-13)


def test_no_cpu_fallback():
    from devis_b200 import MSDeformAttnFunction, clip_geometry as cg, temporal_ms_deform_attn
    g = load_golden("op_d32")
    args = [torch.from_numpy(g[k]) for k in ("value", "shapes", "lsi", "loc", "aw")]
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        MSDeformAttnFunction.apply(*args, 64)
    clip = synthetic.make_clip(n_frames=2, shapes=((4, 4),), heads=2, channels=32, queries=3, device="cpu")
    geom = cg.ClipGeometry(((4, 4),), 2, clip["frame_table"])
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        temporal_ms_deform_attn(clip["value"], clip["loc_curr"], clip["aw_curr"], clip["loc_temporal"],
                                clip["aw_temporal"], geom)


def test_synthetic_workload_is_boundary_safe_and_sized_like_the_survey():
    clip = synthetic.make_clip(n_frames=2, shapes=((9, 16), (5, 8)), heads=2, channels=4, device="cpu", seed=3)
    for key, sizes in (("loc_curr", [(16, 9), (8, 5)]), ("loc_temporal", [(16, 9), (8, 5)])):
        loc = clip[key]
        for lvl in range(loc.shape[3]):
            w, h = sizes[lvl % 2]
            pix = loc[:, :, :, lvl] * torch.tensor([w, h]) - 0.5
            frac = pix - torch.floor(pix)
            assert frac.min() > 0.015 and frac.max() < 0.985
    fwd, bwd = synthetic.algorithmic_bytes(6, 4820, 8, 32, 4820, 96)
    assert (fwd, bwd) == (325754880, 621895680)          # SURVEY.md section 8(d): 325.75 MB / 621.90 MB


def test_host_copies_are_memoised_per_tensor_object_not_per_address():
    """a tensor that re-uses a freed tensor's storage address with other values must not hit a stale cache"""
    a = torch.tensor([[4, 6], [2, 3]])
    lsi_a = torch.tensor([0, 24])
    offs = [torch.tensor([1]), torch.tensor([-1])]
    g1 = clip_geometry.from_reference_args(2, (a, None), (lsi_a, None), offs)
    assert g1.shapes == [(4, 6), (2, 3)]
    assert clip_geometry.from_reference_args(2, (a, None), (lsi_a, None), offs) is g1
    a[0, 0] = 5                                            # in-place edit bumps the version -> re-read
    lsi_b = torch.tensor([0, 30])
    g2 = clip_geometry.from_reference_args(2, (a, None), (lsi_b, None), offs)
    assert g2.shapes == [(5, 6), (2, 3)] and g2 is not g1
    b = torch.tensor([[4, 6], [2, 3]])                     # new object, same values as the first call -> same geometry by value
    assert clip_geometry.from_reference_args(2, (b, None), (lsi_a, None), [torch.tensor([1]), torch.tensor([-1])]) is g1
    offs2 = [offs[0], torch.tensor([-1])]                  # same first tensor, different list -> table recomputed, equal value
    assert clip_geometry.from_reference_args(2, (b, None), (lsi_a, None), offs2) is g1


def _trunk_from_fixture(g, dtype=torch.float64):
    from devis_b200 import DeVISTransformer
    c, t_frames, heads, n_enc, n_dec, ffn, nl, connect_all, window, pc, pt, _ = [int(x) for x in g["cfg"]]
    tr = DeVISTransformer(d_model=c, num_frames=t_frames, nhead=heads, num_encoder_layers=n_enc,
                          num_decoder_layers=n_dec, dim_feedforward=ffn, dropout=0.0, num_feature_levels=nl,
                          enc_connect_all_embeddings=bool(connect_all), enc_temporal_window=window,
                          enc_n_curr_points=pc, enc_n_temporal_points=pt, dec_n_curr_points=pc, dec_n_temporal_points=pt)
    tr.decoder.bbox_embed = torch.nn.ModuleList(
        [torch.nn.Sequential(torch.nn.Linear(c, c), torch.nn.ReLU(), torch.nn.Linear(c, 4)) for _ in range(n_dec)])
    return tr.to(dtype)


@pytest.mark.parametrize("tag", ["all", "window"])
def test_transformer_mirror_has_reference_state_dict_and_bookkeeping(tag):
    """parameter names / shapes of DeVISTransformer are the reference's (checkpoints load), and the host-side parts of
    its forward -- prepare_data, valid ratios, encoder reference points, frame offsets -- reproduce the reference's"""
    g = load_golden(f"trunk_{tag}")
    tr = _trunk_from_fixture(g)
    want = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    have = tr.state_dict()
    assert set(want) == set(have)
    assert all(tuple(have[k].shape) == want[k].shape for k in want)
    tr.load_state_dict({k: torch.from_numpy(v) for k, v in want.items()})

    nl = int(g["cfg"][6])
    srcs = [torch.from_numpy(g[f"src{i}"]) for i in range(nl)]
    masks = [torch.from_numpy(g[f"mask{i}"]) for i in range(nl)]
    pos = [torch.from_numpy(g[f"pos{i}"]) for i in range(nl)]
    src, mask, pos_flat, shapes, lsi, valid = tr.prepare_data(srcs, masks, pos)
    assert np.array_equal(shapes.numpy(), g["shapes"]) and np.array_equal(lsi.numpy(), g["lsi"])
    assert np.abs(valid.numpy() - g["valid_ratios"]).max() < 1e-12
    assert clip_geometry.host_list(shapes) == g["shapes"].tolist()          # attached host copy, no device read
    assert src.shape == (srcs[0].shape[0], int(g["shapes"].prod(1).sum()), srcs[0].shape[1]) and mask.shape == src.shape[:2]
    level0 = pos[0].flatten(2).transpose(1, 2) + tr.level_embed[0].view(1, 1, -1)
    assert torch.equal(pos_flat[:, :level0.shape[1]], level0)

    # encoder reference points and frame offsets against the reference encoder's (book_enc_* fixtures)
    book = load_golden(f"book_enc_{tag}")
    ref = tr.encoder.get_reference_points(torch.from_numpy(book["shapes"]), torch.from_numpy(book["valid_ratios"]), "cpu")
    assert np.abs(ref.numpy() - book["ref"]).max() < 1e-6                    # linspace is float32 in the reference too
    tr.encoder.t_window = int(book["t_window"])
    assert tr.encoder.frame_offsets(book["temporal_offsets"].shape[0]) == book["temporal_offsets"].tolist()


def test_decoder_mirror_scales_reference_points_like_the_reference():
    """2-d points and 4-d boxes are scaled by FRAME 0's valid ratios for every frame (devis_transformer.py:161-166)"""
    from devis_b200 import DeVISTransformerDecoder
    for tag in ("2d", "4d"):
        g = load_golden(f"book_dec_{tag}")
        seen = {}

        class Capture(torch.nn.Module):
            def forward(self, output, query_pos, ref_in, src, shapes_pair, lsi_pair, temporal_offsets):
                seen.update(ref_in=ref_in, tshapes=shapes_pair[1], tlsi=lsi_pair[1], offsets=temporal_offsets)
                return output

        dec = DeVISTransformerDecoder(Capture(), 1)
        ref = torch.from_numpy(g["ref"])
        t_frames = g["valid_ratios"].shape[0]
        s = int(g["shapes"].prod(1).sum())
        hs, refs = dec(torch.zeros(1, ref.shape[1], 8, dtype=torch.float64), ref, torch.zeros(t_frames, s, 8, dtype=torch.float64),
                       torch.from_numpy(g["shapes"]), torch.from_numpy(g["lsi"]), torch.from_numpy(g["valid_ratios"]))
        assert np.abs(seen["ref_in"].numpy() - g["ref_in"]).max() < 1e-15
        assert np.array_equal(seen["tshapes"].numpy(), g["tshapes"]) and np.array_equal(seen["tlsi"].numpy(), g["tlsi"])
        assert seen["offsets"] == g["temporal_offsets"].tolist()
        assert hs.shape[0] == 1 and torch.equal(refs[0], ref)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): one JSON line with the contract's keys,
    same metric / unit / workload as our arm, a cpu_baseline describing the run and zero-copy e2e."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "temporal_msda_fwd_bwd_layer_clips_per_sec"
    assert line["unit"] == "layer-clips/s" and line["higher_is_better"] is True and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert abs(line["value"] - 1e3 / line["ms_per_step"]) < 1e-6 * line["value"]
    assert "workload" in line["config"] and "model" not in line["config"]


def test_bench_dump_outputs_writes_a_fixed_bounded_sample(tmp_path):
    """`bench.py --dump-outputs`: small arrays whole (float64 kept, bf16 widened), large ones as the same seeded sample of
    flat indices in every run, the six arrays of the bench step under 64 MB in all"""
    import bench
    n = bench.DUMP_MAX_ELEMS + 1000
    big = torch.arange(n, dtype=torch.float32)
    arrays = {"big": big, "f64": torch.randn(3, 4, dtype=torch.float64), "bf16": torch.randn(5).bfloat16()}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), {"big": big * 2, **{k: v for k, v in arrays.items() if k != "big"}})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_MAX_ELEMS,)
    assert np.all(np.diff(a) > 0) and a[-1] < n and np.array_equal(b, 2 * a)     # distinct sorted indices, same each run
    f64 = np.load(tmp_path / "a" / "f64.npy")
    assert f64.dtype == np.float64 and np.array_equal(f64, arrays["f64"].numpy())
    bf = np.load(tmp_path / "a" / "bf16.npy")
    assert bf.dtype == np.float32 and np.array_equal(bf, arrays["bf16"].float().numpy())
    assert 6 * bench.DUMP_MAX_ELEMS * 4 < 64e6


def test_weight_gradient_split_rows_equals_one_gemm():
    """deform_conv._wgrad: the batched split-row product (taken for narrow layers with 10^5+ rows) and the single GEMM
    agree; odd row counts exercise the remainder slab."""
    from devis_b200 import deform_conv
    g = torch.Generator().manual_seed(0)
    for rows, cout, kc in ((8 * 2048 + 77, 16, 288), (8 * 2048, 4, 36), (1000, 16, 288), (8 * 2048 + 5, 1, 144)):
        g2 = torch.randn(rows, cout, generator=g, dtype=torch.float64)
        cols = torch.randn(rows + 3, kc, generator=g, dtype=torch.float64)
        got = deform_conv._wgrad(g2, cols[:rows])
        want = g2.t() @ cols[:rows]
        assert got.shape == want.shape and torch.allclose(got, want, rtol=1e-12, atol=1e-10)
