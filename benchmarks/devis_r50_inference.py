"""BASELINE.json config 3: DeVIS R50 T=6 full-model INFERENCE on synthetic 360 x 640 clips, random-init weights, one B200.

    python benchmarks/devis_r50_inference.py [--attn ours|reference|both] [--iters 20] [--num-out 20] [--train]

This is a BENCHMARK ASSEMBLY, not a product module: the hot path of this repository (temporal attention modules, mask-head
deformable convolution) embedded in everything DeVIS runs around it at inference, so that the end-to-end effect of the
kernels can be measured.  Everything outside the hot path is stock PyTorch / torchvision:

  backbone            torchvision resnet50, FrozenBatchNorm2d, layers 1-4 (strides 4 / 8 / 16 / 32)      backbone.py:62-128
  position encoding   2-d sine, normalised                                                              position_encoding.py:64-105
  input projections   1x1 conv + GroupNorm(32) on C3-C5, 3x3 stride-2 conv + GroupNorm for /64           deformable_detr.py:60-88
  transformer         devis_b200.DeVISTransformer (6 + 6 layers, 4 + 4 points, all frames connected)    devis_transformer.py
  heads               class_embed / bbox_embed per decoder layer, box refinement                        deformable_detr.py:51-119
  instance selection  DeVISPostProcessor: trajectory scores, top-k, unique                              devis_segmentation.py:116-186
  mask head           MultiScaleMHAttentionMap + MaskHeadConv (deformable convolutions)                 deformable_segmentation.py:276-380

as wired by DefDETRSegmBase.forward / DeVIS._inference_forward (deformable_segmentation.py:118-135,
devis_segmentation.py:77-112) with the defaults of config.py + configs/devis/YT-19/devis_R_50_YT-19.yaml (60 queries = 10
trajectories x 6 frames, 40 classes, TEST.NUM_OUT 20, mask-head features /32 /16 /8 encoded + /4 backbone).

`--attn reference` evaluates the SAME model and weights the reference's way: per-frame Python loop + gather copies + the
reference's own CUDA op (oracle/_ref) in all 12 attention modules, torchvision.ops.deform_conv2d in the mask head.
Timing: CUDA events around whole clips after warm-up, explicit synchronisation (the reference's FPS counter has none),
median.  Prints one JSON object."""
import argparse
import json
import math
import os
import statistics
import sys
import time

import torch
import torch.nn.functional as F
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from devis_b200 import DeVISTransformer, _lib  # noqa: E402
from devis_b200 import deformable_segmentation as segm  # noqa: E402
from devis_b200.modules import TemporalMSDeformAttnDecoder, TemporalMSDeformAttnEncoder  # noqa: E402


def sine_position(mask, num_pos_feats=128, temperature=10000.0):
    """(T, H, W) padding mask -> (T, 2 * num_pos_feats, H, W), normalised 2-d sine encoding"""
    not_mask = ~mask
    y = not_mask.cumsum(1, dtype=torch.float32)
    x = not_mask.cumsum(2, dtype=torch.float32)
    y = y / (y[:, -1:, :] + 1e-6) * (2 * math.pi)
    x = x / (x[:, :, -1:] + 1e-6) * (2 * math.pi)
    dim_t = torch.arange(num_pos_feats, dtype=torch.float32, device=mask.device)
    dim_t = temperature ** (2 * torch.div(dim_t, 2, rounding_mode="trunc") / num_pos_feats)
    px, py = x[..., None] / dim_t, y[..., None] / dim_t
    px = torch.stack((px[..., 0::2].sin(), px[..., 1::2].cos()), 4).flatten(3)
    py = torch.stack((py[..., 0::2].sin(), py[..., 1::2].cos()), 4).flatten(3)
    return torch.cat((py, px), 3).permute(0, 3, 1, 2)


class MLP(nn.Module):
    def __init__(self, din, hidden, dout, layers):
        super().__init__()
        dims = [din] + [hidden] * (layers - 1) + [dout]
        self.layers = nn.ModuleList(nn.Linear(a, b) for a, b in zip(dims[:-1], dims[1:]))

    def forward(self, x):
        for i, layer in enumerate(self.layers):
            x = layer(x) if i == len(self.layers) - 1 else F.relu(layer(x))
        return x


class DeVISR50(nn.Module):
    def __init__(self, n_frames=6, n_queries=60, n_classes=40, hidden=256, num_out=20):
        super().__init__()
        import torchvision
        from torchvision.models._utils import IntermediateLayerGetter
        from torchvision.ops.misc import FrozenBatchNorm2d
        self.n_frames, self.n_queries, self.num_out = n_frames, n_queries, num_out
        net = torchvision.models.resnet50(weights=None, norm_layer=FrozenBatchNorm2d)
        self.body = IntermediateLayerGetter(net, {"layer1": "0", "layer2": "1", "layer3": "2", "layer4": "3"})
        chans = [256, 512, 1024, 2048]
        proj = [nn.Sequential(nn.Conv2d(c, hidden, 1), nn.GroupNorm(32, hidden)) for c in chans[1:]]
        proj.append(nn.Sequential(nn.Conv2d(chans[-1], hidden, 3, stride=2, padding=1), nn.GroupNorm(32, hidden)))
        self.input_proj = nn.ModuleList(proj)
        self.transformer = DeVISTransformer(d_model=hidden, num_frames=n_frames, nhead=8, num_encoder_layers=6,
                                            num_decoder_layers=6, dim_feedforward=1024, dropout=0.1,
                                            num_feature_levels=4, enc_connect_all_embeddings=True, enc_n_curr_points=4,
                                            enc_n_temporal_points=4, dec_n_curr_points=4, dec_n_temporal_points=4,
                                            dec_instance_aware_att=True, with_gradient=True)
        self.query_embed = nn.Embedding(n_queries, 2 * hidden)
        self.class_embed = nn.ModuleList(nn.Linear(hidden, n_classes + 1) for _ in range(6))
        self.bbox_embed = nn.ModuleList(MLP(hidden, hidden, 4, 3) for _ in range(6))
        self.transformer.decoder.bbox_embed = self.bbox_embed         # iterative box refinement
        self.bbox_attention = segm.MultiScaleMHAttentionMap(hidden, hidden, 8, num_levels=3, dropout=0)
        self.mask_head = segm.MaskHeadConv(hidden, [hidden, hidden, chans[0]], 8, True, ["/32", "/16", "/8"], num_levels=4)

    def trunk(self, frames, pad_mask):
        feats = [v for _, v in sorted(self.body(frames).items())]
        masks = [F.interpolate(pad_mask[None].float(), size=f.shape[-2:]).to(torch.bool)[0] for f in feats]
        srcs = [self.input_proj[i](f) for i, f in enumerate(feats[1:])]
        srcs.append(self.input_proj[3](feats[-1]))
        lvl_masks = masks[1:] + [F.interpolate(pad_mask[None].float(), size=srcs[-1].shape[-2:]).to(torch.bool)[0]]
        pos = [sine_position(m) for m in lvl_masks]
        hs, _, memories, _, inter_refs, *_ = self.transformer(srcs, lvl_masks, pos, self.query_embed.weight)
        return feats, lvl_masks, hs, memories, inter_refs

    def masks_for(self, hs_f, feats, lvl_masks, memories, n):
        """box attention maps and the convolutional mask head on /32, /16, /8 encoded + /4 backbone features"""
        mem = [memories[i][0].transpose(0, 1) for i in (2, 1, 0)]
        bbox_mask = self.bbox_attention(hs_f, mem, mask=[lvl_masks[i] for i in (2, 1, 0)])
        bbox_mask = [b.transpose(1, 0).flatten(0, 1) for b in bbox_mask]
        seg = self.mask_head(mem + [feats[0]], bbox_mask, instances_per_batch=n,
                             expand_func=lambda t, k: t.repeat(k, 1, 1, 1))
        return seg.view((n, self.n_frames) + seg.shape[2:])

    def training_loss(self, frames, pad_mask, n_matched=5):
        """BASELINE config 5's forward: every decoder level's class / box outputs (auxiliary losses) and the masks of
        `n_matched` trajectories at the last level (DeVIS._training_forward with a fixed matching: the Hungarian matcher and
        SetCriterion are CPU / out of scope, devis_segmentation.py:37-45,69-75); a synthetic quadratic loss stands in for
        the criterion so that every parameter on the path gets a gradient."""
        feats, lvl_masks, hs, memories, inter_refs = self.trunk(frames, pad_mask)
        loss = frames.new_zeros(())
        for lvl in range(hs.shape[0]):
            loss = loss + self.class_embed[lvl](hs[lvl]).float().square().mean() + inter_refs[lvl].float().square().mean()
        n_traj = self.n_queries // self.n_frames
        hs_f = hs[-1][0].view(self.n_frames, n_traj, -1)[:, :n_matched]
        seg = self.masks_for(hs_f, feats, lvl_masks, memories, n_matched)
        return loss + seg.float().square().mean() + 1e-3 * sum(m.float().square().mean() for m in memories)

    @torch.no_grad()
    def forward(self, frames, pad_mask):
        """frames (T, 3, H, W), pad_mask (T, H, W) bool -> (masks (n, T, H/4, W/4), scores, labels, boxes)"""
        feats, lvl_masks, hs, memories, inter_refs = self.trunk(frames, pad_mask)
        logits = self.class_embed[-1](hs[-1])                         # (1, T * n_traj, classes + 1)
        boxes = inter_refs[-1]                                        # with_gradient: the refined boxes themselves
        # DeVISPostProcessor (focal loss): trajectory score = mean over frames, top-k over (trajectory, class)
        n_traj = self.n_queries // self.n_frames
        probs = logits.sigmoid()[0].reshape(self.n_frames, n_traj, -1)
        traj = probs.transpose(0, 1).mean(1).flatten()
        scores, top = torch.topk(traj, self.num_out)
        traj_idx = torch.div(top, probs.shape[-1], rounding_mode="trunc")
        labels = top % probs.shape[-1]
        uniq, inverse = torch.unique(traj_idx, return_inverse=True)   # host-visible size, as in the reference
        n = int(uniq.shape[0])
        hs_f = hs[-1][0].view(self.n_frames, n_traj, -1)[:, uniq]
        seg = self.masks_for(hs_f, feats, lvl_masks, memories, n)
        return seg, scores, labels, boxes.view(self.n_frames, n_traj, 4)[:, uniq], inverse


def use_reference_ops(model):
    """evaluate every temporal attention module the reference's way (its CUDA op, per-frame loop, gather copies) and the
    mask head's deformable convolutions with torchvision's operator; parameters untouched"""
    import types

    import torchvision

    from benchmarks.module_bench import RefFunction, reference_style_decoder, reference_style_encoder
    from oracle import ref_cuda_build
    RefFunction.mod = ref_cuda_build.load()

    def enc_forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                    temporal_offsets):
        return reference_style_encoder(self, RefFunction.apply, query, reference_points, input_flatten,
                                       input_spatial_shapes[0], input_level_start_index[0], input_spatial_shapes[1],
                                       input_level_start_index[1], temporal_offsets), None

    def dec_forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                    temporal_offsets):
        offs = [torch.as_tensor(o, device=query.device) for o in temporal_offsets]
        out = reference_style_decoder(self, RefFunction.apply, query, reference_points, input_flatten,
                                      input_spatial_shapes[0], input_level_start_index[0], input_spatial_shapes[1],
                                      input_level_start_index[1], offs)
        return out, None, None, None, None

    def mdc_forward(self, x):
        offset = self.offset_conv(x)
        modulator = 2. * torch.sigmoid(self.modulator_conv(x))
        return torchvision.ops.deform_conv2d(x, offset, self.regular_conv.weight, self.regular_conv.bias,
                                             padding=self.padding, mask=modulator)

    for mod in model.modules():
        if isinstance(mod, TemporalMSDeformAttnEncoder):
            mod.forward = types.MethodType(enc_forward, mod)
        elif isinstance(mod, TemporalMSDeformAttnDecoder):
            mod.forward = types.MethodType(dec_forward, mod)
        elif isinstance(mod, segm.ModulatedDeformableConv2d):
            mod.forward = types.MethodType(mdc_forward, mod)


def time_clips(model, frames, pad, iters, warmup=3):
    for _ in range(warmup):
        model(frames, pad)
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record()
        model(frames, pad)
        b.record()
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in evs]
    return {"ms_per_clip_median": round(statistics.median(ms), 3), "ms_per_clip_min": round(min(ms), 3),
            "clips_per_sec": round(1e3 / statistics.median(ms), 3), "frames_per_sec": round(6e3 / statistics.median(ms), 2),
            "iters": iters}


def stage_breakdown(model, frames, pad):
    """where a clip's time goes (torch profiler, CUDA time by kernel family)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            model(frames, pad)
        torch.cuda.synchronize()
    fam = {"attention (msda / tmsda kernels)": 0.0, "deformable conv (dcn kernels)": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", 0.0) or getattr(ev, "cuda_time_total", 0.0)
        name = ev.key
        if "msda" in name or "ms_deform" in name:                    # this library's / the reference's attention kernels
            fam["attention (msda / tmsda kernels)"] += t
        elif "dcn" in name or "deformable_im2col" in name or "deformable_col2im" in name:   # ours / torchvision's
            fam["deformable conv (dcn kernels)"] += t
        else:
            fam["other"] += t
    return {k: round(v / 3e3, 3) for k, v in fam.items()}      # ms per clip


def run_train(attn="both", iters=8, height=360, width=640, tf32=False, ddp=None, n_matched=5):
    """BASELINE config 5 on the whole model: forward (all decoder levels + masks of `n_matched` trajectories) + backward +
    gradient all-reduce (when `ddp` wraps the model: pass a callable module -> DistributedDataParallel) + clip_grad_norm(0.1)
    + AdamW, one synthetic clip per rank; returns ms per step (CUDA events, median)."""
    torch.manual_seed(0)
    dev = torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    torch.backends.cudnn.allow_tf32 = bool(tf32)
    out = {"config": "DeVIS R50 training step, T=6, %dx%d, 60 queries, 6+6 layers, 4+4 points, dropout 0.1, %d matched "
                     "trajectories in the mask head, aux outputs of all decoder levels, synthetic quadratic loss, fp32 (TF32 %s), "
                     "AdamW + clip_grad_norm 0.1" % (height, width, n_matched, "on" if tf32 else "off")}
    frames = torch.randn(6, 3, height, width, device=dev)
    pad = torch.zeros(6, height, width, dtype=torch.bool, device=dev)

    def measure(model):
        class Step(nn.Module):
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, x):
                return self.m.training_loss(x, pad, n_matched)
        net = Step(model)
        runner = ddp(net) if ddp is not None else net
        params = [p for p in net.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=1e-4)

        def step():
            opt.zero_grad(set_to_none=True)
            runner(frames).backward()
            torch.nn.utils.clip_grad_norm_(params, 0.1)
            opt.step()
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in evs:
            a.record()
            step()
            b.record()
        torch.cuda.synchronize()
        ms = statistics.median(a.elapsed_time(b) for a, b in evs)
        return {"ms_per_step": round(ms, 3), "clips_per_sec": round(1e3 / ms, 3), "iters": iters,
                "trainable_params": sum(p.numel() for p in params)}

    model = DeVISR50().to(dev).train()
    for p in model.body.parameters():                     # the reference trains the backbone at lr 1e-5; kept trainable
        p.requires_grad_(True)
    if attn in ("ours", "both"):
        out["ours"] = measure(model)
    if attn in ("reference", "both"):
        try:
            use_reference_ops(model)
            out["reference_ops"] = measure(model)
            if "ours" in out:
                out["speedup"] = round(out["reference_ops"]["ms_per_step"] / out["ours"]["ms_per_step"], 3)
        except Exception as exc:  # noqa: BLE001
            out["reference_ops"] = {"error": str(exc)[:300]}
    return out


def run_train_determinism(height=360, width=640, tf32=False, n_matched=5, steps=2):
    """Bit-reproducible training with this library's kernels (--train --deterministic, --attn ours): under
    torch.use_deterministic_algorithms(True) run `steps` training steps (forward, backward, clip_grad_norm, AdamW) from
    the same seed twice and report whether every parameter ends bit-identical.  If an op outside this library has no
    deterministic implementation, torch raises and the op is reported instead."""
    dev = torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    torch.backends.cudnn.allow_tf32 = bool(tf32)
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        finals = []
        for _ in range(2):
            torch.manual_seed(0)
            frames = torch.randn(6, 3, height, width, device=dev)
            pad = torch.zeros(6, height, width, dtype=torch.bool, device=dev)
            model = DeVISR50().to(dev).train()
            for p in model.body.parameters():
                p.requires_grad_(True)
            params = [p for p in model.parameters() if p.requires_grad]
            opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=1e-4)
            for _ in range(steps):
                opt.zero_grad(set_to_none=True)
                model.training_loss(frames, pad, n_matched).backward()
                torch.nn.utils.clip_grad_norm_(params, 0.1)
                opt.step()
            finals.append({k: v.detach().clone() for k, v in model.named_parameters()})
            del model, opt
    except RuntimeError as exc:
        return {"error": str(exc)[:500]}
    finally:
        torch.use_deterministic_algorithms(old)
    differ = [k for k in finals[0] if not torch.equal(finals[0][k], finals[1][k])]
    return {"steps": steps, "parameters": len(finals[0]), "bit_identical": not differ, "differing": differ[:20]}


def run(attn="both", iters=20, num_out=20, breakdown=True, height=360, width=640, tf32=False):
    """tf32: torch.backends.{cuda.matmul,cudnn}.allow_tf32 for everything dense (backbone, projections, FFN, mask-head
    GEMMs; the reference's pinned torch 1.11 had both on by default).  The attention kernels are fp32 either way."""
    torch.manual_seed(0)
    dev = torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    torch.backends.cudnn.allow_tf32 = bool(tf32)
    model = DeVISR50(num_out=num_out).to(dev).eval()
    frames = torch.randn(6, 3, height, width, device=dev)
    pad = torch.zeros(6, height, width, dtype=torch.bool, device=dev)
    out = {"config": "DeVIS R50, T=6, %dx%d, 60 queries (10 trajectories), 6+6 layers, 4+4 points, NUM_OUT %d, random "
                     "init, eval mode, fp32 (TF32 %s), synthetic clip resident on the device" % (height, width, num_out, "on" if tf32 else "off"),
           "params": sum(p.numel() for p in model.parameters())}
    if attn in ("ours", "both"):
        before = _lib.launch_count()
        seg, *_ = model(frames, pad)
        assert _lib.launch_count() > before, "the library's kernels did not run"
        out["mask_shape"] = list(seg.shape)
        out["ours"] = time_clips(model, frames, pad, iters)
        if breakdown:
            out["ours"]["cuda_ms_per_clip_by_family"] = stage_breakdown(model, frames, pad)
    if attn in ("reference", "both"):
        try:
            use_reference_ops(model)
            out["reference_ops"] = time_clips(model, frames, pad, max(5, iters // 2))
            out["reference_ops"]["what"] = ("same model and weights; attention = the reference's per-frame loop + its own CUDA op "
                                            "(oracle/_ref), mask head = torchvision.ops.deform_conv2d")
            if breakdown:
                out["reference_ops"]["cuda_ms_per_clip_by_family"] = stage_breakdown(model, frames, pad)
            if "ours" in out:
                out["speedup"] = round(out["reference_ops"]["ms_per_clip_median"] / out["ours"]["ms_per_clip_median"], 3)
        except Exception as exc:  # noqa: BLE001  (oracle/_ref absent: report, do not fail the bench)
            out["reference_ops"] = {"error": str(exc)[:300]}
    return out


def _card():
    """name and power limit of the device the numbers were taken on (part of every absolute number)"""
    import subprocess
    info = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = "not read: %s" % exc
    return info


def run_compile(train=False, iters=10, rounds=3, height=360, width=640, tf32=False, n_matched=5):
    """The model eager and with torch.compile (inductor, default mode) in one process, timed in alternating rounds of
    `iters` calls each (CUDA events, median per round).  Compiled: the trunk (backbone, input projections, the whole
    DeVIS transformer with our attention ops) and the mask head (our deformable convolutions); the box attention maps
    (MultiScaleMHAttentionMap) and the post-processing stay eager -- inductor in torch 2.11 fails on the in-place
    masked_fill_ of the attention-map einsum.  Inference: DeVISR50.forward; train: the training step of run_train
    (forward + backward; clip_grad_norm and AdamW stay eager)."""
    torch.manual_seed(0)
    dev = torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    torch.backends.cudnn.allow_tf32 = bool(tf32)
    frames = torch.randn(6, 3, height, width, device=dev)
    pad = torch.zeros(6, height, width, dtype=torch.bool, device=dev)
    model = DeVISR50().to(dev)
    head, trunk = model.mask_head, torch.compile(model.trunk)
    compiled_head = torch.compile(head)

    def use(compiled):
        if compiled:
            model.trunk, model.mask_head = trunk, compiled_head
        else:
            model.__dict__.pop("trunk", None)
            model.mask_head = head
    if train:
        model.train()
        for p in model.body.parameters():
            p.requires_grad_(True)
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=1e-4)

        def make(flag):
            def step():
                use(flag)
                opt.zero_grad(set_to_none=True)
                model.training_loss(frames, pad, n_matched).backward()
                torch.nn.utils.clip_grad_norm_(params, 0.1)
                opt.step()
            return step
    else:
        model.eval()

        def make(flag):
            def fwd():
                use(flag)
                model(frames, pad)
            return fwd
    eager, compiled = make(False), make(True)
    t0 = time.perf_counter()
    for _ in range(3):
        compiled()                         # compilation + warm-up
    torch.cuda.synchronize()
    compile_s = time.perf_counter() - t0
    for _ in range(3):
        eager()
    before = _lib.launch_count()
    compiled()
    torch.cuda.synchronize()
    assert _lib.launch_count() > before, "the library's kernels did not run in the compiled model"

    def timed(fn):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in evs:
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return statistics.median(a.elapsed_time(b) for a, b in evs)
    per_round = {"eager": [], "compiled": []}
    for _ in range(rounds):
        per_round["eager"].append(round(timed(eager), 3))
        per_round["compiled"].append(round(timed(compiled), 3))
    med = {k: statistics.median(v) for k, v in per_round.items()}
    return {"config": "DeVIS R50 %s, T=6, %dx%d, 60 queries, fp32 (TF32 %s), torch.compile(inductor) vs eager, %d "
                      "alternating rounds x %d calls" % ("training step" if train else "inference", height, width,
                                                         "on" if tf32 else "off", rounds, iters),
            "ms_eager_median": round(med["eager"], 3), "ms_compiled_median": round(med["compiled"], 3),
            "speedup": round(med["eager"] / med["compiled"], 3), "ms_per_round": per_round,
            "compile_and_warmup_s": round(compile_s, 1), **_card()}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--attn", default="both", choices=["ours", "reference", "both"])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--num-out", type=int, default=20)
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--tf32", default="both", choices=["off", "on", "both"])
    ap.add_argument("--train", action="store_true", help="time the training step (config 5) instead of inference (config 3)")
    ap.add_argument("--deterministic", action="store_true",
                    help="with --train --attn ours: check that two seeded training runs end bit-identical instead of timing")
    ap.add_argument("--compile", action="store_true",
                    help="time the whole model (inference, or with --train the training step) eager and under "
                         "torch.compile in alternating rounds")
    a = ap.parse_args()
    if a.deterministic and not (a.train and a.attn == "ours"):
        ap.error("--deterministic needs --train --attn ours")
    if a.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")    # before the first cuBLAS call
    res = {}
    for mode in (["off", "on"] if a.tf32 == "both" else [a.tf32]):
        if a.compile:
            res["tf32_" + mode] = run_compile(a.train, max(4, a.iters // 2), tf32=mode == "on")
        elif a.deterministic:
            res["tf32_" + mode] = run_train_determinism(tf32=mode == "on")
        elif a.train:
            res["tf32_" + mode] = run_train(a.attn, max(4, a.iters // 3), tf32=mode == "on")
        else:
            res["tf32_" + mode] = run(a.attn, a.iters, a.num_out, not a.no_breakdown, tf32=mode == "on")
    print(json.dumps(res))
