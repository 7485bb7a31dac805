"""Times the fused-prologue whole-clip op (TemporalMSDeformAttnFusedFunction: softmax + location arithmetic inside the
kernels) forward and forward+backward at the DeVIS R50 T=6 encoder shape, through autograd, with CUDA events.

    python benchmarks/fused_bench.py [--dtype fp32|bf16|fp16] [--iters 30]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import TemporalMSDeformAttnFusedFunction, clip_geometry, synthetic  # noqa: E402
from benchmarks.sweep import time_us  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--dtype", default="fp32")
ap.add_argument("--iters", type=int, default=30)
a = ap.parse_args()
dtype = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[a.dtype]
torch.manual_seed(0)
T, shapes_l, M, D, pc, pt = 6, synthetic.DEVIS_SHAPES, 8, 32, 4, 4
nl, wt = len(shapes_l), T - 1
S = sum(h * w for h, w in shapes_l)
geom = clip_geometry.ClipGeometry(shapes_l, T, clip_geometry.all_frames_table(T))
order = geom.tile_order("cuda")
ref = synthetic.pixel_reference_points(shapes_l, T, "cuda")
value = torch.randn(T, S, M, D, device="cuda", dtype=dtype).requires_grad_(True)
off_c = (2.0 * torch.randn(T, S, M, nl, pc, 2, device="cuda")).requires_grad_(True)
off_t = (2.0 * torch.randn(T, S, M, wt * nl, pt, 2, device="cuda")).requires_grad_(True)
lg_c = torch.randn(T, S, M, nl * pc, device="cuda").requires_grad_(True)
lg_t = torch.randn(T, S, M, wt * nl * pt, device="cuda").requires_grad_(True)
gout = torch.randn(T, S, M * D, device="cuda", dtype=dtype)


def fwd():
    with torch.no_grad():
        return TemporalMSDeformAttnFusedFunction.apply(value, ref, off_c, lg_c, off_t, lg_t, geom, order)


def fwd_bwd():
    for t in (value, off_c, off_t, lg_c, lg_t):
        t.grad = None
    TemporalMSDeformAttnFusedFunction.apply(value, ref, off_c, lg_c, off_t, lg_t, geom, order).backward(gout)


f = time_us(fwd, a.iters)
fb = time_us(fwd_bwd, a.iters)
print(json.dumps({"dtype": a.dtype, "fused_fwd_us": round(f, 1), "fused_fwd_bwd_us": round(fb, 1), "lib": os.environ.get("DEVIS_MSDA_LIB", "in-tree")}))
