"""Runs a few launches of one whole-clip kernel at the DeVIS R50 T=6 encoder shape: the command ncu wraps.
    python benchmarks/profile_one.py --kind fwd|bwd [--dist local] [--dtype fp32] [--iters 3]"""
import argparse
import os
import sys

import torch

os.environ["DEVIS_MSDA_TUNING"] = "1"      # developer knobs (devis_msda_set_tuning) are inert without it

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from benchmarks.sweep import RawClip  # noqa: E402
from devis_b200 import _lib, clip_geometry, synthetic  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--kind", default="fwd")
ap.add_argument("--dist", default="local")
ap.add_argument("--dtype", default="fp32")
ap.add_argument("--iters", type=int, default=3)
ap.add_argument("--tile", default="8x8")
ap.add_argument("--threads", type=int, default=0)
ap.add_argument("--qpg", type=int, default=0)
ap.add_argument("--sigma", type=float, default=2.0)
ap.add_argument("--bwd-mode", type=int, default=0, help="tuning key 6: 1 = the deterministic mode uses the direct 64-bit scatter instead of the sorted kernel")
ap.add_argument("--margin", type=int, default=0)
ap.add_argument("--min-level", type=int, default=0)
a = ap.parse_args()
clip = synthetic.make_clip(dist=a.dist, dtype={"fp32": torch.float32, "bf16": torch.bfloat16}[a.dtype], device="cuda", sigma_px=a.sigma)
geom = clip_geometry.ClipGeometry(clip["shapes"], 6, clip["frame_table"])
order = None if a.tile == "none" else geom.tile_order("cuda", *[int(x) for x in a.tile.split("x")])
rc = RawClip(clip, order)
for k in (0, 2):
    _lib.set_tuning(k, a.threads)
    _lib.set_tuning(k + 1, a.qpg)
_lib.set_tuning(6, a.bwd_mode)
_lib.set_tuning(7, a.margin)
_lib.set_tuning(9, a.min_level)
for _ in range(a.iters):
    rc.fwd() if a.kind == "fwd" else rc.bwd()
torch.cuda.synchronize()
