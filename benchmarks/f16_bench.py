"""fp16 against bf16 value at the DeVIS R50 T=6 encoder layer-clip: the whole-clip op (C ABI on preallocated buffers, as
benchmarks/sweep.py and tests/test_perf_guard_gpu.py time it) and the fused-prologue op (through autograd, as
benchmarks/fused_bench.py), forward and backward.  The two dtypes alternate round by round in one process, so that clock
and neighbour drift hit both alike; each number is the median over the rounds of a CUDA-event mean.

    python benchmarks/f16_bench.py [--rounds 7] [--iters 20] [--out file.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import TemporalMSDeformAttnFusedFunction, clip_geometry, synthetic  # noqa: E402
from benchmarks.sweep import RawClip, time_us  # noqa: E402


def card():
    """name and power limit of GPU 0: part of every number below"""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = (x.strip() for x in q.split(","))
    except (OSError, ValueError, subprocess.SubprocessError):
        info["power_limit"] = "unknown"
    return info


class Fused:
    """fused-prologue op on raw Linear-like operands at the encoder layer-clip (pixel reference points)"""

    def __init__(self, dtype):
        torch.manual_seed(0)
        T, shapes_l, M, D, pc, pt = 6, synthetic.DEVIS_SHAPES, 8, 32, 4, 4
        nl, wt = len(shapes_l), T - 1
        S = sum(h * w for h, w in shapes_l)
        self.geom = clip_geometry.ClipGeometry(shapes_l, T, clip_geometry.all_frames_table(T))
        self.order = self.geom.tile_order("cuda")
        self.ref = synthetic.pixel_reference_points(shapes_l, T, "cuda")
        self.value = torch.randn(T, S, M, D, device="cuda", dtype=dtype).requires_grad_(True)
        self.off_c = (2.0 * torch.randn(T, S, M, nl, pc, 2, device="cuda")).requires_grad_(True)
        self.off_t = (2.0 * torch.randn(T, S, M, wt * nl, pt, 2, device="cuda")).requires_grad_(True)
        self.lg_c = torch.randn(T, S, M, nl * pc, device="cuda").requires_grad_(True)
        self.lg_t = torch.randn(T, S, M, wt * nl * pt, device="cuda").requires_grad_(True)
        self.gout = torch.randn(T, S, M * D, device="cuda", dtype=dtype)

    def _apply(self):
        return TemporalMSDeformAttnFusedFunction.apply(self.value, self.ref, self.off_c, self.lg_c, self.off_t, self.lg_t,
                                                       self.geom, self.order)

    def fwd(self):
        with torch.no_grad():
            self._apply()

    def fwd_bwd(self):
        for t in (self.value, self.off_c, self.off_t, self.lg_c, self.lg_t):
            t.grad = None
        self._apply().backward(self.gout)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dtypes = {"fp16": torch.float16, "bf16": torch.bfloat16}
    ops = {}
    for name, dt in dtypes.items():
        clip = synthetic.make_clip(device="cuda", dtype=dt, dist="local")
        geom = clip_geometry.ClipGeometry(clip["shapes"], 6, clip["frame_table"])
        ops[name] = (RawClip(clip, geom.tile_order("cuda")), Fused(dt))
    samples = {n: {k: [] for k in ("clip_fwd_us", "clip_bwd_us", "fused_fwd_us", "fused_fwd_bwd_us")} for n in dtypes}
    for _ in range(a.rounds):
        for name in dtypes:
            rc, fu = ops[name]
            s = samples[name]
            s["clip_fwd_us"].append(time_us(rc.fwd, a.iters))
            s["clip_bwd_us"].append(time_us(rc.bwd, a.iters))
            s["fused_fwd_us"].append(time_us(fu.fwd, a.iters))
            s["fused_fwd_bwd_us"].append(time_us(fu.fwd_bwd, a.iters))
    res = {"workload": "DeVIS R50 T=6 encoder layer-clip (S=4820, 8 heads x 32 channels, 4 + 4 points, all frames)",
           "card": card(), "rounds": a.rounds, "iters": a.iters}
    for name in dtypes:
        med = {k: round(statistics.median(v), 1) for k, v in samples[name].items()}
        med["fused_bwd_us"] = round(med["fused_fwd_bwd_us"] - med["fused_fwd_us"], 1)
        med["spread_clip_fwd_us"] = round(max(samples[name]["clip_fwd_us"]) - min(samples[name]["clip_fwd_us"]), 1)
        med["spread_clip_bwd_us"] = round(max(samples[name]["clip_bwd_us"]) - min(samples[name]["clip_bwd_us"]), 1)
        res[name] = med
    print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
