"""Developer sweep (not the contract benchmark -- that is bench.py): times the whole-clip kernels at the
DeVIS R50 T=6 encoder shape for launch-shape variants, calling the C ABI directly on preallocated buffers.

    python benchmarks/sweep.py [--dist local|uniform] [--dtype fp32|bf16|fp16] [--iters 20]
"""
import argparse
import itertools
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import _lib, clip_geometry, synthetic  # noqa: E402


def ptr(t):
    return t.data_ptr() if t is not None else None


class RawClip:
    def __init__(self, clip, order=None):
        self.c = clip
        v = clip["value"]
        self.geom = clip_geometry.ClipGeometry(clip["shapes"], v.shape[0], clip["frame_table"])
        self.t, self.s, self.m, self.d = v.shape
        self.lq, self.pc, self.pt = clip["loc_curr"].shape[1], clip["loc_curr"].shape[4], clip["loc_temporal"].shape[4]
        self.code = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.bfloat16: _lib.BF16,
                     torch.float16: _lib.F16}[v.dtype]
        self.out = torch.empty(self.t, self.lq, self.m * self.d, dtype=v.dtype, device=v.device)
        self.gv = torch.empty(v.shape, dtype=torch.float32, device=v.device)
        self.gv_half = torch.empty(v.shape, dtype=torch.bfloat16, device=v.device) if v.dtype == torch.bfloat16 else None
        self.glc, self.gac = torch.empty_like(clip["loc_curr"]), torch.empty_like(clip["aw_curr"])
        self.glt, self.gat = torch.empty_like(clip["loc_temporal"]), torch.empty_like(clip["aw_temporal"])
        self.order = order
        self.lib = _lib.load()
        self.ws = None          # deterministic-mode workspace, allocated on first use

    def fwd(self):
        c, g = self.c, self.geom
        _lib.check(self.lib.devis_tmsda_forward(
            ptr(c["value"]), g.shapes_ptr, g.lsi_ptr, g.frames_ptr, ptr(c["loc_curr"]), ptr(c["aw_curr"]),
            ptr(c["loc_temporal"]), ptr(c["aw_temporal"]), ptr(self.out), ptr(self.order),
            self.t, self.s, self.m, self.d, g.n_levels, self.lq, self.pc, self.pt, g.t_window, self.code,
            torch.cuda.current_stream().cuda_stream))

    def bwd(self, flags=0):
        c, g = self.c, self.geom
        ws_ptr = None
        ws_bytes = int(self.lib.devis_tmsda_backward_workspace_bytes(
            self.t, self.s, self.m, self.d, g.n_levels, self.lq, self.pc, self.pt, g.t_window, self.code, flags))
        if ws_bytes:
            if self.ws is None or self.ws.numel() < ws_bytes:
                self.ws = torch.empty(ws_bytes, dtype=torch.uint8, device=c["value"].device)
            ws_ptr = self.ws.data_ptr()
        _lib.check(self.lib.devis_tmsda_backward(
            ptr(c["value"]), g.shapes_ptr, g.lsi_ptr, g.frames_ptr, ptr(c["loc_curr"]), ptr(c["aw_curr"]),
            ptr(c["loc_temporal"]), ptr(c["aw_temporal"]), ptr(c["grad_out"]),
            ptr(self.gv_half if flags & _lib.FLAG_BF16_GRAD_VALUE else self.gv), ptr(self.glc),
            ptr(self.gac), ptr(self.glt), ptr(self.gat), ptr(self.order),
            self.t, self.s, self.m, self.d, g.n_levels, self.lq, self.pc, self.pt, g.t_window, self.code, flags,
            ws_ptr, ws_bytes, torch.cuda.current_stream().cuda_stream))


def time_us(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dist", default="local")
    ap.add_argument("--dtype", default="fp32")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--queries", type=int, default=0)
    ap.add_argument("--out", default="")
    ap.add_argument("--sigma", type=float, default=2.0)
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--det", action="store_true", help="also time the deterministic backward")
    a = ap.parse_args()
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[a.dtype]
    clip = synthetic.make_clip(dist=a.dist, dtype=dtype, queries=a.queries or None, device="cuda", sigma_px=a.sigma)
    fb, bb = synthetic.algorithmic_bytes(6, 4820, 8, 32, clip["loc_curr"].shape[1], 96, elem=clip["value"].element_size())
    rows = []
    geom = clip_geometry.ClipGeometry(clip["shapes"], 6, clip["frame_table"])
    orders = {"none": None}
    if not a.queries:
        for th, tw in (((8, 8),) if a.quick else ((4, 8), (8, 8), (8, 16), (16, 16))):
            orders[f"{th}x{tw}"] = geom.tile_order("cuda", th, tw)
    for oname, order in orders.items():
        rc = RawClip(clip, order)
        for threads, qpg in (((256, 1), (256, 2)) if a.quick else itertools.product((128, 256), (1, 2, 4))):
            _lib.set_tuning(0, threads); _lib.set_tuning(1, qpg)
            f = time_us(rc.fwd, a.iters)
            rows.append(dict(kind="fwd", order=oname, threads=threads, qpg=qpg, us=round(f, 1), gbs=round(fb / f / 1e3, 1)))
            print(rows[-1], flush=True)
        for threads, qpg in (((128, 1), (256, 1)) if a.quick else itertools.product((128, 256), (1, 2))):
            _lib.set_tuning(2, threads); _lib.set_tuning(3, qpg)
            b = time_us(rc.bwd, a.iters)
            rows.append(dict(kind="bwd", order=oname, threads=threads, qpg=qpg, us=round(b, 1), gbs=round(bb / b / 1e3, 1)))
            print(rows[-1], flush=True)
            b2 = time_us(lambda: rc.bwd(2), a.iters)
            rows.append(dict(kind="bwd_nogv", order=oname, threads=threads, qpg=qpg, us=round(b2, 1)))
            print(rows[-1], flush=True)
            if a.dtype == "bf16":
                b4 = time_us(lambda: rc.bwd(_lib.FLAG_BF16_GRAD_VALUE), a.iters)
                rows.append(dict(kind="bwd_bf16acc", order=oname, threads=threads, qpg=1, us=round(b4, 1)))
                print(rows[-1], flush=True)
            if a.det:
                b3 = time_us(lambda: rc.bwd(_lib.FLAG_DETERMINISTIC), max(3, a.iters // 4), warmup=2)
                rows.append(dict(kind="bwd_det", order=oname, threads=threads, qpg=qpg, us=round(b3, 1)))
                print(rows[-1], flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    os.environ["DEVIS_MSDA_TUNING"] = "1"      # developer knobs (devis_msda_set_tuning) are inert without it
    main()
