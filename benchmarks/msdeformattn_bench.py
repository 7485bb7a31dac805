"""MSDeformAttn module: fused prologue (softmax, sampling locations and the input padding mask inside the attention
kernels) against fuse_prologue = False (today's unfused path: masked_fill copy of value, softmax kernel, location
arithmetic, MSDeformAttnFunction), alternating in one process, CUDA events, median per iteration.

  encoder: COCO pre-training shape, batch 2, pyramid (100,167) (50,84) (25,42) (13,21), one query per pixel
           (Lq = S = 22 223), 2-d reference points; padding mask as Deformable DETR builds it, image 2 at 75 % of
           image 1's height and width
  decoder: batch 2, Lq = 300 queries with box reference points, the same value pyramid and mask

Module forward (no autograd) and forward + backward, float32 and bfloat16 (the whole module in that type).  Prints one
JSON line: card, power limit, times in microseconds, speed-up, the largest fused / unfused output difference and the
kernel-family launch counts of one forward + backward per path (which kernels served it).

    python benchmarks/msdeformattn_bench.py [--iters 50] [--warmup 10] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import _lib, clip_geometry  # noqa: E402
from devis_b200.modules import MSDeformAttn  # noqa: E402

COCO = ((100, 167), (50, 84), (25, 42), (13, 21))
FAMILIES = ("FWD_GROUPED", "FWD_GENERIC", "BWD_GROUPED", "BWD_GENERIC", "FUSED_FWD", "FUSED_BWD", "BWD_SORTED", "AUX")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q or "unknown"


def detr_mask(n, shapes, valid):
    """True on padding; image-resolution mask resized to each level by nearest interpolation (Deformable DETR)"""
    h0, w0 = shapes[0][0] * 8, shapes[0][1] * 8
    m = torch.ones(n, h0, w0, dtype=torch.bool, device="cuda")
    for i, (fh, fw) in enumerate(valid):
        m[i, :round(h0 * fh), :round(w0 * fw)] = False
    return torch.cat([F.interpolate(m[None].float(), size=hw).to(torch.bool)[0].flatten(1) for hw in shapes], 1)


def encoder_ref(shapes, n):
    """pixel-centre reference points of every level, one per query (deformable_transformer.py get_reference_points
    with valid ratio 1)"""
    pts = []
    for h, w in shapes:
        y, x = torch.meshgrid(torch.arange(h, device="cuda") + 0.5, torch.arange(w, device="cuda") + 0.5, indexing="ij")
        pts.append(torch.stack([x.reshape(-1) / w, y.reshape(-1) / h], -1))
    pts = torch.cat(pts, 0)
    return pts[None, :, None, :].expand(n, -1, len(shapes), -1).contiguous()


def timed(fn, iters):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) * 1e3 for a, b in evs]


def counts(fn):
    before = {f: _lib.kernel_launches(getattr(_lib, "KERNEL_" + f)) for f in FAMILIES}
    fn()
    torch.cuda.synchronize()
    return {f: _lib.kernel_launches(getattr(_lib, "KERNEL_" + f)) - before[f] for f in FAMILIES
            if _lib.kernel_launches(getattr(_lib, "KERNEL_" + f)) - before[f]}


def bench_case(kind, dtype, iters, warmup):
    torch.manual_seed(0)
    n = 2
    shapes, lsi = clip_geometry.pyramid_tensors(COCO, "cuda")
    s = sum(h * w for h, w in COCO)
    mod = MSDeformAttn(256, 4, 8, 4)
    with torch.no_grad():
        mod.sampling_offsets.weight.normal_(0, 0.01)
        mod.attention_weights.weight.normal_(0, 0.01)
    mod = mod.to("cuda", dtype)
    if kind == "encoder":
        lq, ref = s, encoder_ref(COCO, n)
    else:
        lq = 300
        ref = torch.cat([torch.rand(n, lq, 1, 2, device="cuda") * 0.8 + 0.1,
                         torch.rand(n, lq, 1, 2, device="cuda") * 0.3 + 0.05], -1).expand(n, lq, 4, 4).contiguous()
    mask = detr_mask(n, COCO, [(1.0, 1.0), (0.75, 0.75)])
    query = torch.randn(n, lq, 256, device="cuda", dtype=dtype, requires_grad=True)
    inp = torch.randn(n, s, 256, device="cuda", dtype=dtype, requires_grad=True)
    gout = torch.randn(n, lq, 256, device="cuda", dtype=dtype)

    def fwd():
        with torch.no_grad():
            return mod(query, ref, inp, shapes, lsi, mask)[0]

    def train():
        out = mod(query, ref, inp, shapes, lsi, mask)[0]
        out.backward(gout)

    row = {"N": n, "Lq": lq, "S": s, "ref_dim": ref.shape[-1], "dtype": str(dtype).replace("torch.", "")}
    outs, launches = {}, {}
    for fuse in (True, False):
        mod.fuse_prologue = fuse
        outs[fuse] = fwd().float()
        launches["fused" if fuse else "unfused"] = counts(train)
        for _ in range(warmup):
            fwd()
            train()
    torch.cuda.synchronize()
    samples = {(f, p): [] for f in (True, False) for p in ("fwd", "train")}
    rounds = 5
    for _ in range(rounds):                     # alternate the two paths so drift on the shared host hits both
        for fuse in (True, False):
            mod.fuse_prologue = fuse
            samples[(fuse, "fwd")] += timed(fwd, max(1, iters // rounds))
            samples[(fuse, "train")] += timed(train, max(1, iters // rounds))
    for fuse in (True, False):
        tag = "fused" if fuse else "unfused"
        for p in ("fwd", "train"):
            v = samples[(fuse, p)]
            row[f"{tag}_{p}_us"] = round(statistics.median(v), 1)
            row[f"{tag}_{p}_iqr_us"] = round(statistics.quantiles(v, n=4)[2] - statistics.quantiles(v, n=4)[0], 1)
    for p in ("fwd", "train"):
        row[f"speedup_{p}"] = round(row[f"unfused_{p}_us"] / row[f"fused_{p}_us"], 3)
    row["out_nmax_fused_vs_unfused"] = float((outs[True] - outs[False]).abs().max() / outs[False].abs().max())
    row["launches_fwd_bwd"] = launches
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("msdeformattn_bench needs a CUDA device")
    name, power = card()
    res = {"bench": "msdeformattn_fused_vs_unfused", "gpu": name, "power_limit": power, "iters": a.iters,
           "note": "working set (value 45.5 MB fp32) fits the 126 MB L2; both paths see the same inputs"}
    for kind in ("encoder", "decoder"):
        for dtype in (torch.float32, torch.bfloat16):
            res[f"{kind}_{str(dtype).replace('torch.', '')}"] = bench_case(kind, dtype, a.iters, a.warmup)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
