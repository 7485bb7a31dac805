"""Modulated deformable convolution at DeVIS's mask-head layer shapes (BASELINE.json config 4, SURVEY.md appendix A):
this library (devis_b200.deform_conv: hand-written gather/scatter kernels + cuBLAS GEMM) against torchvision's CUDA
operator (the third-party kernel the reference calls, deformable_segmentation.py:265), forward and forward+backward.

    python benchmarks/dcn_bench.py [--instances 60] [--iters 30] [--json out.json] [--deterministic]

`instances` = trajectories x T reaching the mask head (<= TEST.NUM_OUT unique top-k x T at inference; 300/frame is the
synthetic stress shape of config 4 -- pass --instances 1800 if memory allows).  Prints one JSON line per layer and a
total; also the split gather-kernel / GEMM time of this library (C-ABI call on preallocated buffers).
--deterministic also times this library's forward+backward under torch.use_deterministic_algorithms(True) (64-bit
fixed-point grad_input), alternating with the default mode in the same process (median of --repeats rounds each).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# (name, Cin, Cout, H, W): MaskHeadConv.lay1..lay5 + out_lay for dim 256, 8 heads, att maps on /32 /16 /8, R50
LAYERS = [
    ("lay1", 264, 264, 12, 20),
    ("lay2", 264, 128, 12, 20),
    ("lay3", 136, 64, 23, 40),
    ("lay4", 72, 32, 45, 80),
    ("lay5", 32, 16, 90, 160),
    ("out_lay", 16, 1, 90, 160),
]


def _time(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3     # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=60)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--json", default=None)
    ap.add_argument("--tf32", action="store_true")
    ap.add_argument("--layers", default=None, help="comma-separated subset of layer names (e.g. lay5,out_lay)")
    ap.add_argument("--no-torchvision", action="store_true")
    ap.add_argument("--deterministic", action="store_true", help="also time the deterministic backward")
    ap.add_argument("--repeats", type=int, default=5, help="alternating rounds of --deterministic")
    args = ap.parse_args()
    if args.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")    # before the first cuBLAS call
    torch.backends.cuda.matmul.allow_tf32 = args.tf32
    from devis_b200 import _lib
    from devis_b200.deform_conv import deform_conv2d
    try:
        from torchvision.ops import deform_conv2d as tv_deform_conv2d
    except Exception:
        tv_deform_conv2d = None
    lib = _lib.load()
    gen = torch.Generator(device="cuda").manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=gen, device="cuda")
    n = args.instances
    rows, tot = [], {}
    if args.no_torchvision:
        tv_deform_conv2d = None
    for name, cin, cout, h, w in LAYERS:
        if args.layers and name not in args.layers.split(","):
            continue
        x = rn(n, cin, h, w).contiguous(memory_format=torch.channels_last)
        wt, b = rn(cout, cin, 3, 3) / (3 * cin ** 0.5), rn(cout)
        off, m = 1.5 * rn(n, 18, h, w), 2 * torch.sigmoid(rn(n, 9, h, w))
        gout = rn(n, cout, h, w)
        row = {"layer": name, "instances": n, "cin": cin, "cout": cout, "hw": [h, w]}

        leaf_sets = {}

        def step(fn, xin, backward):
            key = (xin.data_ptr(), backward)     # stable leaves, like module parameters (the packed-weight cache hits)
            if key not in leaf_sets:
                leaf_sets[key] = [t.detach().requires_grad_(backward) for t in (xin, off, wt, b, m)]
            leaves = leaf_sets[key]
            out = fn(leaves[0], leaves[1], leaves[2], leaves[3], padding=1, mask=leaves[4])
            if backward:
                out.backward(gout)
                for t in leaves:
                    t.grad = None

        row["ours_fwd_us"] = _time(lambda: step(deform_conv2d, x, False), args.iters)
        if args.deterministic:
            plain, det = [], []
            for _ in range(args.repeats):
                plain.append(_time(lambda: step(deform_conv2d, x, True), args.iters))
                torch.use_deterministic_algorithms(True)
                try:
                    det.append(_time(lambda: step(deform_conv2d, x, True), args.iters))
                finally:
                    torch.use_deterministic_algorithms(False)
            row["ours_fwd_bwd_us"] = statistics.median(plain)
            row["ours_det_fwd_bwd_us"] = statistics.median(det)
            row["ours_fwd_bwd_us_range"] = [round(min(plain), 1), round(max(plain), 1)]
            row["ours_det_fwd_bwd_us_range"] = [round(min(det), 1), round(max(det), 1)]
        else:
            row["ours_fwd_bwd_us"] = _time(lambda: step(deform_conv2d, x, True), args.iters)
        if tv_deform_conv2d is not None:
            xc = x.contiguous()      # torchvision wants NCHW
            try:
                row["torchvision_fwd_us"] = _time(lambda: step(tv_deform_conv2d, xc, False), args.iters)
                row["torchvision_fwd_bwd_us"] = _time(lambda: step(tv_deform_conv2d, xc, True), args.iters)
            except (RuntimeError, NotImplementedError) as exc:
                row["torchvision"] = f"unavailable: {str(exc)[:80]}"
                tv_deform_conv2d = None
        # the gather and scatter kernels alone, through the C ABI on preallocated buffers
        xl = x.permute(0, 2, 3, 1)
        assert xl.is_contiguous()
        cols = torch.empty(n * h * w, 9 * cin, device="cuda")
        gcols = rn(n * h * w, 9 * cin)
        gx, goff, gm = torch.empty_like(xl), torch.empty_like(off), torch.empty_like(m)
        dims = (n, h, w, cin, h, w, 3, 3, 1, 1, 1, 1, 1, 1)
        st = torch.cuda.current_stream().cuda_stream
        row["im2col_kernel_us"] = _time(lambda: _lib.check(lib.devis_dcn_im2col(
            x.data_ptr(), off.data_ptr(), m.data_ptr(), cols.data_ptr(), *dims, _lib.F32, st)), args.iters)
        row["col2im_kernel_us"] = _time(lambda: _lib.check(lib.devis_dcn_col2im(
            x.data_ptr(), off.data_ptr(), m.data_ptr(), gcols.data_ptr(), gx.data_ptr(), goff.data_ptr(), gm.data_ptr(),
            *dims, _lib.F32, st)), args.iters)
        # fused gather + contraction kernels (layers they serve), same way
        form = lib.devis_dcn_fused_form(cin, cout, 3, 3, _lib.F32)
        if form:
            packed = torch.empty(int(lib.devis_dcn_packed_weight_elems(cin, cout, 3, 3)), device="cuda")
            _lib.check(lib.devis_dcn_pack_weight(wt.data_ptr(), packed.data_ptr(), cin, cout, 3, 3, st))
            out = torch.empty(n, h, w, cout, device="cuda")
            gl = gout.permute(0, 2, 3, 1).contiguous()
        if form & 1:
            row["fused_fwd_kernel_us"] = _time(lambda: _lib.check(lib.devis_dcn_fused_forward(
                x.data_ptr(), off.data_ptr(), m.data_ptr(), packed.data_ptr(), b.data_ptr(), out.data_ptr(), *dims, cout,
                st)), args.iters)
            fb = 4 * (x.numel() + off.numel() + m.numel() + out.numel())
            row["fused_fwd_GBps"] = fb / row["fused_fwd_kernel_us"] / 1e3
        if form & 2:
            row["fused_bwd_kernel_us"] = _time(lambda: _lib.check(lib.devis_dcn_fused_backward(
                x.data_ptr(), off.data_ptr(), m.data_ptr(), packed.data_ptr(), gl.data_ptr(), gx.data_ptr(),
                goff.data_ptr(), gm.data_ptr(), *dims, cout, st)), args.iters)
            bb = 4 * (x.numel() + off.numel() + m.numel() + gl.numel() + gx.numel() + goff.numel() + gm.numel())
            row["fused_bwd_GBps"] = bb / row["fused_bwd_kernel_us"] / 1e3
        # algorithmic bytes of the gather: input + offset + mask read once, columns written once
        fwd_bytes = 4 * (x.numel() + off.numel() + m.numel() + cols.numel())
        row["im2col_GBps"] = fwd_bytes / row["im2col_kernel_us"] / 1e3
        bwd_bytes = 4 * (x.numel() + off.numel() + m.numel() + gcols.numel() + gx.numel() + goff.numel() + gm.numel())
        row["col2im_GBps"] = bwd_bytes / row["col2im_kernel_us"] / 1e3
        for k, v in row.items():
            if k.endswith("_us"):
                tot[k] = tot.get(k, 0.0) + v
        rows.append(row)
        print(json.dumps({k: (round(v, 1) if isinstance(v, float) else v) for k, v in row.items()}), flush=True)
        del x, cols, gcols, gx
    total = {"layer": "total", "instances": n, "tf32": args.tf32, **{k: round(v, 1) for k, v in tot.items()}}
    if args.deterministic:
        total["det_overhead"] = round(tot["ours_det_fwd_bwd_us"] / tot["ours_fwd_bwd_us"], 3)
    print(json.dumps(total), flush=True)
    if args.json:
        try:
            smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=60).stdout.strip()
        except (OSError, subprocess.SubprocessError):
            smi = "unavailable"
        with open(args.json, "w") as f:
            json.dump({"layers": rows, "total": total, "device": torch.cuda.get_device_name(0), "nvidia_smi": smi},
                      f, indent=1)


if __name__ == "__main__":
    main()
