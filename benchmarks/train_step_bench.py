"""Benchmarks of the DeVIS transformer trunk (devis_b200.DeVISTransformer: 6 temporal-deformable encoder layers + 6
decoder layers) on synthetic R50 T=6 features -- BASELINE.json configs[2] and configs[4] without backbone / mask head /
criterion, which are out of scope.

  --mode train   forward + backward + gradient all-reduce (DDP over NCCL, one clip per rank like main.py:85,131) +
                 clip_grad_norm_(0.1) + AdamW: the body of train_one_epoch (engine.py:48-77)
  --mode infer   eval-mode forward under no_grad (inference_vis, engine.py:207-232); --graph replays the whole trunk
                 forward as ONE CUDA graph (possible because no layer reads a device tensor back: DeVISTransformer
                 attaches host copies of the pyramid shape, devis_transformer.py prepare_data)

    python benchmarks/train_step_bench.py [--mode train|infer] [--graph] [--steps 10] [--attn ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 benchmarks/train_step_bench.py

`--attn reference` evaluates the encoder's temporal attention the reference's way -- per-frame loop, gather copies of
value, the reference's own CUDA op (oracle/_ref) -- with the same parameters; single GPU only.
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.distributed as dist
from torch import nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import DeVISTransformer, synthetic  # noqa: E402
from devis_b200.modules import TemporalMSDeformAttnEncoder  # noqa: E402


class RefLoopEncoderAttn(TemporalMSDeformAttnEncoder):
    """same parameters, evaluated the reference's way: per-frame loop + gather copies + the reference CUDA op"""

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes, input_level_start_index,
                temporal_offsets):
        from benchmarks.module_bench import RefFunction, reference_style_encoder
        return reference_style_encoder(self, RefFunction.apply, query, reference_points, input_flatten,
                                       input_spatial_shapes[0], input_level_start_index[0], input_spatial_shapes[1],
                                       input_level_start_index[1], temporal_offsets), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="train", choices=["train", "infer"])
    ap.add_argument("--graph", action="store_true", help="infer: replay the trunk forward as one CUDA graph")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--attn", default="ours", choices=["ours", "reference"])
    ap.add_argument("--queries", type=int, default=10)
    ap.add_argument("--out", default="")
    ap.add_argument("--amp", default="off", choices=["off", "bf16", "fp16"],
                    help="bf16: run the step under torch.autocast (Linear layers on the bf16 tensor cores, the attention op "
                         "on bf16 value; the reference's op rejects bf16, cuda/ms_deform_attn_cuda.cu:64); fp16: "
                         "torch.autocast's default dtype, with torch.amp.GradScaler scaling the loss (standard fp16 AMP)")
    ap.add_argument("--tf32", action="store_true", help="allow TF32 in the fp32 GEMMs (torch.backends.cuda.matmul.allow_tf32)")
    a = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = bool(a.tf32)
    torch.backends.cudnn.allow_tf32 = bool(a.tf32)
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    T, shapes_l, C = 6, synthetic.DEVIS_SHAPES, 256
    torch.manual_seed(0)
    # config.py defaults of every released DeVIS model: 4 current + 4 temporal points, all frames connected
    trunk = DeVISTransformer(d_model=C, num_frames=T, enc_n_temporal_points=4, dec_n_temporal_points=4).to(dev)
    query_embed = nn.Embedding(T * a.queries, 2 * C).to(dev)
    if a.attn == "reference":
        from benchmarks.module_bench import RefFunction
        from oracle import ref_cuda_build
        RefFunction.mod = ref_cuda_build.load()
        assert RefFunction.mod is not None and world == 1
        for layer in trunk.encoder.layers:
            layer.self_attn.__class__ = RefLoopEncoderAttn
    model = nn.ModuleDict({"trunk": trunk, "query_embed": query_embed})
    n_params = sum(p.numel() for p in model.parameters())

    g = torch.Generator(device=dev).manual_seed(1 + rank)          # every rank its own clip
    srcs = [torch.randn(T, C, h, w, device=dev, generator=g) for h, w in shapes_l]
    pos = [torch.randn(T, C, h, w, device=dev, generator=g) for h, w in shapes_l]
    masks = [torch.zeros(T, h, w, dtype=torch.bool, device=dev) for h, w in shapes_l]

    class Step(nn.Module):                                         # one module so that DDP sees one forward
        def __init__(self):
            super().__init__()
            self.m = model

        def forward(self):
            amp_dtype = torch.float16 if a.amp == "fp16" else torch.bfloat16
            with torch.autocast("cuda", dtype=amp_dtype, enabled=a.amp != "off"):
                hs, _, memories, *_ = self.m["trunk"](srcs, masks, pos, self.m["query_embed"].weight)
            return hs, memories

    net = Step()
    if a.mode == "train":
        if world > 1:
            net = nn.parallel.DistributedDataParallel(net, device_ids=[local], find_unused_parameters=True)
        opt = torch.optim.AdamW(net.parameters(), lr=2e-4, weight_decay=1e-4)
        scaler = torch.amp.GradScaler("cuda", enabled=a.amp == "fp16")

        def step():
            opt.zero_grad(set_to_none=True)
            hs, memories = net()
            loss = hs[-1].float().square().mean() + 1e-3 * sum(m.float().square().mean() for m in memories)
            scaler.scale(loss).backward()
            scaler.unscale_(opt)
            torch.nn.utils.clip_grad_norm_(net.parameters(), 0.1)
            scaler.step(opt)
            scaler.update()
            return loss
    else:
        net.eval()
        graph, static = None, {}

        def eager():
            with torch.no_grad():
                hs, memories = net()
            return hs[-1].float().square().mean()

        if a.graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    eager()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static["loss"] = eager()

        def step():
            if graph is None:
                return eager()
            graph.replay()
            return static["loss"]

    for _ in range(a.warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    times = []
    for _ in range(a.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if rank == 0:
        what = ("training step: fwd+bwd+grad all-reduce+clip+AdamW" if a.mode == "train"
                else "inference forward (eval, no_grad" + (", one CUDA graph)" if a.graph else ", eager)"))
        res = {"workload": f"DeVIS transformer trunk {what}: 6 enc + 6 dec layers, T=6, S=4820, {a.queries} queries/frame, "
                           + (f"{a.amp} autocast" if a.amp != "off" else "fp32 + TF32 GEMMs" if a.tf32 else "fp32")
                           + ", synthetic features",
               "amp": a.amp, "tf32": bool(a.tf32),
               "mode": a.mode, "cuda_graph": bool(a.graph), "attention": a.attn, "n_gpus": world, "ms_per_step": ms,
               "clips_per_sec": world / (ms * 1e-3), "frames_per_sec": world * T / (ms * 1e-3), "params": n_params,
               "grad_allreduce_bytes_per_step": n_params * 4 if (world > 1 and a.mode == "train") else 0,
               "loss": float(loss), "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9}
        print(json.dumps(res), flush=True)
        if a.out:
            with open(a.out, "w") as fh:
                json.dump(res, fh, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
