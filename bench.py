"""bench.py -- the contract benchmark of the temporal MSDeformAttn hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype fp32|bf16] [--dist local|uniform]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One STEP = one encoder-layer temporal attention over one clip, forward + backward, at the DeVIS R50 T=6
YouTube-VIS shape (BASELINE.json configs[1]; SURVEY.md section 8d "unit U"): T=6 frames, levels
(45,80),(23,40),(12,20),(6,10) -> S=4820 rows per frame, 8 heads x 32 channels, one query per pixel,
4 current + 5x4x4 temporal points -> 96 taps per (query, head).  It is what the reference does with 12
MSDeformAttnFunction calls + 6 gather copies of value (modules/ms_deform_attn.py:435-460) and what this
repository does with one forward launch and one backward launch.

Rank 0 prints ONE JSON line:
  value         whole-job layer-clips per second with inputs resident in HBM (public autograd API, device events)
  us_fwd/us_bwd per-kernel durations (events around each launch): median and mean, steady state and cold L2
  roofline      contract roofline (HBM) of the dominant kernel, plus the on-chip resources that actually bind
  e2e           the same unit of work from pinned HOST buffers through the public API, every step paying the
                host->device copy of its operands and the device->host copy of its results: MEDIAN of 5 runs,
                all runs listed, the measured pure-copy ceiling of the same bytes next to it (e2e.bound)
  e2e.module    second end-to-end row through the MODULE API (TemporalMSDeformAttnEncoder): what a DeVIS caller
                moves -- query, src, grad_out in; out, grad_query, grad_src out -- projections on the device
  gpu_baseline  (N=1) the reference's own CUDA op (oracle/_ref, compiled unmodified) timed in the same process:
                its 12-call + 6-copy sequence and its single-call whole-clip form (SURVEY.md 8d ii, iii)
  cpu_baseline  (N=1) the reference's PyTorch CPU path on whole layer-clips, host cores stated
  also.train_trunk  (every N) trunk training step: fwd + bwd + DDP NCCL gradient all-reduce + clip + AdamW
Multi-GPU: clips are independent, so each rank works on its own clip (weak scaling, no collective on
the op path -- SURVEY.md section 8e).

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller: the output and the
five input gradients, as DIR/<name>.npy (float32; rank 0's clip).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output; see dump_outputs for the sampling that keeps the files under 64 MB.

`--impl reference` times the reference's CPU implementation of the same unit of work (the oracle's
PyTorch restatement of ms_deform_attn_core_pytorch + autograd, all host threads): W warm-up and K timed WHOLE
layer-clips (all 6 query frames, 12 calls + 6 gather copies), stopped early only by a wall-clock cap, with
the number of steps actually timed reported.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "temporal_msda_fwd_bwd_layer_clips_per_sec"
UNIT = "layer-clips/s"
WORKLOAD = "DeVIS R50 T=6 encoder layer-clip: S=4820, M=8, D=32, Lq=4820/frame, K=96 taps, fwd+bwd"
T_FRAMES, S_ROWS, HEADS, CH, K_TAPS = 6, 4820, 8, 32, 96
CLIP_NAMES = ("value", "loc_curr", "aw_curr", "loc_temporal", "aw_temporal")


def workload_config(dist, world, half_acc=False):
    """`config` of the JSON line -- identical for the GPU arm and the reference arm of the same workload"""
    return {"workload": WORKLOAD, "dist": dist, "taps": "boundary-safe",
            "l2_policy": "inputs larger than L2 (326 MB of operands per step vs 126 MB L2); no flush",
            "clips_per_rank_per_step": 1, "parallelism": f"clip-sharded x{world}, no collective",
            "grad_value_accumulation": "bf16 (opt-in flag)" if half_acc else "f32"}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe), through NVML
    (the same counters nvidia-smi prints) every 2 ms from a helper thread."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
               ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []          # (perf_counter, sm MHz, reason mask, watts)
        self.window = None         # (t0, t1): the timed region; samples outside it are dropped
        self.max_mhz = None
        self._stop = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(nvml_index(self.gpu))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # noqa: BLE001
            self.err = f"nvml unavailable: {exc}"
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                watts = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                self.samples.append((time.perf_counter(), mhz, mask, watts))
            except Exception as exc:  # noqa: BLE001
                self.err = str(exc)
                return
            time.sleep(0.002)

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=1)
        t0, t1 = self.window if self.window else (float("-inf"), float("inf"))
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        reasons = sorted({name for _, _, mask, _ in inside for name, bit in self.REASONS if mask & bit})
        out = {"sm_mhz": statistics.median(x[1] for x in inside) if inside else None, "sm_max_mhz": self.max_mhz,
               "samples": len(inside), "reasons": reasons,
               "power_w_max": max(x[3] for x in inside) if inside else None}
        if self.err:
            out["note"] = self.err
        return out


def nvml_index(local_rank):
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    if visible:
        parts = visible.split(",")
        if local_rank < len(parts) and parts[local_rank].strip().isdigit():
            return int(parts[local_rank])
    return local_rank


def bind_to_gpu_numa(local_rank):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, BEFORE any pinned buffer is
    allocated: first-touch then places the pinned pages on the GPU's own NUMA node, and the copy-issuing thread runs
    next to them.  Returns what was done, for the e2e record."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(nvml_index(local_rank))
        n_cpu = os.cpu_count() or 64
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpu + 63) // 64)
        local = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        info["_restore"] = allowed                    # the CPU baseline leg gets every host core back
        target = local & allowed
        info["gpu_local_cpus"] = len(local)
        info["allowed_cpus"] = len(allowed)
        if target and target != allowed:
            os.sched_setaffinity(0, target)
            info["bound"] = True
        info["cpus_used"] = len(target) if target else len(allowed)
        try:
            nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
            info["host_numa_nodes"] = len(nodes)
        except OSError:
            pass
    except Exception as exc:  # noqa: BLE001
        info["note"] = f"nvml affinity unavailable: {str(exc)[:80]}"
    return info


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_summary(kernel_key, field="dram_bytes_per_launch"):
    """per-launch counters of a kernel from the committed ncu --set full capture (profiles/ncu_summary.json)"""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as fh:
            return json.load(fh)[kernel_key][field]
    except Exception:
        return None


DUMP_MAX_ELEMS = 1 << 21        # per array: the six arrays of a step stay under 64 MB in float32


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` as out_dir/<name>.npy, float64 kept, anything else as float32.  A tensor of more than
    DUMP_MAX_ELEMS elements is replaced by DUMP_MAX_ELEMS of them, flattened: the flat indices are drawn without replacement
    from a generator seeded with 0 and sorted, so they depend only on the tensor's size and every run and every build
    writes the same elements."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        x = x.detach()
        if x.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(x.numel(), DUMP_MAX_ELEMS, replace=False))
            x = x.reshape(-1)[torch.from_numpy(idx).to(x.device)]
        x = x.cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (x.double() if x.dtype == torch.float64 else x.float()).numpy())


# ----------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the reference's PyTorch path on WHOLE layer-clips
# ----------------------------------------------------------------------------------------------------
class CpuLayerClip:
    """The reference's CPU path for one layer-clip: for each of the T query frames the current-frame call, the gather
    copy of the other frames' value and the temporal call (ms_deform_attn.py:435-460), with the oracle's PyTorch
    restatement of ms_deform_attn_core_pytorch (grid_sample forward, autograd backward), fp32, all host threads."""

    def __init__(self, dist, seed=0):
        import torch
        from devis_b200 import synthetic
        self.torch = torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.clip = synthetic.make_clip(dist=dist, seed=seed, device="cpu")
        self.shapes = torch.tensor(self.clip["shapes"])

    def step(self):
        from oracle import msda_torch
        torch, clip, shapes = self.torch, self.clip, self.shapes
        leaves = [clip[k].clone().requires_grad_(True) for k in CLIP_NAMES]
        v, lc, ac, lt, at = leaves
        t0 = time.perf_counter()
        frames_out = []
        for t in range(T_FRAMES):
            frames = clip["frame_table"][t]
            tshapes = shapes.repeat(len(frames), 1)
            cur = msda_torch.msda_forward_torch(v[t][None], shapes, lc[t][None], ac[t][None])
            stacked = v[frames].flatten(0, 1)[None]
            tmp = msda_torch.msda_forward_torch(stacked, tshapes, lt[t][None], at[t][None])
            frames_out.append(cur + tmp)
        torch.cat(frames_out, 0).backward(clip["grad_out"])
        return time.perf_counter() - t0

    SAMPLE = "whole layer-clips: 6 query frames x (current call + gather copy + temporal call), fwd + autograd bwd, fp32"


def run_reference(args, rank):
    """Rank 0 only (the other ranks exit without work).  Really runs `warmup` untimed and `steps` timed whole
    layer-clips; a wall-clock cap (--ref-wall-cap seconds, default 240) can end the timed loop early, and `steps`
    in the printed line is the number of steps actually timed."""
    if rank != 0:
        return
    t_wall = time.perf_counter()
    job = CpuLayerClip(args.dist)
    for _ in range(max(args.warmup, 1) if args.warmup else 0):
        job.step()
        if time.perf_counter() - t_wall > args.ref_wall_cap / 3:
            break
    times = []
    while len(times) < max(args.steps, 1):
        times.append(job.step())
        if time.perf_counter() - t_wall > args.ref_wall_cap:
            break
    per_clip = sum(times) / len(times)
    value = 1.0 / per_clip
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": per_clip * 1e3,
        "ms_per_step_median": statistics.median(times) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.dist, args.gpus),        # the SAME dictionary as the GPU arm's (the driver compares them)
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": job.cores, "kind": "port", "sample": job.SAMPLE},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_wall,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# host-fed pipeline (e2e)
# ----------------------------------------------------------------------------------------------------
class HostPipeline:
    """n_buf-deep host-fed pipeline around `step_fn`.

    Per step: ONE host->device copy of a pinned slab holding all operands, `step_fn` on views of the device slab,
    the results packed into a device slab, ONE device->host copy into a pinned slab.  Copies run on their own streams
    and overlap the kernels of neighbouring steps.  Timed on the device: the start event is recorded on the compute
    stream (the copy streams wait for it), the end event after the compute stream has waited for the last D2H."""

    def __init__(self, torch, dev, inputs, step_fn, n_buf=3):
        self.torch, self.dev, self.step_fn, self.n_buf = torch, dev, step_fn, n_buf
        self.specs, off = [], 0
        for x in inputs:
            n = x.numel() * x.element_size()
            self.specs.append((off, n, x.dtype, tuple(x.shape)))
            off += (n + 255) // 256 * 256
        self.in_bytes = off
        self.h2d_payload = sum(n for _, n, _, _ in self.specs)
        self.host_in = torch.empty(self.in_bytes, dtype=torch.uint8).pin_memory()
        for x, view in zip(inputs, self._views(self.host_in)):
            view.copy_(x.detach().cpu())
        self.dev_in = [torch.empty(self.in_bytes, dtype=torch.uint8, device=dev) for _ in range(n_buf)]
        self.dev_views = [self._views(d) for d in self.dev_in]
        self.out_specs = None
        self.dev_out, self.host_out = [None] * n_buf, [None] * n_buf
        self.s_h2d, self.s_d2h, self.s_comp = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
        mk = lambda: [torch.cuda.Event() for _ in range(n_buf)]
        self.ev_in, self.ev_in_free, self.ev_out, self.ev_out_free = mk(), mk(), mk(), mk()

    def _views(self, slab):
        return [slab[o:o + n].view(dt).view(shape) for o, n, dt, shape in self.specs]

    def _pack_setup(self, results):
        torch = self.torch
        self.out_specs, off = [], 0
        for r in results:
            n = r.numel() * r.element_size()
            self.out_specs.append((off, n, r.dtype, tuple(r.shape)))
            off += (n + 255) // 256 * 256
        self.out_bytes = off
        self.d2h_payload = sum(n for _, n, _, _ in self.out_specs)
        for b in range(self.n_buf):
            self.dev_out[b] = torch.empty(off, dtype=torch.uint8, device=self.dev)
            self.host_out[b] = torch.empty(off, dtype=torch.uint8).pin_memory()

    def run(self, n_steps):
        """returns device milliseconds for n_steps steps"""
        torch = self.torch
        s_h2d, s_d2h, s_comp = self.s_h2d, self.s_d2h, self.s_comp
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s_comp)
        s_h2d.wait_event(e0)
        s_d2h.wait_event(e0)
        for b in range(self.n_buf):
            self.ev_in_free[b].record(s_comp)
            self.ev_out_free[b].record(s_d2h)
        for i in range(n_steps):
            b = i % self.n_buf
            with torch.cuda.stream(s_h2d):
                s_h2d.wait_event(self.ev_in_free[b])
                self.dev_in[b].copy_(self.host_in, non_blocking=True)
                self.ev_in[b].record(s_h2d)
            s_comp.wait_event(self.ev_in[b])
            s_comp.wait_event(self.ev_out_free[b])           # the results that last used slot b have left the device
            results = self.step_fn(self.dev_views[b])
            if self.out_specs is None:
                self._pack_setup(results)
            for r, (o, n, dt, shape) in zip(results, self.out_specs):
                self.dev_out[b][o:o + n].view(dt).view(shape).copy_(r)
            self.ev_in_free[b].record(s_comp)
            self.ev_out[b].record(s_comp)
            with torch.cuda.stream(s_d2h):
                s_d2h.wait_event(self.ev_out[b])
                self.host_out[b].copy_(self.dev_out[b], non_blocking=True)
                self.ev_out_free[b].record(s_d2h)
        for b in range(self.n_buf):
            s_comp.wait_event(self.ev_out_free[b])
        e1.record(s_comp)
        torch.cuda.synchronize(self.dev)
        return e0.elapsed_time(e1)

    def copy_ceiling(self, n_steps):
        """the same slabs copied both ways with NO kernels in between: what the host link sustains for these bytes"""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.s_comp)
        self.s_h2d.wait_event(e0)
        self.s_d2h.wait_event(e0)
        for i in range(n_steps):
            b = i % self.n_buf
            with torch.cuda.stream(self.s_h2d):
                self.dev_in[b].copy_(self.host_in, non_blocking=True)
            with torch.cuda.stream(self.s_d2h):
                self.host_out[b].copy_(self.dev_out[b], non_blocking=True)
        self.s_comp.wait_stream(self.s_h2d)
        self.s_comp.wait_stream(self.s_d2h)
        e1.record(self.s_comp)
        torch.cuda.synchronize(self.dev)
        return e0.elapsed_time(e1)


def time_pipeline(pipe, steps_per_run, n_runs, barrier, reduce_max):
    """warm-up (grows the allocator pool and the output slabs), then n_runs timed runs; per-run ms/step as the max
    over ranks; then the pure-copy ceiling"""
    pipe.run(2 * pipe.n_buf)
    pipe.run(2 * pipe.n_buf)
    runs = []
    for _ in range(n_runs):
        barrier()
        runs.append(reduce_max(pipe.run(steps_per_run) / steps_per_run))
    pipe.copy_ceiling(pipe.n_buf)
    barrier()
    ceiling = reduce_max(pipe.copy_ceiling(steps_per_run) / steps_per_run)
    return runs, ceiling


def e2e_record(pipe, runs, ceiling_ms, world, steps_per_run, numa):
    ms = statistics.median(runs)
    bound = "pcie" if ms <= 1.25 * ceiling_ms else "pcie+compute"
    return {"value": world / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "statistic": "median of runs",
            "runs_ms_per_step": [round(x, 3) for x in runs], "steps_per_run": steps_per_run, "n_buffers": pipe.n_buf,
            "h2d_bytes_per_step": pipe.h2d_payload, "d2h_bytes_per_step": pipe.d2h_payload,
            "copies_per_step": {"h2d": 1, "d2h": 1},
            "bound": bound, "h2d_GBps": pipe.h2d_payload / ms / 1e6, "d2h_GBps": pipe.d2h_payload / ms / 1e6,
            "copy_ceiling_ms_per_step": ceiling_ms,
            "copy_ceiling_GBps_per_direction": pipe.h2d_payload / ceiling_ms / 1e6,
            "frac_of_copy_ceiling": ceiling_ms / ms, "numa": numa,
            "timing": "device events on the compute stream; copy streams fenced to it at both ends; max over ranks"}


# ----------------------------------------------------------------------------------------------------
# secondary legs
# ----------------------------------------------------------------------------------------------------
def median_us(torch, fn, iters, warmup=3, flush=None):
    """per-launch durations from events around each launch; flush: called before every timed launch (cold L2)"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        if flush is not None:
            flush()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    us = [a.elapsed_time(b) * 1e3 for a, b in evs]
    return {"median": statistics.median(us), "mean": statistics.mean(us), "min": min(us), "n": iters}


def gpu_baseline_leg(torch, clip, iters):
    """The reference's ORIGINAL CUDA op (oracle/_ref: /root/reference/src/models/ops/src compiled unmodified for sm_100a)
    timed in this process on this step's operands: (ii) the reference's layer-clip sequence -- 12 op calls + 6 gather
    copies + adds forward (ms_deform_attn.py:435-460), 12 backward calls + 6 copies + index_add backward -- and (iii) the
    reference kernel in the single-call whole-clip form (24 'levels', SURVEY.md section 7).  Checker-side code: it is
    a baseline next to the product's numbers, never part of the product path."""
    from oracle import ref_cuda_build
    ref = ref_cuda_build.load()
    if ref is None:
        return {"unavailable": "oracle/_ref not built"}
    dev = clip["value"].device
    T = clip["value"].shape[0]
    shapes = torch.tensor(clip["shapes"], device=dev)
    lsi_of = lambda s: torch.cat([s.new_zeros(1), s.prod(1).cumsum(0)[:-1]])
    lsi = lsi_of(shapes)
    tshapes = shapes.repeat(T - 1, 1)
    tlsi = lsi_of(tshapes)
    v = clip["value"].detach()
    lc = [clip["loc_curr"][t][None].detach().contiguous() for t in range(T)]
    ac = [clip["aw_curr"][t][None].detach().contiguous() for t in range(T)]
    lt = [clip["loc_temporal"][t][None].detach().contiguous() for t in range(T)]
    at = [clip["aw_temporal"][t][None].detach().contiguous() for t in range(T)]
    go = [clip["grad_out"][t][None].contiguous() for t in range(T)]
    idx = [torch.tensor(clip["frame_table"][t], device=dev) for t in range(T)]

    def seq_fwd():
        outs = []
        for t in range(T):
            cur = ref.ms_deform_attn_forward(v[t][None], shapes, lsi, lc[t], ac[t], 64)
            stacked = v[idx[t]].flatten(0, 1)[None]
            outs.append(cur + ref.ms_deform_attn_forward(stacked, tshapes, tlsi, lt[t], at[t], 64))
        return torch.cat(outs, 0)

    def seq_bwd():
        gv = torch.zeros_like(v)
        for t in range(T):
            g1 = ref.ms_deform_attn_backward(v[t][None], shapes, lsi, lc[t], ac[t], go[t], 64)
            stacked = v[idx[t]].flatten(0, 1)[None]
            g2 = ref.ms_deform_attn_backward(stacked, tshapes, tlsi, lt[t], at[t], go[t], 64)
            gv[t] += g1[0][0]
            gv.index_add_(0, idx[t], g2[0][0].view(T - 1, *v.shape[1:]))
        return gv

    out = {"what": "reference CUDA op (oracle/_ref, unmodified sources, sm_100a), same process, same operands, fp32"}
    f, b = median_us(torch, seq_fwd, iters), median_us(torch, seq_bwd, iters)
    out["sequence_12_calls_6_copies"] = {"us_fwd": round(f["median"], 1), "us_bwd": round(b["median"], 1),
                                         "us_fwd_bwd": round(f["median"] + b["median"], 1)}
    L, P = len(clip["shapes"]), clip["loc_curr"].shape[4]
    S, M, Lq = v.shape[1], v.shape[2], clip["loc_curr"].shape[1]
    big_shapes = shapes.repeat(T, 1)
    big_lsi = torch.cat([lsi + f_ * S for f_ in range(T)])
    loc = torch.zeros(1, T * Lq, M, T * L, P, 2, device=dev)
    aw = torch.zeros(1, T * Lq, M, T * L, P, device=dev)
    for t in range(T):
        q0 = slice(t * Lq, (t + 1) * Lq)
        loc[0, q0, :, t * L:(t + 1) * L] = clip["loc_curr"][t].detach()
        aw[0, q0, :, t * L:(t + 1) * L] = clip["aw_curr"][t].detach()
        for j, fr in enumerate(clip["frame_table"][t]):
            loc[0, q0, :, fr * L:(fr + 1) * L] = clip["loc_temporal"][t][:, :, j * L:(j + 1) * L].detach()
            aw[0, q0, :, fr * L:(fr + 1) * L] = clip["aw_temporal"][t][:, :, j * L:(j + 1) * L].detach()
    big_v, big_go = v.reshape(1, T * S, M, -1), clip["grad_out"].reshape(1, T * Lq, -1)
    f = median_us(torch, lambda: ref.ms_deform_attn_forward(big_v, big_shapes, big_lsi, loc, aw, 64), iters)
    b = median_us(torch, lambda: ref.ms_deform_attn_backward(big_v, big_shapes, big_lsi, loc, aw, big_go, 64), iters)
    out["single_call_whole_clip_form"] = {"us_fwd": round(f["median"], 1), "us_bwd": round(b["median"], 1),
                                          "us_fwd_bwd": round(f["median"] + b["median"], 1)}
    return out


def train_trunk_leg(torch, dist_mod, dev, rank, world, local_rank, steps=8, warmup=3, queries=10):
    """BASELINE.json configs[4] on the in-scope part of the model: the DeVIS transformer trunk (6 temporal encoder layers
    + 6 temporal decoder layers, devis_b200.DeVISTransformer) on synthetic R50 T=6 features, one clip per rank
    (main.py:85): forward + backward + DDP's bucketed NCCL gradient all-reduce (main.py:131) + clip_grad_norm_(0.1) +
    AdamW -- the body of train_one_epoch (engine.py:48-77).  The ONE collective DeVIS has."""
    from torch import nn
    from devis_b200 import DeVISTransformer, synthetic
    T, shapes_l, C = T_FRAMES, synthetic.DEVIS_SHAPES, 256
    torch.manual_seed(0)
    trunk = DeVISTransformer(d_model=C, num_frames=T, enc_n_temporal_points=4, dec_n_temporal_points=4).to(dev)
    query_embed = nn.Embedding(T * queries, 2 * C).to(dev)
    model = nn.ModuleDict({"trunk": trunk, "query_embed": query_embed})
    n_params = sum(p.numel() for p in model.parameters())
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    srcs = [torch.randn(T, C, h, w, device=dev, generator=g) for h, w in shapes_l]
    pos = [torch.randn(T, C, h, w, device=dev, generator=g) for h, w in shapes_l]
    masks = [torch.zeros(T, h, w, dtype=torch.bool, device=dev) for h, w in shapes_l]

    class Step(nn.Module):
        def __init__(self):
            super().__init__()
            self.m = model

        def forward(self, level0):                    # DDP wants at least one tensor argument
            hs, _, memories, *_ = self.m["trunk"]([level0] + srcs[1:], masks, pos, self.m["query_embed"].weight)
            return hs, memories

    net = Step()
    ddp = None
    if world > 1:
        ddp = nn.parallel.DistributedDataParallel(net, device_ids=[local_rank], find_unused_parameters=True)
    opt = torch.optim.AdamW(net.parameters(), lr=2e-4, weight_decay=1e-4)

    def step(sync=True):
        opt.zero_grad(set_to_none=True)
        runner = ddp if ddp is not None else net
        if ddp is not None and not sync:
            with ddp.no_sync():
                hs, memories = runner(srcs[0])
                loss = hs[-1].float().square().mean() + 1e-3 * sum(m.float().square().mean() for m in memories)
                loss.backward()
        else:
            hs, memories = runner(srcs[0])
            loss = hs[-1].float().square().mean() + 1e-3 * sum(m.float().square().mean() for m in memories)
            loss.backward()
        torch.nn.utils.clip_grad_norm_(net.parameters(), 0.1)
        opt.step()

    def timed(sync):
        for _ in range(warmup):
            step(sync)
        if world > 1:
            dist_mod.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(sync)
        e1.record()
        if world > 1:
            dist_mod.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    ms = timed(True)
    res = {"workload": f"DeVIS transformer trunk training step: 6 enc + 6 dec layers, T=6, S=4820, {queries} queries/frame, fp32, "
                       "fwd + bwd + DDP gradient all-reduce + clip_grad_norm + AdamW, one clip per rank, synthetic features",
           "ms_per_step": ms, "clips_per_sec": world / (ms * 1e-3), "steps": steps, "warmup": warmup, "params": n_params,
           "allreduce_bytes_per_step": n_params * 4 if world > 1 else 0}
    if world > 1:
        res["ms_per_step_without_allreduce"] = timed(False)
        flat = torch.zeros(n_params, device=dev)
        for _ in range(3):
            dist_mod.all_reduce(flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            dist_mod.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        res["allreduce_ms_standalone"] = e0.elapsed_time(e1) / 10
        res["allreduce_exposed_ms"] = max(0.0, ms - res["ms_per_step_without_allreduce"])
    del opt, net, ddp, model, trunk
    return res


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    numa = bind_to_gpu_numa(local_rank)          # before torch allocates anything pinned
    restore_cpus = numa.pop("_restore", None)
    import torch
    import torch.distributed as dist_mod
    from devis_b200 import _lib, clip_geometry, synthetic, temporal_ms_deform_attn

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist_mod.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16}[args.dtype]
    half_acc = args.bf16_accumulate and dtype == torch.bfloat16
    if half_acc:
        from devis_b200 import MultiScaleDeformableAttention as MSDA
        MSDA.set_bf16_grad_value_accumulation(True)
    bwd_flags = _lib.FLAG_BF16_GRAD_VALUE if half_acc else 0
    clip = synthetic.make_clip(dist=args.dist, dtype=dtype, seed=100 + rank, device=dev)
    geom = clip_geometry.ClipGeometry(clip["shapes"], T_FRAMES, clip["frame_table"])
    order = geom.tile_order(dev, 8, 8)
    leaves = [clip[k].requires_grad_(True) for k in CLIP_NAMES]
    gout = clip["grad_out"]

    def step():
        for x in leaves:
            x.grad = None
        out = temporal_ms_deform_attn(*leaves, geom, order)
        out.backward(gout)
        return out

    def barrier():
        if world > 1:
            dist_mod.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
            return float(t.item())
        return float(x)

    # ---- headline: K steps, device resident, public autograd API
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()        # started before the warm-up so that NVML's slow first calls are over by the timed region
    for _ in range(warmup):
        step()
    barrier()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_region0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    barrier()
    sampler.window = (t_region0, time.perf_counter())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": out, **{"grad_" + k: x.grad for k, x in zip(CLIP_NAMES, leaves)}})
    ms_total = reduce_max(e0.elapsed_time(e1))
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist_mod.all_reduce(lt, op=dist_mod.ReduceOp.SUM)
        launches = int(lt.item())
    ms_step = ms_total / args.steps
    value = world / (ms_step * 1e-3)

    # ---- per-kernel durations (events around each launch, same stream, same operands) for the roofline: steady state
    # (operands of one step are 326 MB >> 126 MB L2, so "steady" already streams them from HBM; value and grad_value
    # stay L2-resident as in the real model) and COLD L2 (a 512 MB fill before every timed launch evicts everything)
    from benchmarks.sweep import RawClip
    raw = RawClip({k: (v.detach() if hasattr(v, "detach") else v) for k, v in clip.items()}, order)
    n_k = max(20, min(args.steps, 100))
    k_fwd = median_us(torch, raw.fwd, n_k)
    k_bwd = median_us(torch, lambda: raw.bwd(bwd_flags), n_k)
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    flush = lambda: flush_buf.fill_(1)
    n_c = max(10, min(args.steps, 30))
    c_fwd = median_us(torch, raw.fwd, n_c, flush=flush)
    c_bwd = median_us(torch, lambda: raw.bwd(bwd_flags), n_c, flush=flush)
    del flush_buf
    us_fwd, us_bwd = k_fwd["median"], k_bwd["median"]
    elem = clip["value"].element_size()
    bytes_f, bytes_b = synthetic.algorithmic_bytes(T_FRAMES, S_ROWS, HEADS, CH, S_ROWS, K_TAPS, elem=elem)
    peak, peak_src = measured_peak_gbs()

    # ---- secondary rows (N = 1 only, not part of the headline): the same unit of work with bf16 value, and the
    # fused-prologue form the encoder module runs (raw Linear outputs in, softmax + location arithmetic in the kernels)
    extra = {}
    if world == 1 and dtype == torch.float32 and not args.only_headline:
        try:
            from benchmarks.sweep import time_us
            clip16 = synthetic.make_clip(dist=args.dist, dtype=torch.bfloat16, seed=100 + rank, device=dev)
            raw16 = RawClip(clip16, order)
            f16, b16 = time_us(raw16.fwd, 20), time_us(raw16.bwd, 20)
            extra["bf16_value"] = {"us_fwd": round(f16, 1), "us_bwd": round(b16, 1),
                                   "layer_clips_per_sec": round(1e6 / (f16 + b16), 1)}
            del clip16, raw16
            from devis_b200 import TemporalMSDeformAttnFusedFunction
            g = torch.Generator(device=dev).manual_seed(7)
            nl, wt = len(clip["shapes"]), T_FRAMES - 1
            ref = synthetic.pixel_reference_points(clip["shapes"], T_FRAMES, dev)
            shp = (T_FRAMES, S_ROWS, HEADS)
            ops = [clip["value"].detach().clone().requires_grad_(True), ref,
                   (2.0 * torch.randn(*shp, nl, 4, 2, generator=g, device=dev)).requires_grad_(True),
                   torch.randn(*shp, nl * 4, generator=g, device=dev).requires_grad_(True),
                   (2.0 * torch.randn(*shp, wt * nl, 4, 2, generator=g, device=dev)).requires_grad_(True),
                   torch.randn(*shp, wt * nl * 4, generator=g, device=dev).requires_grad_(True)]

            def fused_fwd():
                with torch.no_grad():
                    TemporalMSDeformAttnFusedFunction.apply(*ops, geom, order)

            def fused_fwd_bwd():
                for x in ops:
                    x.grad = None
                TemporalMSDeformAttnFusedFunction.apply(*ops, geom, order).backward(gout)

            extra["fused_prologue_f32"] = {"us_fwd": round(time_us(fused_fwd, 20), 1),
                                           "us_fwd_bwd": round(time_us(fused_fwd_bwd, 20), 1)}
            del ops
        except Exception as exc:   # noqa: BLE001 -- secondary rows must never take the headline down
            extra["error"] = str(exc)[:200]
    fwd_kernel = "msda_fwdv_kernel" if dtype == torch.float32 else "msda_fwd8v_kernel"   # what the launcher picks at D = 32

    # ---- the on-chip resources that actually bind (DESIGN.md 3.6): every tap gathers 4 value rows through the SM's
    # L1 data pipe (128 B/clk/SM), every live corner leaves the SM as one row reduction (cycles per 128-B row measured
    # by benchmarks/micro/tma_reduce.cu, recorded in profiles/ncu_summary.json).  Counted from this step's own taps.
    def live_corners():
        n = 0
        for loc, reps in ((clip["loc_curr"], 1), (clip["loc_temporal"], T_FRAMES - 1)):
            size = torch.tensor([[w, h] for h, w in clip["shapes"]], device=dev, dtype=torch.float32).repeat(reps, 1)
            pix = loc.detach().float() * size[None, None, None, :, None, :] - 0.5
            x, y = pix[..., 0], pix[..., 1]
            wl, hl = size[:, 0][None, None, None, :, None], size[:, 1][None, None, None, :, None]
            inr = (x > -1) & (y > -1) & (x < wl) & (y < hl)
            x0, y0 = torch.floor(x), torch.floor(y)
            lft, rgt, top, bot = x0 >= 0, x0 + 1 <= wl - 1, y0 >= 0, y0 + 1 <= hl - 1
            n += int(((inr & top & lft).sum() + (inr & top & rgt).sum() + (inr & bot & lft).sum() + (inr & bot & rgt).sum()).item())
        return n

    props = torch.cuda.get_device_properties(dev)
    sm_count = props.multi_processor_count
    sm_mhz = float((clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or props.clock_rate / 1e3)
    sm_hz = 1e6 * sm_mhz
    cycles_per_row = float(ncu_summary("microbench", "reduction_cycles_per_128B_row") or 5.16)
    l1_bytes_per_clk = float(ncu_summary("microbench", "l1_data_pipe_bytes_per_clk_per_sm") or 128)
    row_bytes = CH * elem
    gather_bytes = T_FRAMES * S_ROWS * HEADS * K_TAPS * 4 * row_bytes
    l1_peak = sm_count * l1_bytes_per_clk * sm_hz         # bytes per second through the L1/shared data pipes
    red_rows = live_corners()
    on_chip = {
        "fwd_l1_gather": {"bytes": gather_bytes, "achieved_TBps": gather_bytes / us_fwd / 1e6, "peak_TBps": l1_peak / 1e12,
                          "frac": gather_bytes / (us_fwd * 1e-6) / l1_peak,
                          # since round 2 the forward gathers only the live corners; the figure above keeps round 1's
                          # definition (all 4 corners of every tap) so that rounds compare
                          "live_row_bytes": red_rows * row_bytes,
                          # one 128-bit gather instruction covers 4 rows (fp32, 8 lanes per row) or 8 (bf16, 4 lanes)
                          "gather_instructions_per_sm": T_FRAMES * S_ROWS * HEADS * K_TAPS * 4 // (4 if elem == 4 else 8) // sm_count,
                          "cycles_per_gather_instruction": us_fwd * 1e-6 * sm_hz /
                                                           (T_FRAMES * S_ROWS * HEADS * K_TAPS * 4 / (4 if elem == 4 else 8) / sm_count)},
        "bwd_reduction_egress": {"row_reductions": red_rows, "cycles_per_row": cycles_per_row,
                                 "busy_frac": red_rows / sm_count * cycles_per_row / (us_bwd * 1e-6 * sm_hz)},
        "sm_count": sm_count, "sm_mhz": sm_mhz,
        "note": "gathered value rows through the SMs' L1 data pipes (bytes/clk/SM at the sampled SM clock) and grad_value row "
                "reductions leaving the SMs (cycles per 128-B row measured); these, not HBM, bound the kernels",
    }

    # ---- e2e: public autograd API driven from pinned HOST buffers
    e2e_steps = max(6, min(args.steps, 20))

    def op_step(views):
        ins = [v.detach().requires_grad_(True) for v in views[:5]]
        out = temporal_ms_deform_attn(*ins, geom, order)
        out.backward(views[5])
        return [out.detach()] + [x.grad for x in ins]

    pipe = HostPipeline(torch, dev, [x.detach() for x in leaves] + [gout], op_step, n_buf=3)
    runs, ceiling = time_pipeline(pipe, e2e_steps, 5, barrier, reduce_max)
    e2e = e2e_record(pipe, runs, ceiling, world, e2e_steps, numa)
    del pipe

    # ---- e2e through the MODULE API: what a DeVIS caller moves (query, src, grad_out in; out and the two input
    # gradients back); value / offset / weight projections and the fused-prologue kernels run on the device
    if not args.only_headline:
        try:
            from devis_b200 import TemporalMSDeformAttnEncoder
            torch.manual_seed(11)
            enc = TemporalMSDeformAttnEncoder(n_frames=T_FRAMES, d_model=HEADS * CH, n_levels=4, t_window=T_FRAMES - 1,
                                              n_heads=HEADS, n_curr_points=4, n_temporal_points=4).to(dev)
            with torch.no_grad():
                for lin in (enc.sampling_offsets, enc.temporal_sampling_offsets, enc.attention_weights,
                            enc.temporal_attention_weights):
                    lin.weight.normal_(0, 0.02)
            m_ref = synthetic.pixel_reference_points(clip["shapes"], T_FRAMES, dev)
            m_shapes = torch.tensor(clip["shapes"], device=dev)
            m_lsi = torch.tensor(synthetic.level_start_index(clip["shapes"]), device=dev)
            m_tshapes = m_shapes.repeat(T_FRAMES - 1, 1)
            m_tlsi = torch.cat([m_tshapes.new_zeros(1), m_tshapes.prod(1).cumsum(0)[:-1]])
            m_offs = [torch.tensor([d for d in range(-t, T_FRAMES - t) if d != 0], device=dev) for t in range(T_FRAMES)]
            gm = torch.Generator(device=dev).manual_seed(5 + rank)
            m_in = [torch.randn(T_FRAMES, S_ROWS, HEADS * CH, generator=gm, device=dev) for _ in range(3)]

            def module_step(views):
                q = views[0].detach().requires_grad_(True)
                x = views[1].detach().requires_grad_(True)
                for p in enc.parameters():
                    p.grad = None
                out, _ = enc(q, m_ref, x, (m_shapes, m_tshapes), (m_lsi, m_tlsi), m_offs)
                out.backward(views[2])
                return [out.detach(), q.grad, x.grad]

            mpipe = HostPipeline(torch, dev, m_in, module_step, n_buf=3)
            fam0 = _lib.kernel_launches(_lib.KERNEL_FUSED_FWD)
            m_steps = max(6, min(args.steps, 12))
            m_runs, m_ceiling = time_pipeline(mpipe, m_steps, 5, barrier, reduce_max)
            rec = e2e_record(mpipe, m_runs, m_ceiling, world, m_steps, numa)
            rec["api"] = ("TemporalMSDeformAttnEncoder.forward/backward (d_model 256, fp32 cuBLAS projections, fused-prologue "
                          "kernels): H2D query + src + grad_out, D2H out + grad_query + grad_src")
            rec["fused_kernel_launches"] = _lib.kernel_launches(_lib.KERNEL_FUSED_FWD) - fam0
            rec["bound"] = "pcie" if rec["ms_per_step"] <= 1.25 * m_ceiling else "compute (projection GEMMs + attention kernels)"
            e2e["module"] = rec
            del mpipe, enc
        except Exception as exc:   # noqa: BLE001
            e2e["module"] = {"error": str(exc)[:300]}

    # ---- GPU baseline (N = 1): the reference's own CUDA op in this process
    gpu_base = None
    if world == 1 and dtype == torch.float32 and not args.only_headline and not args.no_gpu_baseline:
        try:
            gpu_base = gpu_baseline_leg(torch, clip, 20)
            if "sequence_12_calls_6_copies" in gpu_base:
                ours_us = us_fwd + us_bwd
                gpu_base["ours_us_fwd_bwd"] = round(ours_us, 1)
                gpu_base["speedup_vs_sequence"] = round(gpu_base["sequence_12_calls_6_copies"]["us_fwd_bwd"] / ours_us, 2)
                gpu_base["speedup_vs_single_call"] = round(gpu_base["single_call_whole_clip_form"]["us_fwd_bwd"] / ours_us, 2)
        except Exception as exc:   # noqa: BLE001
            gpu_base = {"error": str(exc)[:300]}

    # ---- training config (every N): the one collective DeVIS has
    if not args.only_headline and not args.no_train_trunk and dtype == torch.float32:
        try:
            del raw
            torch.cuda.empty_cache()
            extra["train_trunk"] = train_trunk_leg(torch, dist_mod, dev, rank, world, local_rank)
        except Exception as exc:   # noqa: BLE001
            import traceback
            extra["train_trunk"] = {"error": str(exc)[:300], "where": traceback.format_exc()[-700:]}

    # ---- BASELINE.json config 5 on the WHOLE model (every N): ResNet-50 + transformer + heads + mask head, forward + backward +
    #      DDP gradient all-reduce + clip_grad_norm + AdamW, one synthetic clip per rank (benchmarks/devis_r50_inference.py)
    if not args.only_headline and not args.no_train_trunk and dtype == torch.float32:
        try:
            torch.cuda.empty_cache()
            from torch import nn as _nn
            from benchmarks import devis_r50_inference
            wrap = (lambda net: _nn.parallel.DistributedDataParallel(net, device_ids=[local_rank], find_unused_parameters=True)) \
                if world > 1 else None
            r = devis_r50_inference.run_train("ours", iters=6, tf32=False, ddp=wrap)
            ms = float(r["ours"]["ms_per_step"])
            if world > 1:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
                ms = float(t.item())
            extra["full_model_train"] = {"config": r["config"], "ms_per_step": ms, "clips_per_sec": world / (ms * 1e-3),
                                         "params": r["ours"]["trainable_params"],
                                         "allreduce_bytes_per_step": r["ours"]["trainable_params"] * 4 if world > 1 else 0,
                                         "note": "max over ranks; at N = 1 the same step on the reference's ops takes 1.86x as long "
                                                 "(profiles/r2ae_devis_r50_train_step.json)"}
        except Exception as exc:   # noqa: BLE001
            extra["full_model_train"] = {"error": str(exc)[:300]}

    # ---- BASELINE.json config 3: DeVIS R50 T=6 full-model inference (rank 0, one GPU's rate; benchmarks/devis_r50_inference.py)
    if rank == 0 and not args.only_headline and dtype == torch.float32:
        try:
            torch.cuda.empty_cache()
            from benchmarks import devis_r50_inference
            full = {}
            for mode in ("off", "on"):
                r = devis_r50_inference.run("both", iters=10, breakdown=False, tf32=mode == "on")
                full["tf32_" + mode] = {"ours_ms_per_clip": r.get("ours", {}).get("ms_per_clip_median"),
                                        "ours_clips_per_sec": r.get("ours", {}).get("clips_per_sec"),
                                        "reference_ops_ms_per_clip": r.get("reference_ops", {}).get("ms_per_clip_median"),
                                        "speedup": r.get("speedup"), "config": r.get("config")}
                if "error" in r.get("reference_ops", {}):
                    full["tf32_" + mode]["reference_ops_error"] = r["reference_ops"]["error"]
            full["what"] = ("whole model on one GPU: torchvision ResNet-50 + DeVIS transformer (6 + 6 layers) + box heads + top-k + "
                            "mask head; 'reference_ops' = same weights with the reference's attention loop / CUDA op and "
                            "torchvision's deform_conv2d")
            extra["full_model_inference"] = full
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
        except Exception as exc:   # noqa: BLE001
            extra["full_model_inference"] = {"error": str(exc)[:300]}

    if rank == 0:
        bwd_kernel = "msda_bwd_kernel"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if dtype == torch.float32 else "bf16", "data": "synthetic",
            "config": workload_config(args.dist, world, half_acc),
            "us_fwd": us_fwd, "us_bwd": us_bwd,
            "kernel_us": {"fwd": {k: round(v, 1) for k, v in k_fwd.items()}, "bwd": {k: round(v, 1) for k, v in k_bwd.items()},
                          "fwd_cold_l2": {k: round(v, 1) for k, v in c_fwd.items()},
                          "bwd_cold_l2": {k: round(v, 1) for k, v in c_bwd.items()},
                          "note": "events around each launch; us_fwd / us_bwd are the steady-state medians; cold = 512 MB "
                                  "L2 flush before every timed launch"},
            "roofline": {"bound": "hbm", "kernel": bwd_kernel, "achieved": bytes_b / us_bwd / 1e3, "peak": peak,
                         "unit": "GB/s", "frac": bytes_b / us_bwd / 1e3 / peak, "traffic": ncu_summary(bwd_kernel),
                         "algorithmic_bytes": bytes_b, "peak_source": peak_src,
                         "fwd": {"kernel": fwd_kernel, "achieved": bytes_f / us_fwd / 1e3,
                                 "frac": bytes_f / us_fwd / 1e3 / peak, "algorithmic_bytes": bytes_f,
                                 "traffic": ncu_summary(fwd_kernel)},
                         "fwd_bwd": {"achieved": (bytes_f + bytes_b) / (us_fwd + us_bwd) / 1e3,
                                     "frac": (bytes_f + bytes_b) / (us_fwd + us_bwd) / 1e3 / peak},
                         "cold_l2": {"frac_bwd": bytes_b / c_bwd["median"] / 1e3 / peak,
                                     "frac_fwd": bytes_f / c_fwd["median"] / 1e3 / peak},
                         "note": "contract roofline (HBM). Binding resources measured with ncu + microbenchmarks: forward = SM "
                                 "L1/shared data pipe, backward = SM reduction egress together with the data pipe; "
                                 "DESIGN.md 3.6, profiles/README.md",
                         "on_chip": on_chip},
            "e2e": e2e,
            "gpu_launches": launches, "clocks": clocks,
        }
        if gpu_base is not None:
            line["gpu_baseline"] = gpu_base
        if extra:
            line["also"] = extra
        if world == 1 and not args.no_cpu_baseline and not args.only_headline:
            if restore_cpus:
                os.sched_setaffinity(0, restore_cpus)
            job = CpuLayerClip(args.dist)
            job.step()                                     # warm-up (thread pool, allocator)
            t0, times = time.perf_counter(), []
            while len(times) < 8 and (time.perf_counter() - t0 < 16 or not times):
                times.append(job.step())
            sec = sum(times) / len(times)
            line["cpu_baseline"] = {"value": 1.0 / sec, "unit": UNIT, "cores": job.cores, "kind": "port",
                                    "sample": f"{len(times)} {job.SAMPLE}; {sec:.2f} s per layer-clip after 1 warm-up"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist_mod.barrier()
        dist_mod.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--dist", default="local", choices=["local", "uniform"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-train-trunk", action="store_true")
    ap.add_argument("--only-headline", action="store_true", help="value, kernels, roofline and the op-level e2e only")
    ap.add_argument("--ref-wall-cap", type=float, default=240.0,
                    help="--impl reference: stop timing after this many seconds of wall clock (steps reported honestly)")
    ap.add_argument("--bf16-accumulate", action="store_true",
                    help="with --dtype bf16: accumulate grad_value in bf16 (DEVIS_MSDA_FLAG_BF16_GRAD_VALUE, opt-in)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the output and the input gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
