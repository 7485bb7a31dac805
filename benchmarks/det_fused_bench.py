import json, os, sys, statistics, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import TemporalMSDeformAttnEncoder, synthetic, clip_geometry, MultiScaleDeformableAttention as MSDA
torch.manual_seed(0)
T, C = 6, 256
shapes_l = synthetic.DEVIS_SHAPES
S = sum(h * w for h, w in shapes_l)
mod = TemporalMSDeformAttnEncoder(T, C, 4, T - 1, 8, 4, 4).cuda()
with torch.no_grad():
    for lin in (mod.sampling_offsets, mod.temporal_sampling_offsets, mod.attention_weights, mod.temporal_attention_weights):
        lin.weight.normal_(0, 0.02)
shapes, lsi = clip_geometry.pyramid_tensors(shapes_l, "cuda")
tshapes = shapes.repeat(T - 1, 1)
tlsi = torch.cat([tshapes.new_zeros(1), tshapes.prod(1).cumsum(0)[:-1]])
offs = [torch.tensor([d for d in range(-t, T - t) if d != 0], device="cuda") for t in range(T)]
ref = synthetic.pixel_reference_points(shapes_l, T, "cuda")
q = torch.randn(T, S, C, device="cuda", requires_grad=True)
x = torch.randn(T, S, C, device="cuda", requires_grad=True)
gout = torch.randn(T, S, C, device="cuda")
def step():
    out, _ = mod(q, ref, x, (shapes, tshapes), (lsi, tlsi), offs)
    out.backward(gout)
def med(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return round(statistics.median(a.elapsed_time(b) for a, b in ev), 3)
res = {}
for det in (False, True):
    MSDA.set_deterministic(det)
    for fused in (True, False):
        mod.fuse_prologue = fused
        res[f"det={det} fused={fused} fwd+bwd ms"] = med(step)
MSDA.set_deterministic(False)
print(json.dumps(res))
