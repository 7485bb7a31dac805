import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200.deform_conv import deform_conv2d
from torch.profiler import ProfilerActivity, profile
torch.backends.cuda.matmul.allow_tf32 = False
g = torch.Generator(device="cuda").manual_seed(0)
rn = lambda *s: torch.randn(*s, generator=g, device="cuda")
for name, cin, cout, h, w in (("lay5", 32, 16, 90, 160), ("lay4", 72, 32, 45, 80), ("out_lay", 16, 1, 90, 160), ("lay1", 264, 264, 12, 20)):
    n = 60
    x = rn(n, cin, h, w).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    wt = (rn(cout, cin, 3, 3) / (3 * cin ** 0.5)).requires_grad_(True)
    b = rn(cout).requires_grad_(True)
    off = (1.5 * rn(n, 18, h, w)).requires_grad_(True)
    m = (2 * torch.sigmoid(rn(n, 9, h, w))).requires_grad_(True)
    gout = rn(n, cout, h, w)
    def step():
        out = deform_conv2d(x, off, wt, b, padding=1, mask=m)
        out.backward(gout)
        for t in (x, wt, b, off, m):
            t.grad = None
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            step()
        torch.cuda.synchronize()
    print("=====", name)
    print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12, max_name_column_width=70))
