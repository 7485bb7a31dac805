import os, sys, json, statistics, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from conftest import nmax
from devis_b200 import _lib, deform_conv
from devis_b200.deform_conv import IGemmDeformConv2dFunction, deform_conv2d
torch.backends.cuda.matmul.allow_tf32 = False
def med(fn, iters=30):
    for _ in range(5): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return round(statistics.median(a.elapsed_time(b) for a, b in ev) * 1e3, 1)
for c, cout, (h, w), n in [(72, 32, (45, 80), 60), (32, 16, (90, 160), 60), (16, 4, (90, 160), 60)]:
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, c, h, w, device="cuda", generator=gen).contiguous(memory_format=torch.channels_last)
    off = 1.5 * torch.randn(n, 18, h, w, device="cuda", generator=gen)
    msk = torch.rand(n, 9, h, w, device="cuda", generator=gen)
    wt = torch.randn(cout, c, 3, 3, device="cuda", generator=gen) / (9 * c) ** 0.5
    b = torch.randn(cout, device="cuda", generator=gen)
    ok = bool(_lib.load().devis_dcn_igemm_supported(c, cout, 3, 3, _lib.F32))
    row = {"igemm_supported": ok}
    with torch.no_grad():
        want = deform_conv2d(x, off, wt, b, padding=1, mask=msk)
        row["current_us"] = med(lambda: deform_conv2d(x, off, wt, b, padding=1, mask=msk))
        if ok:
            got = IGemmDeformConv2dFunction.apply(x, off, wt, b, msk, (1, 1), (1, 1), (1, 1))
            row["err_vs_current"] = nmax(got.cpu().numpy(), want.cpu().numpy())
            row["igemm_3xtf32_us"] = med(lambda: IGemmDeformConv2dFunction.apply(x, off, wt, b, msk, (1, 1), (1, 1), (1, 1)))
            torch.backends.cuda.matmul.allow_tf32 = True
            row["igemm_tf32_us"] = med(lambda: IGemmDeformConv2dFunction.apply(x, off, wt, b, msk, (1, 1), (1, 1), (1, 1)))
            torch.backends.cuda.matmul.allow_tf32 = False
    print(f"{c}->{cout} @{h}x{w} x{n}", json.dumps(row), flush=True)
