"""tests/golden/make_dcn_offset_groups.py -- generates the dcn_og_*.npz fixtures in this directory.

torchvision.ops.deform_conv2d on the CPU in float64, forward and autograd backward, with offset groups (offset of
2 * G * kh * kw channels, mask of G * kh * kw).  Same keys and `cfg` = [stride, padding, dilation, use_mask] as the
dcn_*.npz fixtures of make_golden.py; G is offset.shape[1] // (2 * kh * kw).  Needs only torch and torchvision.

Usage:  python tests/golden/make_dcn_offset_groups.py
"""
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

# name: (N, Cin, Cout, H, W, k, stride, pad, dil, mask, offset scale, offset groups)
CASES = {
    "dcn_og_g2_c8": (2, 8, 5, 7, 9, 3, 1, 1, 1, True, 1.5, 2),             # Cg = 4: vector path, 4 lanes
    "dcn_og_g4_c32": (1, 32, 6, 6, 8, 3, 1, 1, 1, True, 3.0, 4),           # Cg = 8: vector path, taps leaving the map
    "dcn_og_g2_c6": (1, 6, 4, 5, 6, 3, 1, 1, 1, True, 1.0, 2),             # Cg = 3: scalar path, 8 lanes
    "dcn_og_g2_c66": (1, 66, 3, 4, 5, 3, 1, 1, 1, True, 1.0, 2),           # Cg = 33: scalar path, 32 lanes
    "dcn_og_g6_c6_s2_nomask": (2, 6, 4, 9, 8, 3, 2, 2, 2, False, 1.0, 6),  # G = C, Cg = 1; stride / dilation, no mask
    # lane-group fused kernels at G > 1 (Cout in {1, 2, 4, 8, 16}, Cg % 4 == 0)
    "dcn_og_fused_c12_o2_k1_g3": (1, 12, 2, 5, 5, 1, 1, 0, 1, True, 0.7, 3),     # 1 x 1 kernel
    "dcn_og_fused_c32_o16_g2": (2, 32, 16, 6, 7, 3, 1, 1, 1, True, 1.5, 2),      # the 90x160 layer of the mask head
    "dcn_og_fused_c16_o1_g4": (2, 16, 1, 6, 5, 3, 1, 1, 1, True, 1.0, 4),        # out_lay
    "dcn_og_fused_c64_o8_s2_g2": (2, 64, 8, 9, 8, 3, 2, 2, 2, False, 1.0, 2),    # 8 lanes; stride / dilation, no mask
    "dcn_og_fused_c72_o4_g2": (1, 72, 4, 5, 6, 3, 1, 1, 1, True, 3.0, 2),        # Cg = 36: ragged last channel block
    # layers whose G = 1 form (constant bank / tensor cores) does not serve G > 1: im2col
    "dcn_og_c72_o32_g2": (1, 72, 32, 5, 6, 3, 1, 1, 1, True, 3.0, 2),
    "dcn_og_c264_o4_g4": (1, 264, 4, 3, 4, 3, 1, 1, 1, True, 1.0, 4),           # Cg = 66: scalar path
}


def reference(x, offset, weight, bias, mask, cfg):
    """torchvision's CPU operator: out and the gradients of (x, offset, weight, bias[, mask]) for grad_out gout"""
    from torchvision.ops import deform_conv2d
    st, pd, dl, _ = [int(v) for v in cfg]
    leaves = [t.clone().requires_grad_(True) for t in (x, offset, weight, bias)]
    if mask is not None:
        leaves.append(mask.clone().requires_grad_(True))
    out = deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], stride=st, padding=pd, dilation=dl,
                        mask=leaves[4] if mask is not None else None)
    return out, leaves


def main():
    gen = torch.Generator().manual_seed(13)
    rn = lambda *s: torch.randn(*s, generator=gen, dtype=torch.float64)
    for name, (n, cin, cout, h, w, k, st, pd, dl, use_mask, osc, og) in CASES.items():
        ho = (h + 2 * pd - (dl * (k - 1) + 1)) // st + 1
        wo = (w + 2 * pd - (dl * (k - 1) + 1)) // st + 1
        x, wt, b = rn(n, cin, h, w), rn(cout, cin, k, k), rn(cout)
        off = osc * rn(n, 2 * og * k * k, ho, wo)
        m = torch.rand(n, og * k * k, ho, wo, generator=gen, dtype=torch.float64) * 2 if use_mask else None
        cfg = np.array([st, pd, dl, int(use_mask)])
        out, leaves = reference(x, off, wt, b, m, cfg)
        gout = rn(*out.shape)
        out.backward(gout)
        arrays = dict(x=x, offset=off, weight=wt, bias=b, gout=gout, out=out, gx=leaves[0].grad, goffset=leaves[1].grad,
                      gweight=leaves[2].grad, gbias=leaves[3].grad, cfg=cfg)
        if use_mask:
            arrays.update(mask=m, gmask=leaves[4].grad)
        arrays = {key: v.detach().numpy() if isinstance(v, torch.Tensor) else np.asarray(v) for key, v in arrays.items()}
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
