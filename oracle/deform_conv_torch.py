"""ORACLE -- test infrastructure only (never imported by devis_b200/).

Pure-PyTorch, differentiable restatement of torchvision's modulated deformable convolution, the third-party operator
DeVIS's mask head calls (src/models/deformable_segmentation.py:265; torchvision pinned at 0.12 by docs/INSTALL.md:9,
0.26 in this image).  Follows torchvision/csrc/ops/cpu/deform_conv2d_kernel.cpp:
  bilinear_interpolate   : the sample is 0 unless -1 < h < H and -1 < w < W; corners outside the map contribute 0 and
                           are never read (a non-finite pixel only reaches the taps whose live corners include it)
  deformable_im2col      : sample point = (ho*stride - pad + ky*dil + offset[2k], wo*stride - pad + kx*dil + offset[2k+1]),
                           column value = mask[k] * interpolated input
  deform_conv2d forward  : out = weight (Cout, Cin*kh*kw) x columns + bias
Gradients come from autograd on this restatement (fp64).  Pinned against torchvision's own CPU operator in
tests/test_oracle_golden.py and against the fixtures tests/golden/dcn_*.npz generated from it.  groups = offset_groups = 1.
"""
import torch


def deform_conv2d_torch(x, offset, weight, bias=None, stride=(1, 1), padding=(0, 0), dilation=(1, 1), mask=None):
    n, c, h, w = x.shape
    cout, _, kh, kw = weight.shape
    (sh, sw), (ph, pw), (dh, dw) = stride, padding, dilation
    ho = (h + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    wo = (w + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    k = kh * kw
    dev, dt = x.device, x.dtype
    base_y = (torch.arange(ho, device=dev, dtype=dt) * sh - ph)[None, None, :, None]
    base_x = (torch.arange(wo, device=dev, dtype=dt) * sw - pw)[None, None, None, :]
    ky = (torch.arange(k, device=dev) // kw).to(dt)[None, :, None, None] * dh
    kx = (torch.arange(k, device=dev) % kw).to(dt)[None, :, None, None] * dw
    off = offset.view(n, k, 2, ho, wo)
    py = base_y + ky + off[:, :, 0]                      # (N, K, Ho, Wo)
    px = base_x + kx + off[:, :, 1]
    inside = (py > -1) & (px > -1) & (py < h) & (px < w)
    y0, x0 = torch.floor(py), torch.floor(px)
    ly, lx = py - y0, px - x0
    hy, hx = 1 - ly, 1 - lx
    flat = x.reshape(n, c, h * w)

    def corner(yy, xx, wgt):
        ok = inside & (yy >= 0) & (yy <= h - 1) & (xx >= 0) & (xx <= w - 1)
        idx = (yy.clamp(0, h - 1) * w + xx.clamp(0, w - 1)).long().reshape(n, 1, -1).expand(n, c, -1)
        # a corner outside the map is never read (torchvision's bilinear_interpolate): its gathered value is replaced by
        # 0 before it is weighted, so a non-finite pixel at the clamped position cannot leak in as 0 * Inf = NaN.  The
        # select is on the value, not on the product, for the same reason in the weight and offset gradients.
        val = torch.where(ok[:, None], torch.gather(flat, 2, idx).view(n, c, k, ho, wo), 0)
        return val * (wgt * ok.to(dt))[:, None]

    cols = corner(y0, x0, hy * hx) + corner(y0, x0 + 1, hy * lx) + corner(y0 + 1, x0, ly * hx) + corner(y0 + 1, x0 + 1, ly * lx)
    if mask is not None:
        cols = cols * mask[:, None]
    out = torch.einsum("ock,nckyx->noyx", weight.reshape(cout, c, k), cols)
    if bias is not None:
        out = out + bias[None, :, None, None]
    return out
