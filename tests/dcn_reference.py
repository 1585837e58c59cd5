"""Modulated deformable 3x3 convolution written as explicit index arithmetic: the yardstick of rv_dcn3x3.

Restates mmcv's modulated_deform_conv2d (stride 1, pad 1, dilation 1, groups 1) as EDVR's ModulatedDCNPack calls it
(models/archs/edvr_net.py:49-58), taking conv_offset's raw output: for deform group g and tap k = 3*ky + kx
    dy = om[18g + 2k], dx = om[18g + 2k + 1], m = sigmoid(om[144 + 9g + k])
(torch.chunk(out, 3) + torch.cat((o1, o2)) leaves the first 144 channels in place).  Sampling follows mmcv's
modulated_deformable_im2col / dmcn_im2col_bilinear: a sample at (h, w) is 0 unless -1 < h < H and -1 < w < W, and each
bilinear corner outside the map contributes 0.
"""
import torch


def split_offset_mask(om, groups=8):
    """om (..., 27 * groups) raw conv_offset output -> (offset (..., 18 * groups), mask (..., 9 * groups)), as the pack does"""
    return om[..., :18 * groups], torch.sigmoid(om[..., 18 * groups:27 * groups])


def modulated_deform_conv3x3(x, om, weight, bias, groups=8):
    """x (H, W, Cin) NHWC, om (H, W, >= 27 * groups) raw conv_offset output, weight (cout, Cin, 3, 3), bias (cout,)
    -> (H, W, cout), in x's floating dtype"""
    H, W, Cin = x.shape
    cg = Cin // groups
    offset, mask = split_offset_mask(om.to(x), groups)
    ys = torch.arange(H, dtype=x.dtype, device=x.device).view(H, 1)
    xs = torch.arange(W, dtype=x.dtype, device=x.device).view(1, W)
    col = x.new_zeros(H, W, Cin, 9)
    for g in range(groups):
        xg = x[..., g * cg:(g + 1) * cg]
        for k in range(9):
            ky, kx = divmod(k, 3)
            h = ys - 1 + ky + offset[..., 18 * g + 2 * k]
            w = xs - 1 + kx + offset[..., 18 * g + 2 * k + 1]
            inside = (h > -1) & (w > -1) & (h < H) & (w < W)
            h0, w0 = torch.floor(h), torch.floor(w)
            lh, lw = h - h0, w - w0
            val = x.new_zeros(H, W, cg)
            for oy, ox, wt in ((0, 0, (1 - lh) * (1 - lw)), (0, 1, (1 - lh) * lw), (1, 0, lh * (1 - lw)), (1, 1, lh * lw)):
                yy, xx = h0 + oy, w0 + ox
                ok = inside & (yy >= 0) & (yy <= H - 1) & (xx >= 0) & (xx <= W - 1)
                v = xg[yy.clamp(0, H - 1).long(), xx.clamp(0, W - 1).long()]
                val = val + torch.where(ok, wt, torch.zeros_like(wt)).unsqueeze(-1) * v
            col[..., g * cg:(g + 1) * cg, k] = val * mask[..., 9 * g + k].unsqueeze(-1)
    out = torch.einsum('hwck,nck->hwn', col, weight.to(x).reshape(weight.shape[0], Cin, 9))
    return out + bias.to(x)


def random_offset_map(H, W, seed, span=4.0, groups=8):
    """raw conv_offset output (H, W, 27 * groups) fp32 whose offsets are uniform in [-span, span] px (so that samples cross
    integer cells and leave the map at the border) and whose mask logits are uniform in [-4, 4]"""
    gen = torch.Generator().manual_seed(seed)
    off = (torch.rand(H, W, 18 * groups, generator=gen) * 2 - 1) * span
    logit = (torch.rand(H, W, 9 * groups, generator=gen) * 2 - 1) * 4
    return torch.cat([off, logit], -1)
