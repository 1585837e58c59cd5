"""The explicit-index modulated deformable conv (tests/dcn_reference.py, the yardstick of rv_dcn3x3) against torchvision's
deform_conv2d, and the packed operand rv_dcn3x3's tensor-core path reads.  No GPU needed."""
import pytest
import torch

from dcn_reference import modulated_deform_conv3x3, random_offset_map, split_offset_mask
from refvsr_b200 import packing
from refvsr_b200.lib import IMPL_SIMT, IMPL_TC


@pytest.mark.parametrize('H,W,span,cout', [(9, 13, 4.0, 64), (17, 11, 0.3, 48), (5, 6, 8.0, 64)])
def test_reference_dcn_matches_torchvision(H, W, span, cout):
    tvops = pytest.importorskip('torchvision.ops')
    gen = torch.Generator().manual_seed(H * 100 + W)
    x = torch.randn(H, W, 64, generator=gen)
    wt = torch.randn(cout, 64, 3, 3, generator=gen) / 24
    b = torch.randn(cout, generator=gen) * 0.1
    om = random_offset_map(H, W, seed=H + W, span=span)
    ours = modulated_deform_conv3x3(x, om, wt, b)
    off, mask = split_offset_mask(om)
    tv = tvops.deform_conv2d(x.permute(2, 0, 1)[None], off.permute(2, 0, 1)[None], wt, b, padding=1,
                             mask=mask.permute(2, 0, 1)[None])[0].permute(1, 2, 0)
    assert (ours - tv).abs().max().item() <= 1e-5 * max(1.0, tv.abs().max().item())


def test_random_offsets_reach_the_border_and_cross_cells():
    """the generated offset maps exercise what small trained offsets would not: samples beyond the map and across cells"""
    H, W = 12, 16
    om = random_offset_map(H, W, seed=1)
    off = om[..., :144]
    assert off.abs().max() > 3.5 and (off.abs() > 1).float().mean() > 0.5
    ys = torch.arange(H).view(H, 1, 1).float()
    dy = off[..., 0::2]
    h = ys - 1 + dy
    assert ((h <= -1) | (h >= H)).any()


def test_pack_dcn_layouts():
    """16-bit activations get the single-box tensor-core image [9 taps][nb][64] (16-byte chunk j of row n at j ^ (n % 8)),
    fp32 the CUDA-core [576][ceil4(cout)] matrix in (tap, channel) order"""
    gen = torch.Generator().manual_seed(5)
    w = torch.randn(48, 64, 3, 3, generator=gen)
    b = torch.randn(48, generator=gen)
    tc = packing.pack_dcn('d', w, b, torch.bfloat16, 'cpu')
    assert tc.impl == IMPL_TC and tc.nb == 48 and tc.layout == 1 and tuple(tc.wpack.shape) == (1, 1, 9, 48, 64)
    img = tc.wpack.view(9, 48, 8, 8).float()
    for k, n, j in ((0, 0, 0), (4, 13, 5), (8, 47, 7), (5, 9, 2)):
        ky, kx = divmod(k, 3)
        assert torch.equal(img[k, n, j ^ (n % 8)], w[n, 8 * j:8 * j + 8, ky, kx].bfloat16().float())
    simt = packing.pack_dcn('d', w, b, torch.float32, 'cpu')
    assert simt.impl == IMPL_SIMT and tuple(simt.wpack.shape) == (576, 48)
    assert torch.equal(simt.wpack[4 * 64 + 10, 7], w[7, 10, 1, 1])
    with pytest.raises(AssertionError):
        packing.pack_dcn('d', torch.zeros(64, 48, 3, 3), torch.zeros(64), torch.bfloat16, 'cpu')


def test_dcn_entry_point_rejects_bad_arguments_without_a_gpu():
    from refvsr_b200.lib import load_library
    lib = load_library()
    assert lib.rv_dcn3x3(None, None, 216, 8, 8, 2, None, None, 64, 64, 0, 1, None, 64, None) == -1
    assert b'null argument' in lib.rv_last_error()


def test_dcn_op_refuses_a_tensor_core_layer_in_another_layout():
    """a layer packed for rv_conv2d's per-kx boxes (layout 0) must not reach the DCN kernel, which reads the single-box image;
    the check runs before any device work"""
    from refvsr_b200.lib import CudaOps
    w = torch.zeros(64, 64, 3, 3)
    layer = packing.pack_conv('d', w, torch.zeros(64), [(64, 64)], 1, 1, torch.bfloat16, 'cpu', tc_layout=0)
    ops = CudaOps.__new__(CudaOps)           # no device needed: the assertion precedes the launch
    x = torch.zeros(4, 4, 64, dtype=torch.bfloat16)
    with pytest.raises(AssertionError, match='layout-1'):
        ops.dcn3x3(layer, x, torch.zeros(4, 4, 216), torch.zeros_like(x))
