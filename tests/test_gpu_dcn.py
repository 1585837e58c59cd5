"""-m gpu: rv_dcn3x3 (tcgen05 and CUDA-core variants) against the explicit-index modulated deformable conv of
tests/dcn_reference.py, evaluated in float64 on the same dtype-rounded inputs.  Offsets span +-4 px, so samples cross
integer cells and fall off the map at the border; mask logits span [-4, 4]."""
import pytest
import torch
import torch.nn.functional as F

from dcn_reference import modulated_deform_conv3x3, random_offset_map
from refvsr_b200 import packing
from refvsr_b200.lib import ACT_LRELU01, ACT_NONE, IMPL_SIMT, IMPL_TC

pytestmark = pytest.mark.gpu

DT = {'fp32': torch.float32, 'fp16': torch.float16, 'bf16': torch.bfloat16}
TOL = {torch.float32: 1e-4, torch.float16: 4e-3, torch.bfloat16: 3e-2}

# H, W, cout, out_cs, act: the three PCD pyramid levels of a 270x480 clip (padded to 272x480) and an odd size whose last
# 128-pixel tile is partial, with 48 output channels and a row pitch that is not a multiple of 16 bytes
CASES = [(68, 120, 64, 64, ACT_NONE), (136, 240, 64, 64, ACT_LRELU01), (272, 480, 64, 64, ACT_LRELU01), (37, 53, 48, 50, ACT_NONE)]


def _inputs(H, W, cout, dtype, seed, span=4.0):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(H, W, 64, generator=gen).to(dtype)
    w = (torch.randn(cout, 64, 3, 3, generator=gen) / 24).to(dtype if dtype != torch.float32 else torch.float32)
    b = torch.randn(cout, generator=gen) * 0.1
    om = random_offset_map(H, W, seed=seed + 1, span=span)
    return x, w.float(), b, om


def _expected(x, om, w, b, act):
    ref = modulated_deform_conv3x3(x.cuda().double(), om.cuda().double(), w.cuda().double(), b.cuda().double())
    return F.leaky_relu(ref, 0.1) if act == ACT_LRELU01 else ref


@pytest.mark.parametrize('dt', ['bf16', 'fp16', 'fp32'])
@pytest.mark.parametrize('case', CASES, ids=[f'{c[0]}x{c[1]}' for c in CASES])
def test_dcn_matches_reference(cuda_ops, case, dt):
    H, W, cout, out_cs, act = case
    dtype = DT[dt]
    x, w, b, om = _inputs(H, W, cout, dtype, seed=H + W)
    layer = packing.pack_dcn('dcn', w, b, dtype, 'cuda')
    assert layer.impl == (IMPL_SIMT if dtype == torch.float32 else IMPL_TC)
    out = torch.full((H, W, out_cs), 7.0, dtype=dtype, device='cuda')
    n0 = cuda_ops.launch_count()
    cuda_ops.dcn3x3(layer, x.cuda(), om.cuda(), out, act=act)
    torch.cuda.synchronize()
    assert cuda_ops.launch_count() - n0 == 1
    exp = _expected(x, om, w, b, act)
    err = (out[..., :cout].double() - exp).abs().max().item()
    ref = exp.abs().max().item()
    assert err <= TOL[dtype] * max(1.0, ref), f'{dt} {H}x{W}: max err {err:.3e} (ref max {ref:.3e})'
    assert bool((out[..., cout:] == 7.0).all()), 'channels beyond cout were written'


@pytest.mark.parametrize('dt', ['bf16', 'fp16'])
def test_tensor_core_and_cuda_core_variants_agree(cuda_ops, dt):
    """same 16-bit inputs through both implementations: they differ only by the 16-bit rounding of the sampled operand"""
    dtype = DT[dt]
    H, W = 70, 66
    x, w, b, om = _inputs(H, W, 64, dtype, seed=11)
    tc = packing.pack_dcn('dcn', w, b, dtype, 'cuda')
    simt = packing.pack_conv('dcn', w, b, [(64, 64)], 1, 1, dtype, 'cuda', prefer_tc=False)
    o1 = torch.empty(H, W, 64, dtype=dtype, device='cuda')
    o2 = torch.empty_like(o1)
    cuda_ops.dcn3x3(tc, x.cuda(), om.cuda(), o1, act=ACT_LRELU01)
    cuda_ops.dcn3x3(simt, x.cuda(), om.cuda(), o2, act=ACT_LRELU01)
    torch.cuda.synchronize()
    ref = o2.float().abs().max().item()
    assert (o1.float() - o2.float()).abs().max().item() <= TOL[dtype] * max(1.0, ref)


def test_zero_offsets_reduce_to_a_masked_conv(cuda_ops):
    """integral sample positions (zero offsets) with mask logit 0 (m = 0.5): the DCN is 0.5 x a zero-padded 3x3 conv"""
    H, W = 40, 72
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(H, W, 64, generator=gen)
    w = torch.randn(64, 64, 3, 3, generator=gen) / 24
    b = torch.randn(64, generator=gen) * 0.1
    om = torch.zeros(H, W, 216)
    layer = packing.pack_dcn('dcn', w, b, torch.float32, 'cuda')
    out = torch.empty(H, W, 64, device='cuda')
    cuda_ops.dcn3x3(layer, x.cuda(), om.cuda(), out)
    exp = F.conv2d(x.permute(2, 0, 1)[None].double(), 0.5 * w.double(), b.double(), padding=1)[0].permute(1, 2, 0)
    assert (out.cpu().double() - exp).abs().max().item() <= 1e-4


def test_dcn_rejects_a_short_offset_map(cuda_ops):
    x = torch.zeros(8, 8, 64, dtype=torch.bfloat16, device='cuda')
    layer = packing.pack_dcn('dcn', torch.zeros(64, 64, 3, 3), torch.zeros(64), torch.bfloat16, 'cuda')
    with pytest.raises(ValueError, match='216'):
        cuda_ops.dcn3x3(layer, x, torch.zeros(8, 8, 144, device='cuda'), torch.empty_like(x))
