"""Times rv_dcn3x3 at the three PCD pyramid levels of a 270x480 clip and prints one JSON line.

EDVR's PCD alignment (models/archs/edvr_net.py:61-296) runs its modulated deformable convs on 64-channel maps at the
reflect-padded input size and its two stride-2 levels: 272x480, 136x240, 68x120.  Per size and implementation the line
holds the kernel time (CUDA events around `--iters` launches after a warm-up), the FLOP and compulsory bytes derived from
the shapes, the achieved rates, the fraction of the larger of the two data-sheet bounds and which bound that is.  The
baseline is torchvision's CUDA deform_conv2d (fp32, NCHW, mask given), fed the same inputs split the way the reference's
ModulatedDCNPack splits them.  Inputs are rotated through enough copies that every timed launch reads them from HBM, not
L2.  `offset_bf16_effect` runs the bf16 kernel on fp32 offsets and on the same offsets rounded to bf16 and compares both
with a float64 evaluation, which is why the kernel reads an fp32 offset map.  The card's name and power limit are read in
the same run.

usage: python tools/bench_dcn.py [--iters 200]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from dcn_reference import modulated_deform_conv3x3, random_offset_map, split_offset_mask  # noqa: E402
from refvsr_b200 import packing  # noqa: E402
from refvsr_b200.lib import ACT_LRELU01, CudaOps  # noqa: E402

SIZES = [(68, 120), (136, 240), (272, 480)]
PEAK_BYTES = 7.7e12          # HGX B200 data sheet, one GPU, HBM3e
PEAK_FLOPS_16 = 2.25e15      # dense BF16 / FP16 tensor
L2_BYTES = 126 << 20


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'name': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip().splitlines()[0] if q.stdout else q.stderr.strip()}


def time_launches(fn, nsets, iters):
    for i in range(min(nsets, 3) * 2):
        fn(i % nsets)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i % nsets)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / iters


def roofline(t, flops, nbytes, peak_flops=None):
    """peak_flops None (fp32 CUDA-core paths): only the HBM bound is stated"""
    tb, tf = nbytes / PEAK_BYTES, (flops / peak_flops if peak_flops else 0.0)
    return {'us': round(t * 1e6, 2), 'tflops': round(flops / t / 1e12, 2), 'gbytes_per_s': round(nbytes / t / 1e9, 1),
            'bound': 'hbm' if tb >= tf else 'compute', 'fraction_of_bound': round(max(tb, tf) / t, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_dcn needs a CUDA device'
    ops = CudaOps()
    res = {'kind': 'dcn3x3', 'card': card(), 'sizes': {}}
    gen = torch.Generator().manual_seed(0)
    w = torch.randn(64, 64, 3, 3, generator=gen) / 24
    b = torch.randn(64, generator=gen) * 0.1
    layers = {dt: packing.pack_dcn('dcn', w, b, dt, 'cuda') for dt in (torch.bfloat16, torch.float16, torch.float32)}
    try:
        from torchvision.ops import deform_conv2d
    except Exception as ex:                                         # noqa: BLE001
        deform_conv2d, res['torchvision_error'] = None, repr(ex)
    for H, W in SIZES:
        P = H * W
        flops = 2.0 * 9 * 64 * 64 * P
        row = {'pixels': P, 'gflop': round(flops / 1e9, 3),
               'gathered_bytes_per_pixel': 9 * 8 * 4 * 16}          # 4 corners x 16-byte vectors per (tap, group)
        for name, dt in (('bf16_tc', torch.bfloat16), ('fp16_tc', torch.float16), ('fp32_simt', torch.float32)):
            e = torch.tensor([], dtype=dt).element_size()
            nbytes = P * (64 * e + 216 * 4 + 64 * e)                 # x + fp32 offset / mask map + out
            nsets = max(2, -(-2 * L2_BYTES // nbytes))
            xs = [torch.randn(H, W, 64, device='cuda').to(dt) for _ in range(nsets)]
            oms = [random_offset_map(H, W, seed=s).cuda() for s in range(nsets)]
            outs = [torch.empty(H, W, 64, dtype=dt, device='cuda') for _ in range(nsets)]
            t = time_launches(lambda i: ops.dcn3x3(layers[dt], xs[i], oms[i], outs[i], act=ACT_LRELU01), nsets, args.iters)
            row[name] = roofline(t, flops, nbytes, None if dt == torch.float32 else PEAK_FLOPS_16)
            row[name]['bytes'] = nbytes
            del xs, oms, outs
        if deform_conv2d is not None:
            nbytes = P * (64 * 4 + 216 * 4 + 64 * 4)
            nsets = max(2, -(-2 * L2_BYTES // nbytes))
            xs = [torch.randn(1, 64, H, W, device='cuda') for _ in range(nsets)]
            sp = [split_offset_mask(random_offset_map(H, W, seed=s).cuda()) for s in range(nsets)]
            sp = [(o.permute(2, 0, 1)[None].contiguous(), m.permute(2, 0, 1)[None].contiguous()) for o, m in sp]
            wc, bc = w.cuda(), b.cuda()
            t = time_launches(lambda i: deform_conv2d(xs[i], sp[i][0], wc, bc, padding=1, mask=sp[i][1]), nsets, args.iters)
            row['torchvision_fp32'] = roofline(t, flops, nbytes)
            row['speedup_bf16_tc_vs_torchvision'] = round(row['torchvision_fp32']['us'] / row['bf16_tc']['us'], 2)
            del xs, sp
        res['sizes'][f'{H}x{W}'] = row
    # fp32 vs bf16 offsets: error of the bf16 kernel against float64, with the offset map as read and rounded to bf16
    H, W = SIZES[0]
    x = torch.randn(H, W, 64, generator=gen).bfloat16()
    eff = {}
    for span in (0.3, 4.0):
        om = random_offset_map(H, W, seed=7, span=span)
        exp = modulated_deform_conv3x3(x.cuda().double(), om.cuda().double(), w.bfloat16().cuda().double(), b.cuda().double())
        errs = {}
        for tag, o in (('fp32_offsets', om), ('bf16_offsets', om.bfloat16().float())):
            out = torch.empty(H, W, 64, dtype=torch.bfloat16, device='cuda')
            ops.dcn3x3(layers[torch.bfloat16], x.cuda(), o.cuda(), out)
            d = out.double() - exp
            peak = exp.abs().max().item()
            errs[tag] = {'max_abs': d.abs().max().item(), 'rms': d.pow(2).mean().sqrt().item(),
                         'psnr_db_vs_peak': round(10 * torch.log10(torch.tensor(peak ** 2 / d.pow(2).mean().item())).item(), 2)}
        eff[f'offset_span_{span}px'] = errs
    res['offset_bf16_effect'] = eff
    print(json.dumps(res), flush=True)


if __name__ == '__main__':
    main()
