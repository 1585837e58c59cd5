"""Weight repacking: nn.Conv2d parameters (cout, cin, kh, kw) -> the layouts rv_conv2d consumes.

Two layouts (see include/refvsr_b200.h):
  * SIMT : fp32 [K][ceil4(cout)],  k = (ky*kw + kx)*(alloc0+alloc1) + c   (c over the *allocated*
           channels of src0 then src1; padding channels get zero weights)
  * TC   : 16-bit [nblk][S][kh][NB][64], S = kw * (chunks0 + chunks1), stage s = kx*nchunks + chunk;
           every [NB][64] slab is the byte image of a K-major SWIZZLE_128B UMMA operand tile
           (16-byte chunk j of row r stored at chunk j ^ (r % 8)), so the kernel fetches it with a plain
           bulk copy and hands it to tcgen05.mma unchanged.
"""
import hashlib
import os
from dataclasses import dataclass

import torch

from .lib import IMPL_SIMT, IMPL_TC

with open(__file__, 'rb') as _f:
    _SELF_DIGEST = hashlib.sha256(_f.read()).digest()


@dataclass
class PackedConv:
    name: str
    cout: int
    kh: int
    kw: int
    stride: int
    pad: int
    alloc0: int
    alloc1: int
    impl: int
    nb: int
    k_real: int
    wpack: torch.Tensor
    bias: torch.Tensor
    layout: int = 0


def _expand_inputs(weight, srcs):
    """weight (cout, sum(real), kh, kw) -> (cout, sum(alloc), kh, kw) with zero columns for padding."""
    cout, cin, kh, kw = weight.shape
    assert cin == sum(r for r, _ in srcs), f'weight has {cin} input channels, sources give {srcs}'
    parts, o = [], 0
    for real, alloc in srcs:
        w = weight[:, o:o + real]
        if alloc > real:
            w = torch.cat([w, weight.new_zeros(cout, alloc - real, kh, kw)], 1)
        parts.append(w)
        o += real
    return torch.cat(parts, 1)


def s2d_weights(weight, srcs, pad):
    """Re-index a stride-2 k x k convolution (k in {3,5}, pad = k//2) as a stride-1 3x3 convolution over the
    space-to-depth input:  iy = 2*oy + ky - pad = 2*(oy + dy) + ry  with dy = floor((ky-pad)/2), ry = (ky-pad) mod 2,
    so  W'[n, (ry*2+rx)*alloc + c, dy+1, dx+1] = W[n, c, ky, kx].  Returns (W', srcs') with every s2d channel
    marked real (padding channels simply carry zero weights)."""
    cout, cin, kh, kw = weight.shape
    assert kh == kw and kh in (3, 5) and pad == kh // 2
    outs, new_srcs, o = [], [], 0
    for real, alloc in srcs:
        w = weight[:, o:o + real].float()
        o += real
        wp = weight.new_zeros((cout, 4 * alloc, 3, 3), dtype=torch.float32)
        for ky in range(kh):
            dy, ry = (ky - pad) // 2, (ky - pad) % 2
            for kx in range(kw):
                dx, rx = (kx - pad) // 2, (kx - pad) % 2
                base = (ry * 2 + rx) * alloc
                wp[:, base:base + real, dy + 1, dx + 1] = w[:, :, ky, kx]
        outs.append(wp)
        new_srcs.append((4 * alloc, 4 * alloc))
    return torch.cat(outs, 1), new_srcs


def pack_simt(weight, srcs):
    w = _expand_inputs(weight.float(), srcs)            # (cout, ct, kh, kw)
    cout, ct, kh, kw = w.shape
    ldw = (cout + 3) // 4 * 4
    wk = w.permute(2, 3, 1, 0).reshape(kh * kw * ct, cout)  # k = (ky*kw+kx)*ct + c
    out = w.new_zeros(kh * kw * ct, ldw)
    out[:, :cout] = wk
    return out.contiguous()


def choose_nb(cout):
    """output channels per CTA column block for the TC kernel (multiple of 16, <= 96 so that 3x3
    weights of a two-source conv stay resident in shared memory)."""
    c16 = (cout + 15) // 16 * 16
    if c16 <= 96:
        return c16
    for nb in (96, 80, 64, 48, 32, 16):
        if c16 % nb == 0:
            return nb
    return 64


def pack_tc_sw32(weight, srcs, dtype, nb):
    """layout 2: [nblk][kx][ky][quad][NB][16], every [NB][16] slab = byte image of a K-major SWIZZLE_32B operand
    (32-byte rows; 16-byte chunk j of row r at j ^ ((r >> 2) & 1)).  Quads = 16-channel groups of src0 then src1."""
    cout, _, kh, kw = weight.shape
    w = weight.float()
    nblk = (cout + nb - 1) // nb
    quads, o = [], 0
    for real, alloc in srcs:
        ws = w[:, o:o + real]
        o += real
        for j in range((alloc + 15) // 16):
            sl = ws[:, 16 * j: min(16 * j + 16, real)] if 16 * j < real else ws[:, :0]
            if sl.shape[1] < 16:
                sl = torch.cat([sl, w.new_zeros(cout, 16 - sl.shape[1], kh, kw)], 1)
            quads.append(sl)
    nq = len(quads)
    wq = torch.stack(quads, 0)                                  # (nq, cout, 16, kh, kw)
    wpad = w.new_zeros(nq, nblk * nb, 16, kh, kw)
    wpad[:, :cout] = wq
    t = wpad.view(nq, nblk, nb, 16, kh, kw).permute(1, 5, 4, 0, 2, 3).contiguous()   # (nblk, kx, ky, q, n, c)
    t = t.view(nblk, kw, kh, nq, nb, 2, 8)
    out = torch.empty_like(t)
    for m in range(2):                                          # rows with ((r >> 2) & 1) == m swap their two chunks iff m
        rows = [r for r in range(nb) if ((r >> 2) & 1) == m]
        idx = torch.tensor(rows, device=t.device)
        src = t.index_select(4, idx)
        out.index_copy_(4, idx, src.flip(5) if m else src)
    return out.view(nblk, kw, kh, nq, nb, 16).to(dtype).contiguous()


def pack_tc(weight, srcs, dtype, nb, layout=0):
    cout, _, kh, kw = weight.shape
    w = weight.float()
    nblk = (cout + nb - 1) // nb
    # split input channels into 64-wide chunks per source
    chunks = []      # (weight slice (cout, <=64 real-or-pad, kh, kw))
    o = 0
    for real, alloc in srcs:
        ws = w[:, o:o + real]
        o += real
        nch = (alloc + 63) // 64
        for j in range(nch):
            sl = ws[:, 64 * j: min(64 * j + 64, real)] if 64 * j < real else ws[:, :0]
            pad = 64 - sl.shape[1]
            if pad:
                sl = torch.cat([sl, w.new_zeros(cout, pad, kh, kw)], 1)
            chunks.append(sl)
    nchunks = len(chunks)
    S = kw * nchunks
    wc = torch.stack(chunks, 0)                               # (nchunks, cout, 64, kh, kw)
    wpad = w.new_zeros(nchunks, nblk * nb, 64, kh, kw)
    wpad[:, :cout] = wc
    if layout in (1, 3):   # [nblk][chunk][ky][kx][n][c]: one stage per chunk holding all kh*kw taps (3 = same image, no kx-fold)
        S, kh_eff = nchunks, kh * kw
        t = wpad.view(nchunks, nblk, nb, 64, kh, kw).permute(1, 0, 4, 5, 2, 3).contiguous()
    else:             # [nblk][kx][chunk][ky][n][c]
        kh_eff = kh
        t = wpad.view(nchunks, nblk, nb, 64, kh, kw).permute(1, 5, 0, 4, 2, 3).contiguous()
    t = t.view(nblk, S, kh_eff, nb, 8, 8)                     # 64 channels = 8 chunks x 8 elements
    out = torch.empty_like(t)
    ar = torch.arange(8, device=t.device)
    for m in range(8):
        out[:, :, :, m::8] = t[:, :, :, m::8][..., ar ^ m, :]
    return out.view(nblk, S, kh_eff, nb, 64).to(dtype).contiguous()


DEFAULT_TC_LAYOUT = 1                    # 1: one box per tile (falls back to 0 when the taps do not fit), 0: boxes per (kx, chunk),
                                         # 2: 32B-swizzled 16-channel quads
SMEM_BUDGET = 232448 - 1024 - 4096      # opt-in shared memory per CTA minus alignment and static (conv_tc.cu)


def layout1_fits(kh, kw, srcs, nb):
    """layout 1 needs all taps of all chunks resident in shared memory next to >= 3 activation boxes
    (box = (16 + kh - 1) rows x (8 + kw - 1) pixels x 128 B, slot pitch rounded up to 1024 B - conv_tc.cu)"""
    if kh != kw or kh not in (1, 3, 5, 7):
        return False
    nchunks = sum((a + 63) // 64 for _, a in srcs)
    w_all = nchunks * kh * kw * nb * 128
    a_bytes = ((16 + kh - 1) * (8 + kw - 1) * 128 + 1023) // 1024 * 1024
    return w_all + 3 * a_bytes <= SMEM_BUDGET


def choose_layout(kh, kw, srcs, nb):
    """Default: layout 1 (ONE TMA box per tile and channel chunk; the kh x kw taps are shifted UMMA descriptor views
    of it) whenever all taps stay resident in shared memory, else layout 0 (one box per (kx, chunk) stage).  Layout 1
    moves 1.7x fewer bytes from L2 and keeps >= 3 whole tiles in flight, which the multi-issuer MMA path needs
    (profiles/r01_conv_timeline.md: 13.5 vs 16.2 ms / window).  REFVSR_TC_LAYOUT=0|1|2 forces a layout."""
    import os
    forced = int(os.environ.get('REFVSR_TC_LAYOUT', str(DEFAULT_TC_LAYOUT)))
    if forced in (1, 3):     # 3 = layout-1 weight image with the kx-folded 3x3 mode disabled (A/B measurements)
        return forced if layout1_fits(kh, kw, srcs, nb) else 0
    return forced


def _cache_dir():
    """Directory of the hash-keyed cache of packed layers (SURVEY 8f row 4: one-time repack of a checkpoint), or None.  Opt-in:
    REFVSR_PACK_CACHE=<dir> (or config.b200_pack_cache through network.py, which sets the same variable)."""
    d = os.environ.get('REFVSR_PACK_CACHE', '')
    return d if d not in ('', '0') else None


def _pack_key(weight, bias, srcs, stride, pad, act_dtype, prefer_tc, bias_add, tc_layout):
    """sha256 over the layer's parameters, every packing argument and this file's source (a change of the packing code
    invalidates the cache by itself); environment switches that steer the layout choice are part of the key."""
    h = hashlib.sha256()
    h.update(_SELF_DIGEST)
    h.update(repr((tuple(weight.shape), str(weight.dtype), [tuple(x) for x in srcs], stride, pad, str(act_dtype), bool(prefer_tc),
                   float(bias_add), tc_layout, os.environ.get('REFVSR_TC_LAYOUT', ''))).encode())
    h.update(weight.detach().contiguous().cpu().numpy().tobytes())
    h.update(bias.detach().float().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def pack_conv(name, weight, bias, srcs, stride, pad, act_dtype, device, prefer_tc=True, bias_add=0.0, tc_layout=None):
    """pack_conv_uncached behind the optional on-disk cache: a hit loads the packed operand image and bias instead of
    re-deriving them (bit-identical by construction: what is stored is the output of the same function)."""
    cdir = _cache_dir()
    if cdir is None:
        return pack_conv_uncached(name, weight, bias, srcs, stride, pad, act_dtype, device, prefer_tc, bias_add, tc_layout)
    path = os.path.join(cdir, _pack_key(weight, bias, srcs, stride, pad, act_dtype, prefer_tc, bias_add, tc_layout) + '.pt')
    if os.path.isfile(path):
        try:
            d = torch.load(path, map_location='cpu')
            return PackedConv(name, d['cout'], d['kh'], d['kw'], d['stride'], d['pad'], d['alloc0'], d['alloc1'], d['impl'], d['nb'],
                              d['k_real'], d['wpack'].to(device), d['bias'].to(device), d['layout'])
        except Exception:                       # unreadable / truncated entry: fall through and rewrite it
            pass
    pc = pack_conv_uncached(name, weight, bias, srcs, stride, pad, act_dtype, 'cpu', prefer_tc, bias_add, tc_layout)
    try:
        os.makedirs(cdir, exist_ok=True)
        tmp = f'{path}.{os.getpid()}.tmp'
        torch.save(dict(cout=pc.cout, kh=pc.kh, kw=pc.kw, stride=pc.stride, pad=pc.pad, alloc0=pc.alloc0, alloc1=pc.alloc1,
                        impl=pc.impl, nb=pc.nb, k_real=pc.k_real, wpack=pc.wpack, bias=pc.bias, layout=pc.layout), tmp)
        os.replace(tmp, path)                   # atomic: concurrent ranks may pack the same layer
    except OSError:
        pass                                    # read-only / full cache directory: the cache is an optimisation only
    pc.wpack, pc.bias = pc.wpack.to(device), pc.bias.to(device)
    return pc


def pack_conv_uncached(name, weight, bias, srcs, stride, pad, act_dtype, device, prefer_tc=True, bias_add=0.0, tc_layout=None):
    """Pick the implementation and build the packed tensors.  `srcs` = [(real, alloc), ...] (1 or 2)."""
    cout, _, kh, kw = weight.shape
    alloc0 = srcs[0][1]
    alloc1 = srcs[1][1] if len(srcs) > 1 else 0
    tc_ok = (prefer_tc and stride == 1 and act_dtype in (torch.float16, torch.bfloat16)
             and all(a % 8 == 0 for _, a in srcs) and kh <= 7 and kw <= 7)
    b = bias.detach().float() + bias_add
    if tc_ok:
        nb = choose_nb(cout)
        layout = choose_layout(kh, kw, srcs, nb) if tc_layout is None else tc_layout
        wp = (pack_tc_sw32(weight.detach(), srcs, act_dtype, nb) if layout == 2
              else pack_tc(weight.detach(), srcs, act_dtype, nb, layout)).to(device)
        return PackedConv(name, cout, kh, kw, stride, pad, alloc0, alloc1, IMPL_TC, nb,
                          kh * kw * (alloc0 + alloc1), wp, b.to(device).contiguous(), layout)
    wp = pack_simt(weight.detach(), srcs).to(device)
    return PackedConv(name, cout, kh, kw, stride, pad, alloc0, alloc1, IMPL_SIMT, 0,
                      kh * kw * (alloc0 + alloc1), wp, b.to(device).contiguous())


def pack_dcn(name, weight, bias, act_dtype, device):
    """weight (cout <= 64, 64, 3, 3) of a ModulatedDCNPack -> the operand rv_dcn3x3 reads: the single-box tensor-core image
    ([9 taps][nb][64], layout 1) for 16-bit activations, fp32 [576][ceil4(cout)] for the CUDA-core variant"""
    assert weight.shape[1:] == (64, 3, 3) and weight.shape[0] <= 64, f'{name}: {tuple(weight.shape)} is not a 64-channel 3x3 DCN'
    return pack_conv(name, weight, bias, [(64, 64)], 1, 1, act_dtype, device, tc_layout=1)


@dataclass
class PackedResBlock:
    name: str
    cout: int
    alloc: int
    nb: int
    w1: torch.Tensor
    b1: torch.Tensor
    w2: torch.Tensor
    b2: torch.Tensor


def resblock_fusable(w1, w2, alloc, act_dtype):
    c = w1.shape[0]
    return (act_dtype in (torch.float16, torch.bfloat16) and tuple(w1.shape) == (c, c, 3, 3) and tuple(w2.shape) == (c, c, 3, 3)
            and alloc % 8 == 0 and c <= alloc <= 64)


def pack_resblock(name, w1, b1, w2, b2, alloc, act_dtype, device):
    """both 3x3 convs of a residual block in the single-box layout ([1][1][9 taps][nb][64]) for rv_resblock"""
    c = w1.shape[0]
    nb = (c + 15) // 16 * 16
    p1 = pack_tc(w1.detach(), [(c, alloc)], act_dtype, nb, layout=1).to(device)
    p2 = pack_tc(w2.detach(), [(c, alloc)], act_dtype, nb, layout=1).to(device)
    return PackedResBlock(name, c, alloc, nb, p1, b1.detach().float().to(device).contiguous(), p2,
                          b2.detach().float().to(device).contiguous())


@dataclass
class PackedChainLayer:
    name: str
    nb: int
    wpack: torch.Tensor      # [1][1][9][nb][64] layout-1 image
    bias: torch.Tensor       # nb floats, zero beyond cout


def chain_nb(alloc):
    return (alloc + 15) // 16 * 16


def chain_ok(weight, alloc, act_dtype):
    """can this conv be a layer of rv_conv_chain?  3x3, C -> C, 16-bit activations, C <= 48 allocated channels"""
    c = weight.shape[0]
    return (act_dtype in (torch.float16, torch.bfloat16) and tuple(weight.shape) == (c, c, 3, 3) and alloc % 8 == 0
            and c <= alloc <= 48)


def pack_chain(name, weight, bias, alloc, act_dtype, device):
    c = weight.shape[0]
    nb = chain_nb(alloc)
    wp = pack_tc(weight.detach(), [(c, alloc)], act_dtype, nb, layout=1).to(device)
    b = torch.zeros(nb, dtype=torch.float32)
    b[:c] = bias.detach().float().cpu()
    return PackedChainLayer(name, nb, wp, b.to(device).contiguous())
