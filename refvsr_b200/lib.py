"""ctypes binding of the C-ABI library (include/refvsr_b200.h) and the `CudaOps` operator set.

`CudaOps` is the ONLY implementation of the operator interface that ships in the product: every
method launches hand-written sm_100a kernels from `librefvsr_b200.so` on torch's current CUDA stream.
There is no CPU / eager fallback - constructing `CudaOps` without the built library or without a
CUDA device raises.  torch is used for device memory and streams only.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'librefvsr_b200.so')

RV_F32, RV_F16, RV_BF16 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_LRELU01, ACT_LRELU02, ACT_CLAMP3 = 0, 1, 2, 3, 4
IMPL_SIMT, IMPL_TC = 0, 1

DTYPE_CODE = {torch.float32: RV_F32, torch.float16: RV_F16, torch.bfloat16: RV_BF16}


class rv_conv_desc(C.Structure):
    _fields_ = [
        ('src0', C.c_void_p), ('src1', C.c_void_p), ('c0', C.c_int32), ('c1', C.c_int32),
        ('in_dtype', C.c_int32), ('H', C.c_int32), ('W', C.c_int32),
        ('wpack', C.c_void_p), ('bias', C.c_void_p), ('cout', C.c_int32),
        ('kh', C.c_int32), ('kw', C.c_int32), ('stride', C.c_int32), ('pad', C.c_int32),
        ('act_pre', C.c_int32), ('act_post', C.c_int32),
        ('gate', C.c_void_p), ('gate_cs', C.c_int32),
        ('res', C.c_void_p), ('res_cs', C.c_int32), ('res_dtype', C.c_int32),
        ('out', C.c_void_p), ('out_cs', C.c_int32), ('out_dtype', C.c_int32),
        ('pixel_shuffle', C.c_int32), ('impl', C.c_int32), ('nb', C.c_int32), ('k_real', C.c_int32),
        ('layout', C.c_int32),
    ]


class rv_resblock_desc(C.Structure):
    _fields_ = [
        ('src', C.c_void_p), ('c', C.c_int32), ('dtype', C.c_int32), ('H', C.c_int32), ('W', C.c_int32),
        ('w1', C.c_void_p), ('b1', C.c_void_p), ('w2', C.c_void_p), ('b2', C.c_void_p),
        ('cout', C.c_int32), ('nb', C.c_int32), ('act_mid', C.c_int32), ('act_post', C.c_int32),
        ('out', C.c_void_p), ('out_cs', C.c_int32),
    ]


class rv_chain_layer(C.Structure):
    _fields_ = [('wpack', C.c_void_p), ('bias', C.c_void_p), ('src', C.c_int32), ('res', C.c_int32), ('dst', C.c_int32),
                ('act_pre', C.c_int32), ('act_post', C.c_int32)]


class rv_conv_chain_desc(C.Structure):
    _fields_ = [('buf', C.c_void_p * 6), ('nbuf', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('C', C.c_int32),
                ('dtype', C.c_int32), ('nb', C.c_int32), ('layers', C.POINTER(rv_chain_layer)), ('nlayers', C.c_int32),
                ('flags', C.c_void_p), ('max_ctas', C.c_int32)]


CHAIN_MAX_LAYERS, CHAIN_MAX_BUFFERS = 64, 6

# name -> (restype, argtypes); mirrors include/refvsr_b200.h one to one (tests check the export list)
_P, _I, _F = C.c_void_p, C.c_int, C.c_float
SIGNATURES = {
    'rv_last_error': (C.c_char_p, []),
    'rv_version': (_I, []),
    'rv_launch_count': (C.c_uint64, []),
    'rv_conv2d': (_I, [C.POINTER(rv_conv_desc), _P]),
    'rv_set_conv_cta_cap': (_I, [_I]),
    'rv_conv2d_tc_plan': (_I, [C.POINTER(rv_conv_desc), _I, _I, C.POINTER(C.c_int32)]),
    'rv_resblock': (_I, [C.POINTER(rv_resblock_desc), _P]),
    'rv_conv_chain': (_I, [C.POINTER(rv_conv_chain_desc), _P]),
    'rv_dcn3x3': (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _I, _I, _I, _I, _P, _I, _P]),
    'rv_space_to_depth2': (_I, [_P, _I, _I, _I, _I, _P, _P]),
    'rv_prep_image': (_I, [_P, _I, _I, _P, _I, _P, _I, _I, _P]),
    'rv_spynet_resize_norm': (_I, [_P, _I, _I, _P, _I, _I, _P]),
    'rv_avgpool2': (_I, [_P, _I, _I, _I, _P, _P]),
    'rv_maxpool2': (_I, [_P, _I, _I, _I, _I, _P, _P]),
    'rv_resize_planes': (_I, [_P, _I, _I, _I, _F, _I, _I, _I, _I, _P, _P]),
    'rv_spynet_level_input': (_I, [_P, _P, _P, _I, _I, _P, _I, _P, _P]),
    'rv_flow_resize': (_I, [_P, _I, _I, _P, _I, _I, _P]),
    'rv_warp': (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P, _P]),
    'rv_warp3': (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    'rv_patch_pack': (_I, [_P, _I, _I, _I, _I, _I, _P, _I, _P]),
    'rv_match_argmax': (_I, [_P, _I, _P, _I, _I, _F, _P, _P, _I, _P]),
    'rv_gather_blocks': (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P, _P]),
    'rv_aligned_sample': (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P]),
    'rv_bicubic_up2_image': (_I, [_P, _I, _I, _P, _I, _I, _P]),
    'rv_conf_pair': (_I, [_P, _P, _I, _I, _I, _P, _I, _I, _P]),
    'rv_conf_max': (_I, [_P, _P, _P, _I, _P]),
    'rv_frames_differ': (_I, [_P, _P, _P, _I, _P, _P]),
    'rv_reconstruct': (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _P, _P]),
}

_lib = None


def load_library(path=LIB_PATH):
    """dlopen the kernels library and attach prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(path):
        raise RuntimeError(
            f'{path} not found: build the CUDA extension first (python -c "import __graft_entry__ as g; '
            'g.build()").  refvsr_b200 has no CPU fallback.')
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _check(lib, rc, what):
    if rc != 0:
        msg = lib.rv_last_error().decode('utf-8', 'replace')
        if rc == -1:
            raise ValueError(f'{what}: {msg}')
        raise RuntimeError(f'{what}: {msg} (code {rc})')


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _chk_dev(*ts):
    for t in ts:
        if t is not None:
            assert t.is_cuda and t.is_contiguous(), 'operands must be contiguous CUDA tensors'


class CudaOps:
    """Operator set backed by librefvsr_b200.so.  Shapes: activations (H, W, C); images (3, H, W)
    fp32; flows (H, W, 2) fp32; confidence maps (H, W) fp32; index maps (H*W,) int32."""

    name = 'cuda'

    def __init__(self, device='cuda'):
        if not torch.cuda.is_available():
            raise RuntimeError('refvsr_b200 requires a CUDA device (no CPU fallback)')
        self.lib = load_library()
        self.device = torch.device(device)

    # -- helpers ---------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch_count(self):
        return int(self.lib.rv_launch_count())

    def set_conv_cta_cap(self, cap):
        """persistent-grid bound of the following tensor-core conv launches (0 = one CTA per SM); returns the previous value"""
        return int(self.lib.rv_set_conv_cta_cap(int(cap)))

    # -- convolution ------------------------------------------------------------------------------
    def conv2d(self, layer, src0, src1, out, gate=None, res=None, act_pre=ACT_NONE, act_post=ACT_NONE,
               pixel_shuffle=False):
        """`layer` is a packing.PackedConv.  Output geometry is checked by the caller (engine)."""
        _chk_dev(src0, src1, out, gate, res)
        d = rv_conv_desc()
        d.src0 = src0.data_ptr()
        d.src1 = src1.data_ptr() if src1 is not None else None
        d.c0 = src0.shape[2]
        d.c1 = src1.shape[2] if src1 is not None else 0
        assert (d.c0, d.c1) == (layer.alloc0, layer.alloc1), \
            f'{layer.name}: source channels {(d.c0, d.c1)} != packed layout {(layer.alloc0, layer.alloc1)}'
        d.in_dtype = DTYPE_CODE[src0.dtype]
        d.H, d.W = src0.shape[0], src0.shape[1]
        d.wpack = layer.wpack.data_ptr()
        d.bias = layer.bias.data_ptr()
        d.cout = layer.cout
        d.kh, d.kw, d.stride, d.pad = layer.kh, layer.kw, layer.stride, layer.pad
        d.act_pre, d.act_post = act_pre, act_post
        d.gate = gate.data_ptr() if gate is not None else None
        d.gate_cs = gate.shape[2] if gate is not None else 0
        d.res = res.data_ptr() if res is not None else None
        d.res_cs = res.shape[2] if res is not None else 0
        d.res_dtype = DTYPE_CODE[res.dtype] if res is not None else 0
        d.out = out.data_ptr()
        d.out_cs = out.shape[2]
        d.out_dtype = DTYPE_CODE[out.dtype]
        d.pixel_shuffle = 1 if pixel_shuffle else 0
        d.impl = layer.impl
        d.nb = layer.nb
        d.k_real = layer.k_real
        d.layout = getattr(layer, 'layout', 0)
        _check(self.lib, self.lib.rv_conv2d(C.byref(d), self._stream()), f'rv_conv2d[{layer.name}]')

    def resblock(self, rb, src, out, act_mid, act_post=ACT_NONE):
        """`rb` is a packing.PackedResBlock; out = act_post(src + conv2(act_mid(conv1(src))))"""
        _chk_dev(src, out)
        assert src.shape[2] == rb.alloc and src.dtype == out.dtype and src.data_ptr() != out.data_ptr()
        d = rv_resblock_desc()
        d.src, d.c, d.dtype = src.data_ptr(), src.shape[2], DTYPE_CODE[src.dtype]
        d.H, d.W = src.shape[0], src.shape[1]
        d.w1, d.b1, d.w2, d.b2 = rb.w1.data_ptr(), rb.b1.data_ptr(), rb.w2.data_ptr(), rb.b2.data_ptr()
        d.cout, d.nb, d.act_mid, d.act_post = rb.cout, rb.nb, act_mid, act_post
        d.out, d.out_cs = out.data_ptr(), out.shape[2]
        _check(self.lib, self.lib.rv_resblock(C.byref(d), self._stream()), f'rv_resblock[{rb.name}]')

    def conv_chain(self, bufs, layers, flags, max_ctas=0):
        """bufs: list of (H, W, C) tensors of one dtype / geometry; layers: [(packing.PackedChainLayer, src, res, dst, act_pre,
        act_post)] with buffer indices (res = -1: none); flags: int32 scratch with >= ceil(H/16)*ceil(W/8) entries.
        Launches ceil(len(layers) / 64) persistent kernels (rv_conv_chain)."""
        _chk_dev(*bufs)
        H, W, Cc = bufs[0].shape
        assert all(tuple(b.shape) == (H, W, Cc) and b.dtype == bufs[0].dtype for b in bufs) and len(bufs) <= CHAIN_MAX_BUFFERS
        assert flags.dtype == torch.int32 and flags.numel() >= ((H + 15) // 16) * ((W + 7) // 8)
        nb = layers[0][0].nb
        for i in range(0, len(layers), CHAIN_MAX_LAYERS):
            part = layers[i:i + CHAIN_MAX_LAYERS]
            arr = (rv_chain_layer * len(part))()
            for j, (pk, src, res, dst, a0, a1) in enumerate(part):
                assert pk.nb == nb
                arr[j].wpack, arr[j].bias = pk.wpack.data_ptr(), pk.bias.data_ptr()
                arr[j].src, arr[j].res, arr[j].dst, arr[j].act_pre, arr[j].act_post = src, res, dst, a0, a1
            d = rv_conv_chain_desc()
            for b, t in enumerate(bufs):
                d.buf[b] = t.data_ptr()
            d.nbuf, d.H, d.W, d.C, d.dtype, d.nb = len(bufs), H, W, Cc, DTYPE_CODE[bufs[0].dtype], nb
            d.layers, d.nlayers, d.flags, d.max_ctas = arr, len(part), flags.data_ptr(), int(max_ctas)
            _check(self.lib, self.lib.rv_conv_chain(C.byref(d), self._stream()), 'rv_conv_chain')

    def dcn3x3(self, layer, x, om, out, act=ACT_NONE):
        """modulated deformable 3x3 conv (rv_dcn3x3): `layer` = packing.pack_dcn(...), x (H, W, 64), om (H, W, >= 216) fp32 raw
        conv_offset output, out (H, W, >= cout) in x's dtype"""
        assert (layer.kh, layer.kw, layer.alloc0, layer.alloc1) == (3, 3, 64, 0), f'{layer.name}: not a 64-channel 3x3 DCN'
        assert layer.impl != IMPL_TC or layer.layout == 1, f'{layer.name}: the tensor-core DCN reads the layout-1 image ([9][nb][64])'
        _chk_dev(x, om, out)
        H, W, Cc = x.shape
        assert Cc == 64, f'{layer.name}: x has {Cc} channels, the DCN reads 64'
        assert om.dtype == torch.float32 and tuple(om.shape[:2]) == (H, W) and tuple(out.shape[:2]) == (H, W)
        assert out.dtype == x.dtype
        _check(self.lib, self.lib.rv_dcn3x3(_ptr(x), _ptr(om), om.shape[2], H, W, DTYPE_CODE[x.dtype], _ptr(layer.wpack),
                                            _ptr(layer.bias), layer.cout, layer.nb, act, layer.impl, _ptr(out), out.shape[2],
                                            self._stream()), f'rv_dcn3x3[{layer.name}]')

    def space_to_depth2(self, src, out):
        _chk_dev(src, out)
        _check(self.lib, self.lib.rv_space_to_depth2(_ptr(src), src.shape[0], src.shape[1], src.shape[2],
                                                     DTYPE_CODE[src.dtype], _ptr(out), self._stream()),
               'rv_space_to_depth2')

    # -- image / pyramid prep ---------------------------------------------------------------------
    def prep_image(self, src, out, mat12=None, pool2=False):
        _chk_dev(src, out)
        H, W = src.shape[1], src.shape[2]
        m = None
        if mat12 is not None:
            m = (C.c_float * 12)(*[float(v) for v in mat12])
        _check(self.lib, self.lib.rv_prep_image(_ptr(src), H, W, m, int(pool2), _ptr(out), out.shape[2],
                                                DTYPE_CODE[out.dtype], self._stream()), 'rv_prep_image')

    def spynet_resize_norm(self, src, out):
        _chk_dev(src, out)
        _check(self.lib, self.lib.rv_spynet_resize_norm(_ptr(src), src.shape[1], src.shape[2], _ptr(out),
                                                        out.shape[0], out.shape[1], self._stream()),
               'rv_spynet_resize_norm')

    def avgpool2(self, src, out):
        _chk_dev(src, out)
        _check(self.lib, self.lib.rv_avgpool2(_ptr(src), src.shape[0], src.shape[1], src.shape[2], _ptr(out),
                                              self._stream()), 'rv_avgpool2')

    def maxpool2(self, src, out):
        """NHWC (H,W,C) -> (H/2,W/2,C) 2x2 max (vgg19.features[4], flag_HD_in matching)"""
        _chk_dev(src, out)
        assert src.dtype == out.dtype and tuple(out.shape) == (src.shape[0] // 2, src.shape[1] // 2, src.shape[2])
        _check(self.lib, self.lib.rv_maxpool2(_ptr(src), src.shape[0], src.shape[1], src.shape[2], DTYPE_CODE[src.dtype],
                                              _ptr(out), self._stream()), 'rv_maxpool2')

    def resize_planes(self, src, out, inv_scale, mode='bicubic', clamp01=False):
        """planar fp32 (n,H,W) -> (n,Ho,Wo): F.interpolate(scale_factor=1/inv_scale, mode=bicubic|nearest) [+ clamp(0,1)]"""
        _chk_dev(src, out)
        assert src.dtype == out.dtype == torch.float32 and src.dim() == 3 and out.dim() == 3 and src.shape[0] == out.shape[0]
        _check(self.lib, self.lib.rv_resize_planes(_ptr(src), src.shape[0], src.shape[1], src.shape[2], float(inv_scale),
                                                   out.shape[1], out.shape[2], 0 if mode == 'bicubic' else 1,
                                                   int(clamp01), _ptr(out), self._stream()), 'rv_resize_planes')

    def spynet_level_input(self, ref, supp, flow_prev, out8, flow_up):
        _chk_dev(ref, supp, flow_prev, out8, flow_up)
        _check(self.lib, self.lib.rv_spynet_level_input(_ptr(ref), _ptr(supp), _ptr(flow_prev), ref.shape[0],
                                                        ref.shape[1], _ptr(out8), DTYPE_CODE[out8.dtype],
                                                        _ptr(flow_up), self._stream()), 'rv_spynet_level_input')

    def flow_resize(self, flow, out):
        _chk_dev(flow, out)
        _check(self.lib, self.lib.rv_flow_resize(_ptr(flow), flow.shape[0], flow.shape[1], _ptr(out),
                                                 out.shape[0], out.shape[1], self._stream()), 'rv_flow_resize')

    # -- warp -------------------------------------------------------------------------------------
    def warp(self, src, flow, out, flow_up2=False):
        _chk_dev(src, flow, out)
        if src.dim() == 2:
            Hi, Wi, Cc = src.shape[0], src.shape[1], 1
        else:
            Hi, Wi, Cc = src.shape
        _check(self.lib, self.lib.rv_warp(_ptr(src), Hi, Wi, Cc, DTYPE_CODE[src.dtype], _ptr(flow), flow.shape[0],
                                          flow.shape[1], int(flow_up2), _ptr(out), self._stream()), 'rv_warp')

    def warp3(self, feat, featUP, conf, flow, out_feat, out_featUP, out_conf):
        """the three warps of one propagation step in one launch (16-bit features)"""
        _chk_dev(feat, featUP, conf, flow, out_feat, out_featUP, out_conf)
        h, w, Cc = feat.shape
        assert tuple(featUP.shape) == (2 * h, 2 * w, Cc) and tuple(conf.shape) == (h, w) and tuple(flow.shape) == (h, w, 2)
        assert feat.dtype == featUP.dtype == out_feat.dtype == out_featUP.dtype and conf.dtype == torch.float32
        _check(self.lib, self.lib.rv_warp3(_ptr(feat), _ptr(featUP), _ptr(conf), _ptr(flow), h, w, Cc, DTYPE_CODE[feat.dtype],
                                           _ptr(out_feat), _ptr(out_featUP), _ptr(out_conf), self._stream()), 'rv_warp3')

    # -- matching ---------------------------------------------------------------------------------
    def patch_pack(self, feat, out, mode):
        _chk_dev(feat, out)
        _check(self.lib, self.lib.rv_patch_pack(_ptr(feat), feat.shape[0], feat.shape[1], feat.shape[2],
                                                DTYPE_CODE[feat.dtype], mode, _ptr(out), out.shape[1],
                                                self._stream()), 'rv_patch_pack')

    def match_argmax(self, A, B, conf, idx, impl=1):
        _chk_dev(A, B, conf, idx)
        assert A.dtype == torch.float16 and B.dtype == torch.float16 and idx.dtype == torch.int32
        _check(self.lib, self.lib.rv_match_argmax(_ptr(A), A.shape[0], _ptr(B), B.shape[0], A.shape[1],
                                                  1.0 / 4096.0, _ptr(conf), _ptr(idx), impl, self._stream()),
               'rv_match_argmax')

    # -- reference alignment ----------------------------------------------------------------------
    def gather_blocks(self, value, idx, hq, wq, ks, out):
        _chk_dev(value, idx, out)
        _check(self.lib, self.lib.rv_gather_blocks(_ptr(value), value.shape[0], value.shape[1], value.shape[2],
                                                   DTYPE_CODE[value.dtype], _ptr(idx), hq, wq, ks, _ptr(out),
                                                   self._stream()), 'rv_gather_blocks')

    def aligned_sample(self, x, affine, ks, out):
        _chk_dev(x, affine, out)
        h, w = affine.shape[0], affine.shape[1]
        _check(self.lib, self.lib.rv_aligned_sample(_ptr(x), h, w, ks, x.shape[2], DTYPE_CODE[x.dtype],
                                                    _ptr(affine), _ptr(out), self._stream()), 'rv_aligned_sample')

    def bicubic_up2_image(self, src, out):
        _chk_dev(src, out)
        _check(self.lib, self.lib.rv_bicubic_up2_image(_ptr(src), src.shape[1], src.shape[2], _ptr(out),
                                                       out.shape[2], DTYPE_CODE[out.dtype], self._stream()),
               'rv_bicubic_up2_image')

    # -- confidence maps --------------------------------------------------------------------------
    def conf_pair(self, a, b, out, up2=False):
        _chk_dev(a, b, out)
        _check(self.lib, self.lib.rv_conf_pair(_ptr(a), _ptr(b), a.shape[0], a.shape[1], int(up2), _ptr(out),
                                               out.shape[2], DTYPE_CODE[out.dtype], self._stream()), 'rv_conf_pair')

    def conf_max(self, a, b, out):
        _chk_dev(a, b, out)
        _check(self.lib, self.lib.rv_conf_max(_ptr(a), _ptr(b), _ptr(out), a.numel(), self._stream()), 'rv_conf_max')

    def frames_differ(self, pairs, flag):
        """pairs: [(a, b)] contiguous same-size CUDA tensors; flag (1,) int32, zeroed here, set non-zero iff any pair differs"""
        n = len(pairs)
        assert 0 < n <= 16
        for a, b in pairs:
            _chk_dev(a, b)
            assert a.numel() * a.element_size() == b.numel() * b.element_size() and a.dtype == b.dtype
        pa = (C.c_void_p * n)(*[a.data_ptr() for a, _ in pairs])
        pb = (C.c_void_p * n)(*[b.data_ptr() for _, b in pairs])
        nb = (C.c_uint64 * n)(*[a.numel() * a.element_size() for a, _ in pairs])
        flag.zero_()
        _check(self.lib, self.lib.rv_frames_differ(pa, pb, nb, n, _ptr(flag), self._stream()), 'rv_frames_differ')

    # -- tail -------------------------------------------------------------------------------------
    def reconstruct(self, x, lr, scale, clamp01, out):
        _chk_dev(x, lr, out)
        _check(self.lib, self.lib.rv_reconstruct(_ptr(x), x.shape[2], DTYPE_CODE[x.dtype], _ptr(lr), lr.shape[1],
                                                 lr.shape[2], scale, int(clamp01), _ptr(out), self._stream()),
               'rv_reconstruct')
