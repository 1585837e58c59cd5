"""TEST / BENCH INFRASTRUCTURE - imports the UNMODIFIED reference (codeslake/RefVSR) as a Python package tree.

Source: the byte-for-byte copy build() stages under oracle/_ref/RefVSR (oracle/build_ref.py).  Third-party packages
the reference imports but this image lacks (mmcv, easydict, termcolor) come from oracle/shims.  Only tests/, bench.py's
reference / eager_b200 / cpu_baseline legs and __graft_entry__.smoke() may use this.
"""
import importlib
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_loaded = {}


def reference_srnet_class():
    """the reference's own `models.SRNet.SRNet` (None when no checkout is available)"""
    if 'cls' in _loaded:
        return _loaded['cls']
    from .build_ref import ref_root
    root = ref_root()
    if root is None:
        _loaded['cls'] = None
        return None
    import torchvision
    for p in (root, os.path.join(_HERE, 'shims')):
        if p not in sys.path:
            sys.path.insert(0, p)
    if not getattr(torchvision.models.vgg19, '_refvsr_patched', False):
        _vgg19 = torchvision.models.vgg19

        def vgg19(pretrained=False, **kw):                 # attention.py:28 asks for a download; weights come from the state_dict
            return _vgg19(weights=None)
        vgg19._refvsr_patched = True
        torchvision.models.vgg19 = vgg19
    from models.SRNet import SRNet                         # noqa: E402  (the reference's class)
    _loaded['cls'], _loaded['root'] = SRNet, root
    return SRNet


def reference_root():
    reference_srnet_class()
    return _loaded.get('root')


def build_reference(config_name, device='cpu', seed=1234, **overrides):
    """reference SRNet(config) in eval mode on `device` with refvsr_b200.modules.seeded_test_weights(seed) loaded"""
    import torch
    from refvsr_b200.modules import seeded_test_weights
    cls = reference_srnet_class()
    if cls is None:
        raise RuntimeError('no reference copy staged under oracle/_ref/RefVSR (python oracle/build_ref.py)')
    cfg = importlib.import_module('configs.' + config_name).get_config('p', 'm', config_name)
    is_cuda = str(device).startswith('cuda')
    cfg.cuda, cfg.device, cfg.dist = is_cuda, ('cuda' if is_cuda else 'cpu'), False      # run.py:399-405
    for k, v in overrides.items():
        setattr(cfg, k, v)
    torch.manual_seed(0)
    net = cls(cfg).eval()
    seeded_test_weights(net, seed=seed)
    return cfg, net.to(device)


def prime_steady_state(net, h, w, device, seed=7):
    """Put a reference network into the state it has after a first window WITHOUT computing one (CPU timing legs only: a first
    window at 270x480 costs minutes): random propagated state of the right shapes, frame counter at 1.  The cost of the
    following steady window does not depend on the values (RefVSR.py:256-260)."""
    import torch
    N = net.Network
    C = N.mid_channels if hasattr(N, 'mid_channels') else N.config.mid_channels
    g = torch.Generator().manual_seed(seed)
    N.forward_feat_prop_prev = torch.randn(1, C, h, w, generator=g).to(device) * 0.1
    N.forward_feat_prop_UP_prev = torch.randn(1, C, 2 * h, 2 * w, generator=g).to(device) * 0.1
    N.forward_conf_map_prop_prev = torch.rand(1, 1, h, w, generator=g).to(device)
    N.forward_flow_prev = torch.randn(1, 2, h, w, generator=g).to(device)
    N.frame_itr_num = 1
