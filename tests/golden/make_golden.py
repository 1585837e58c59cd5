"""Generate golden vectors by running the UNMODIFIED reference (/root/reference) on CPU.

Run once in the build container (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
Writes tests/golden/<case>.npz.  Weights are NOT stored: they come from
refvsr_b200.modules.seeded_test_weights(seed) (deterministic CPU generator) and are loaded into the
reference with strict=True, so both implementations see identical parameters.
"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

CASES = {
    # name: dict(config, overrides, T, h, w, ref_scale, calls, seed)
    'small_t3_32x48': dict(config='config_RefVSR_small_L1', over=dict(num_blocks=3, reset_branch=2), T=3, h=32, w=48,
                           ref_scale=1, frames=4, seed=11),
    'mfid_t5_40x56_ref2x': dict(config='config_RefVSR_MFID', over=dict(num_blocks=2), T=5, h=40, w=56,
                                ref_scale=2, frames=3, seed=12),
    'small_t7_24x32': dict(config='config_RefVSR_small_MFID', over=dict(num_blocks=1), T=7, h=24, w=32,
                           ref_scale=1, frames=5, seed=13),
    # flag_HD_in ("8K") configs: VGG[0:7] matching at 1/4 resolution, matching_ksize 8, aa1 scale 4 / aa2 scale 8
    'small8k_t3_32x48': dict(config='config_RefVSR_small_MFID_8K', over=dict(num_blocks=1, reset_branch=2), T=3, h=32, w=48,
                             ref_scale=1, frames=5, seed=21),
    'mfid8k_t5_48x64_noreset': dict(config='config_RefVSR_MFID_8K', over=dict(num_blocks=1), T=5, h=48, w=64,
                                    ref_scale=1, frames=3, seed=22),
}


def load_reference():
    import torchvision
    sys.path[:0] = [os.path.join(ROOT, 'oracle', 'shims'), '/root/reference']
    _vgg19 = torchvision.models.vgg19
    torchvision.models.vgg19 = lambda pretrained=False, **kw: _vgg19(weights=None)   # attention.py:28 wants a download
    from models.SRNet import SRNet                      # the reference's own class
    return SRNet


def build_case(name, spec, RefSRNet):
    from refvsr_b200.modules import seeded_test_weights
    from refvsr_b200.synth import make_clip, sliding_windows
    cfg = importlib.import_module('configs.' + spec['config']).get_config('p', 'm', spec['config'])
    cfg.cuda, cfg.device, cfg.dist = False, 'cpu', False
    for k, v in spec['over'].items():
        setattr(cfg, k, v)
    torch.manual_seed(0)
    ref = RefSRNet(cfg).eval()
    seeded_test_weights(ref, seed=spec['seed'])
    lrs, refs = make_clip(spec['frames'], spec['h'], spec['w'], spec['ref_scale'], seed=spec['seed'])
    out = {}
    rec = {}
    net = ref.Network
    orig_flow, orig_match = net.FlowNet.forward, net.feature_match.forward

    def flow_hook(a, b):
        r = orig_flow(a, b)
        rec.setdefault('flows', []).append(r.clone())
        return r

    def match_hook(lr, rf, *a, **k):
        conf, idx = orig_match(lr, rf, *a, **k)
        rec.setdefault('conf', []).append(conf.clone())
        rec.setdefault('idx', []).append(idx.clone())
        return conf, idx

    net.FlowNet.forward = flow_hook
    net.feature_match.forward = match_hook
    with torch.no_grad():
        for k, wl, wr, first in sliding_windows(lrs, refs, spec['T']):
            rec.clear()
            res = ref(wl, wr, first, False, False)['result']
            out[f'result_{k}'] = res[0].numpy().astype(np.float32)
            if k == 0:
                # first window: 2(T-1) flows in reference order (forward j=0.., then backward j=T-1..1)
                out['flows_0'] = torch.cat(rec['flows'], 0).numpy().astype(np.float32)
                out['conf_0'] = torch.cat(rec['conf'], 0).numpy().astype(np.float32)
                out['idx_0'] = torch.cat(rec['idx'], 0).numpy().astype(np.int32)
    out['meta'] = np.array([spec['T'], spec['h'], spec['w'], spec['ref_scale'], spec['frames'], spec['seed']])
    path = os.path.join(ROOT, 'tests', 'golden', name + '.npz')
    np.savez_compressed(path, **out)
    print(name, 'written', os.path.getsize(path) // 1024, 'KiB')


# tests/test_oracle_golden.py::test_oracle_matches_live_reference: a shape / seed outside CASES.  A full result per window
# would make a large file, so a seeded sample of each result is stored, with its mean and mean square.
LIVE = dict(config='config_RefVSR_small_MFID', over=dict(num_blocks=2), T=5, h=28, w=36, ref_scale=1, frames=3, seed=77)
LIVE_NAME, LIVE_SAMPLES = 'live_small_mfid_t5_28x36', 4096


def build_live(RefSRNet):
    from refvsr_b200.modules import seeded_test_weights
    from refvsr_b200.synth import make_clip, sliding_windows
    spec = LIVE
    cfg = importlib.import_module('configs.' + spec['config']).get_config('p', 'm', spec['config'])
    cfg.cuda, cfg.device, cfg.dist = False, 'cpu', False
    for k, v in spec['over'].items():
        setattr(cfg, k, v)
    ref = RefSRNet(cfg).eval()
    seeded_test_weights(ref, seed=spec['seed'])
    lrs, refs = make_clip(spec['frames'], spec['h'], spec['w'], spec['ref_scale'], seed=spec['seed'])
    n = 3 * 16 * spec['h'] * spec['w']
    out = {'sample_idx': np.sort(np.random.default_rng(spec['seed']).choice(n, LIVE_SAMPLES, replace=False)).astype(np.int32)}
    with torch.no_grad():
        for k, wl, wr, first in sliding_windows(lrs, refs, spec['T']):
            res = ref(wl, wr, first, False, False)['result'][0].double().flatten()
            out[f'sample_{k}'] = res[torch.from_numpy(out['sample_idx']).long()].numpy().astype(np.float32)
            out[f'moments_{k}'] = np.array([float(res.mean()), float((res * res).mean())])
    out['meta'] = np.array([spec['T'], spec['h'], spec['w'], spec['ref_scale'], spec['frames'], spec['seed']])
    path = os.path.join(ROOT, 'tests', 'golden', LIVE_NAME + '.npz')
    np.savez_compressed(path, **out)
    print(LIVE_NAME, 'written', os.path.getsize(path) // 1024, 'KiB')


if __name__ == '__main__':
    RefSRNet = load_reference()
    for name, spec in CASES.items():
        if len(sys.argv) > 1 and name not in sys.argv[1:]:
            continue
        build_case(name, spec, RefSRNet)
    if len(sys.argv) == 1 or LIVE_NAME in sys.argv[1:]:
        build_live(RefSRNet)
