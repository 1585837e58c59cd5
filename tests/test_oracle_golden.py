"""Pins the oracle against the committed golden vectors generated from the UNMODIFIED reference
(tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from util import CASES, GOLDEN_DIR, build_case


@pytest.mark.parametrize('name', list(CASES))
def test_oracle_matches_reference_golden(name):
    from oracle.refvsr_oracle import OracleRefVSR
    from refvsr_b200.synth import sliding_windows
    spec, cfg, net, lrs, refs, golden = build_case(name, 'cpu')
    orc = OracleRefVSR(cfg, net.state_dict())
    for k, wl, wr, first in sliding_windows(lrs, refs, spec['T']):
        orc.trace = {} if k == 0 else None
        out = orc.forward(wl, wr, first)
        err = np.abs(out[0].numpy() - golden[f'result_{k}']).max()
        assert err < 5e-6, f'{name} window {k}: oracle differs from the reference by {err:.2e}'
        if k == 0:
            T = spec['T']
            fl = golden['flows_0']            # reference call order: forward j=0..T-2, then backward j=T-1..1
            for j, f in orc.trace['fw'].items():
                assert np.abs(f[0].numpy() - fl[j]).max() < 1e-4
            for j, f in orc.trace['bw'].items():
                assert np.abs(f[0].numpy() - fl[(T - 1) + (T - 2 - j)]).max() < 1e-4
            for i, c in orc.trace['conf'].items():
                assert np.abs(c[0].numpy() - golden['conf_0'][i]).max() < 1e-5
                assert (orc.trace['idx'][i][0].numpy() != golden['idx_0'][i]).mean() == 0.0
    assert orc.frame_itr_num >= 1


def test_golden_generator_is_committed_and_current():
    src = open(os.path.join(GOLDEN_DIR, 'make_golden.py')).read()
    for name, spec in CASES.items():
        assert name in src and os.path.isfile(os.path.join(GOLDEN_DIR, name + '.npz'))
        meta = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))['meta']
        assert list(meta) == [spec['T'], spec['h'], spec['w'], spec['ref_scale'], spec['frames'], spec['seed']]


def test_oracle_matches_live_reference():
    """a shape / seed outside CASES against the reference's results stored by make_golden.py (a seeded sample of every
    window's result plus its mean and mean square)."""
    from oracle.refvsr_oracle import OracleRefVSR
    from refvsr_b200 import SRNet, get_config
    from refvsr_b200.modules import seeded_test_weights
    from refvsr_b200.synth import make_clip, sliding_windows
    golden = np.load(os.path.join(GOLDEN_DIR, 'live_small_mfid_t5_28x36.npz'))
    T, h, w, ref_scale, frames, seed = (int(v) for v in golden['meta'])
    cfg = get_config('config_RefVSR_small_MFID', device='cpu', num_blocks=2)
    net = SRNet(cfg).eval()
    seeded_test_weights(net, seed=seed)
    orc = OracleRefVSR(cfg, net.state_dict())
    lrs, refs = make_clip(frames, h, w, ref_scale, seed=seed)
    idx = torch.from_numpy(golden['sample_idx']).long()
    worst, windows = 0.0, 0
    for k, wl, wr, first in sliding_windows(lrs, refs, T):
        b = orc.forward(wl, wr, first)[0].double().flatten()
        worst = max(worst, float(np.abs(b[idx].numpy() - golden[f'sample_{k}']).max()))
        mean, mean_sq = golden[f'moments_{k}']
        worst = max(worst, abs(float(b.mean()) - mean), abs(float((b * b).mean()) - mean_sq))
        windows += 1
    assert windows == frames
    assert worst < 5e-6
