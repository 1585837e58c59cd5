"""The drop-in boundary, proven through the reference's OWN entry point: `python run.py --config ... ` (run.py:218-426 ->
eval.py -> evaluation/eval_qual_quan.py -> trainers/trainer.py::Trainer.evaluation -> models.SRNet) is executed twice on a
synthetic RealMCVSR-style tree - once unmodified, once with `<repo>/refvsr_b200/dropin` in front of the checkout on
PYTHONPATH (INTEGRATION.md section 1, verbatim) - and the per-frame PSNR / SSIM lines it prints must agree.

  * CPU (here): the drop-in's operator set is the oracle test double (injected by tests/runpy_env/sitecustomize.py, never
    by the product), fp32 -> agreement to 1e-4 dB.  Checks: package shadowing (models.utils / models.loss / models.archs.*
    still come from the reference), SRNet ctor / state_dict schema through CKPT_Manager.load_ckpt, forward contract,
    the data_loader drop-in, is_first handling across two videos.
  * GPU (-m gpu): the real CUDA path under DataParallel, the ptflops init forward, and autocast, against the unmodified
    reference in eager PyTorch on the same GPU (staged copy oracle/_ref/RefVSR).  Bar: |dPSNR| < 0.01 dB (north_star).
The reference checkout is the copy build() stages under oracle/_ref (oracle/build_ref.py); without one these tests skip."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ENV_DIR = os.path.join(ROOT, 'tests', 'runpy_env')
SHIMS = os.path.join(ROOT, 'oracle', 'shims')


def _ref_root():
    from oracle.build_ref import ref_root
    return ref_root()


def make_tree(root, h, w, videos=2, frames=3, seed=5):
    """<root>/RealMCVSR/test/{LRx4,LRx2,HR}/{UW,W,T}/<vid>/<frame>.png  (README.md:49-65, configs/config.py:120-152)"""
    import cv2
    from refvsr_b200.synth import make_clip
    for v in range(videos):
        # ground truth = the HR scene the LR frames were area-downsampled from (NOT bicubic(LR): with GT == the network's own
        # bicubic base the printed PSNR would measure nothing but the residual branch and amplify any difference in it)
        lrs, refs, hr = make_clip(frames, h, w, 1, seed=seed + v, return_hr=True)
        x2 = torch.nn.functional.interpolate(lrs, scale_factor=2, mode='bicubic', align_corners=False).clamp(0, 1)
        for res, uw, wide in (('LRx4', lrs, refs), ('LRx2', x2, x2), ('HR', hr, hr)):
            for cam, t in (('UW', uw), ('W', wide), ('T', wide)):
                d = os.path.join(root, 'RealMCVSR', 'test', res, cam, f'{v:04d}')
                os.makedirs(d, exist_ok=True)
                for f in range(frames):
                    img = (t[f].permute(1, 2, 0).numpy() * 255.0 + 0.5).astype(np.uint8)
                    cv2.imwrite(os.path.join(d, f'{f:04d}.png'), cv2.cvtColor(img, cv2.COLOR_RGB2BGR))


def make_ckpt(path, config_name, **over):
    from refvsr_b200 import SRNet, get_config
    from refvsr_b200.modules import seeded_test_weights
    net = SRNet(get_config(config_name, device='cpu', **over))
    seeded_test_weights(net, seed=77)
    torch.save({'module.' + k: v for k, v in net.state_dict().items()}, path)     # ckpt_manager.py:50-60


def run_py(ref, tmp, tag, config, dropin, extra_env=None, cpu=True, frame_num=3, timeout=1500):
    out = os.path.join(tmp, 'out_' + tag)
    pp = [ENV_DIR] + ([os.path.join(ROOT, 'refvsr_b200', 'dropin'), ROOT] if dropin else [ROOT]) + [SHIMS]
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(pp), REFVSR_TEST_ENV='1', PYTHONDONTWRITEBYTECODE='1')
    env.update(extra_env or {})
    cmd = [sys.executable, '-B', 'run.py', '--mode', 'dropin_' + tag, '--project', os.path.join(tmp, 'logs_' + tag),
           '--config', config, '--data', 'RealMCVSR', '--ckpt_abs_name', os.path.join(tmp, 'ckpt.pytorch'),
           '--data_offset', os.path.join(tmp, 'data'), '--output_offset', out, '--frame_num', str(frame_num)]
    if cpu:
        cmd.append('-cpu')
    r = subprocess.run(cmd, cwd=ref, env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, f'run.py ({tag}) failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}'
    lines = re.findall(r'\[EVAL [^\]]*\]\[(\d+)/\d+\]\[(\d+)/\d+\] \S+ PSNR: ([-\d.naninf]+) SSIM: ([-\d.naninf]+)', r.stdout)
    assert 'All keys matched successfully' in r.stdout, r.stdout[-2000:]
    return [(int(a), int(b), float(p), float(s)) for a, b, p, s in lines], r.stdout


def test_reference_imports_resolve_through_the_dropin():
    """trainers/trainer.py:19-21 and models/SRNet.py:20-21 with INTEGRATION.md's sys.path order (ADVICE r1, high)"""
    ref = _ref_root()
    if ref is None:
        pytest.skip('no reference checkout (build oracle/_ref with oracle/build_ref.py)')
    code = ('import importlib, models, models.archs\n'
            'import models.utils, models.loss.Loss\n'
            'import trainers.trainer\n'
            'from models.SRNet import SRNet\n'
            'a = importlib.import_module("models.archs.RefVSR"); b = importlib.import_module("models.archs.RefVSR_IR") if False else None\n'
            'c = importlib.import_module("models.archs.SPyNet")\n'
            'import refvsr_b200\n'
            'assert SRNet is refvsr_b200.SRNet and a.Network is refvsr_b200.Network, (SRNet, a.Network)\n'
            'assert trainers.trainer.SRNet is refvsr_b200.SRNet\n'
            'assert "reference" in c.__file__ or "_ref" in c.__file__, c.__file__\n'
            'assert models.utils.__file__.startswith(%r), models.utils.__file__\n'
            'print("ok")\n' % ref)
    pp = [ENV_DIR, os.path.join(ROOT, 'refvsr_b200', 'dropin'), ROOT, SHIMS]
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(pp), REFVSR_TEST_ENV='1')
    r = subprocess.run([sys.executable, '-B', '-c', code], cwd=ref, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stdout + r.stderr


def test_run_py_eval_unmodified_vs_dropin_cpu(tmp_path):
    ref = _ref_root()
    if ref is None:
        pytest.skip('no reference checkout')
    tmp = str(tmp_path)
    make_tree(os.path.join(tmp, 'data'), 24, 32)
    make_ckpt(os.path.join(tmp, 'ckpt.pytorch'), 'config_RefVSR_small_L1')
    base, _ = run_py(ref, tmp, 'ref', 'config_RefVSR_small_L1', dropin=False)
    ours, log = run_py(ref, tmp, 'b200', 'config_RefVSR_small_L1', dropin=True, extra_env={'REFVSR_TEST_ORACLE_OPS': '1'})
    assert len(base) == 6 and [x[:2] for x in base] == [x[:2] for x in ours], (base, ours)
    for (v, f, p0, s0), (_, _, p1, s1) in zip(base, ours):
        assert abs(p0 - p1) <= 1e-4 and abs(s0 - s1) <= 1e-5, f'video {v} frame {f}: PSNR {p0} vs {p1}, SSIM {s0} vs {s1}'
    assert '[TOTAL' in log
    # the evaluation-loop drop-in (refvsr_b200/dropin/evaluation) writes the same image tree and score file as the reference's loop
    import cv2

    def tree(tag):
        root = os.path.join(tmp, 'out_' + tag)
        return {os.path.relpath(os.path.join(d, f), root).split(os.sep, 4)[-1] if False else
                re.sub(r'/\d{4}_\d{2}_\d{2}_\d{4}/', '/DATE/', os.path.relpath(os.path.join(d, f), root)): os.path.join(d, f)
                for d, _, fs in os.walk(root) for f in fs}
    ta, tb = tree('ref'), tree('b200')
    strip = lambda t, tag: {k.replace('dropin_' + tag, 'MODE'): v for k, v in t.items()}
    ta, tb = strip(ta, 'ref'), strip(tb, 'b200')
    assert set(ta) == set(tb) and sum(k.endswith('.png') for k in ta) == 12, sorted(set(ta) ^ set(tb))[:6]
    for k in ta:
        if k.endswith('.png'):
            assert np.abs(cv2.imread(ta[k]).astype(int) - cv2.imread(tb[k]).astype(int)).max() <= 1, k


@pytest.mark.gpu
@pytest.mark.parametrize('config,prec,frame_num', [('config_RefVSR_MFID', 'bf16', 7), ('config_RefVSR_small_MFID', None, 7)])
def test_run_py_eval_unmodified_vs_dropin_gpu(tmp_path, config, prec, frame_num):
    """the real thing: no -cpu => DataParallel wrap (trainer.py:67), ptflops forward at init (trainer.py:85-90), autocast for
    the small (is_amp) config (trainer.py:237-239); reference arm = the unmodified modules in eager PyTorch on the same GPU"""
    ref = _ref_root()
    if ref is None:
        pytest.skip('no reference checkout staged under oracle/_ref')
    tmp = str(tmp_path)
    make_tree(os.path.join(tmp, 'data'), 64, 96, videos=2, frames=4)
    make_ckpt(os.path.join(tmp, 'ckpt.pytorch'), config)
    base, _ = run_py(ref, tmp, 'ref', config, dropin=False, cpu=False, frame_num=frame_num)
    env = {'REFVSR_TEST_PRECISION': prec} if prec else {}
    ours, log = run_py(ref, tmp, 'b200', config, dropin=True, cpu=False, frame_num=frame_num, extra_env=env)
    assert len(base) == 8 and [x[:2] for x in base] == [x[:2] for x in ours]
    worst = max(abs(a[2] - b[2]) for a, b in zip(base, ours))
    print(f'{config}: max |dPSNR| vs the unmodified reference on the same GPU = {worst:.5f} dB over {len(base)} frames')
    assert worst < 0.01, (base, ours)
