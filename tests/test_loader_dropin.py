"""Drop-in `data_loader` (decoded-frame cache): the reference's own Test_datasets returns bit-identical items with
and without it, and decodes each file once per stream instead of T times.  Needs the reference copy that build()
stages under oracle/_ref (oracle/build_ref.py); skips where none is staged."""
import json
import os
import subprocess
import sys

import pytest

from oracle.build_ref import ref_root

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = ref_root()

CODE = r'''
import sys, os, json, hashlib, time
import numpy as np
from PIL import Image
root, tmp, use_dropin, ref_root = sys.argv[1], sys.argv[2], sys.argv[3] == '1', sys.argv[4]
sys.path[:0] = ([os.path.join(root, 'refvsr_b200', 'dropin')] if use_dropin else []) + [os.path.join(root, 'oracle', 'shims'), ref_root, root]
import importlib
cfg = importlib.import_module('configs.config_RefVSR_small_MFID').get_config('p', 'm', 'config_RefVSR_small_MFID')
cfg.dist = False
cfg.frame_num = 5
for k, sub in (('LR_data_path', 'LR'), ('HR_data_path', 'HR'), ('HR_ref_data_W_path', 'HR'), ('HR_ref_data_T_path', 'HR')):
    cfg.EVAL[k] = os.path.join(tmp, sub)
cfg.UW_path, cfg.W_path, cfg.T_path = 'UW', 'W', 'T'
cfg.EVAL.vid_name = None
from data_loader.datasets import Test_datasets
import data_loader.utils as U
import data_loader.datasets as D
ds = Test_datasets(cfg, is_valid=False)
t0 = time.perf_counter()
for i in range(len(ds)):            # timed pass: what an evaluation loop pays per item
    it = ds[i]
dt = time.perf_counter() - t0
first_pass = (dict(getattr(U, 'stats', None) or {}), dict(getattr(D, 'stats', None) or {}))
h = hashlib.sha256()
meta = []
for i in range(len(ds)):            # second pass: content hash of every tensor of every item
    it = ds[i]
    for k in ('LR_UW', 'LR_REF_W', 'LR_REF_T', 'HR_UW'):
        h.update(np.ascontiguousarray(it[k].numpy()).tobytes())
    meta.append([bool(it['is_first']), int(it['frame_idx']), it['video_name'], it['frame_name'], list(it['LR_UW'].shape)])
print(json.dumps({'sha': h.hexdigest(), 'meta': meta, 'items': len(ds), 'seconds': dt,
                  'stats': first_pass[0] or None, 'tensor_stats': first_pass[1] or None, 'utils_file': U.__file__,
                  'keys': sorted(it.keys()), 'types': {k: type(v).__name__ for k, v in it.items()}}))
'''


def _make_clip(tmp):
    import numpy as np
    from PIL import Image
    rng = np.random.default_rng(7)
    for vid, n in (('0001', 6), ('0002', 4)):
        for sub, stream, (h, w) in (('LR', 'UW', (36, 48)), ('LR', 'W', (36, 48)), ('LR', 'T', (36, 48)),
                                    ('HR', 'UW', (144, 192)), ('HR', 'W', (144, 192)), ('HR', 'T', (144, 192))):
            d = os.path.join(tmp, sub, stream, vid)
            os.makedirs(d, exist_ok=True)
            for k in range(n):
                Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(os.path.join(d, f'{k:04d}.png'))


@pytest.mark.skipif(REF is None, reason='no reference copy staged under oracle/_ref')
def test_cached_loader_returns_identical_items(tmp_path):
    _make_clip(str(tmp_path))
    out = {}
    for flag in ('0', '1'):
        r = subprocess.run([sys.executable, '-c', CODE, ROOT, str(tmp_path), flag, REF], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        out[flag] = json.loads(r.stdout.strip().splitlines()[-1])
    ref, ours = out['0'], out['1']
    assert ref['utils_file'].startswith(REF) and 'dropin' in ours['utils_file']
    assert ours['items'] == ref['items'] == 10
    assert ours['meta'] == ref['meta']
    assert ours['sha'] == ref['sha'], 'every tensor of every item must be bit-identical'
    assert ours['keys'] == ref['keys'] and ours['types'] == ref['types']
    # 10 files x 3 streams (LR, Ref-W, ground truth) are decoded once = 30, instead of 10 items x 5 frames x 4 streams
    # = 200 in the reference (which also decodes the Ref-T stream and then discards it, data_loader/utils.py:103)
    assert ours['tensor_stats']['misses'] == 30
    assert ours['tensor_stats']['hits'] == 10 * 5 * 3 - 30
