"""Recipe: stage the UNMODIFIED reference (codeslake/RefVSR, /root/reference) under oracle/_ref/RefVSR.

The reference is pure Python with no setup.py / pyproject (SURVEY.md section 1), so `pip install --target` does not apply;
"building" it is copying its Python sources byte for byte.  oracle/_ref/ is git-ignored (reference sources never enter
this repository's history) but NOT gpurun-ignored, so the staged tree travels to the GPU box, where /root/reference does
not exist.  Consumers (test infrastructure and bench legs only - never the product):
  * bench.py --impl reference        the reference's own CPU forward on the box's host cores (kind "reference")
  * bench.py eager_b200 leg          the same unmodified modules in eager PyTorch on the B200
  * tests/test_dropin_runpy.py       run.py / eval.py / Trainer.evaluation with and without the drop-in
Missing third-party packages (mmcv, easydict, termcolor, ...) come from oracle/shims and tests/runpy_env.

    python oracle/build_ref.py            # idempotent; prints the number of files staged
"""
import filecmp
import os
import shutil
import sys

SRC = '/root/reference'
HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, '_ref', 'RefVSR')
KEEP_EXT = ('.py', '.txt', '.yaml', '.sh', '.md')


def build(src=SRC, dst=DST, verbose=True):
    if not os.path.isdir(src):
        if verbose:
            print(f'oracle/build_ref: {src} not present (GPU box): using the staged copy' if os.path.isdir(dst)
                  else f'oracle/build_ref: neither {src} nor {dst} exist')
        return os.path.isdir(dst)
    n = 0
    for root, dirs, files in os.walk(src):
        dirs[:] = [d for d in dirs if d not in ('.git', '__pycache__', 'ckpt')]
        rel = os.path.relpath(root, src)
        for f in files:
            if not f.endswith(KEEP_EXT):
                continue
            s, d = os.path.join(root, f), os.path.join(dst, rel, f)
            os.makedirs(os.path.dirname(d), exist_ok=True)
            if not (os.path.isfile(d) and filecmp.cmp(s, d, shallow=False)):
                shutil.copyfile(s, d)
            n += 1
    if verbose:
        print(f'oracle/build_ref: {n} files staged under {dst}')
    return True


def ref_root():
    """path of the staged reference copy (what build() made), None when nothing is staged"""
    if os.path.isfile(os.path.join(DST, 'models', 'SRNet.py')):
        return DST
    return None


if __name__ == '__main__':
    sys.exit(0 if build() else 1)
