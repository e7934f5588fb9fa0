"""Copies the upstream GAST-Net project's CALLER files (never its model/: that is what this repository replaces)
into oracle/_ref/, so that tests/test_unchanged_callers.py can run reconstruction.reconstruction() and main.train()
unchanged over the drop-in package on a machine that has no upstream checkout.  oracle/_ref/ is git-ignored: no
upstream source enters the history.

The upstream checkout is the first of $GAST_NET_REFERENCE, a directory named `reference` next to this repository, and
/root/reference (where the project's build environment keeps it, read-only) that holds reconstruction.py.  Without
one nothing is copied and an existing oracle/_ref/ is left as it is.  Called by __graft_entry__.build().
"""
import glob
import os
import shutil
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEST = os.path.join(REPO, 'oracle', '_ref')
FILES = ['reconstruction.py', 'main.py', 'tools/utils.py', 'tools/mpii_coco_h36m.py', 'tools/visualization.py',
         'data/keypoints/baseball.json', 'data/video/baseball.mp4']
# the drop-in owns these two modules of the `common` namespace package (same contract; the tests compare them)
SHADOWED = ('graph_utils.py', 'skeleton.py')


def upstream():
    for src in (os.environ.get('GAST_NET_REFERENCE'), os.path.join(os.path.dirname(REPO), 'reference'),
                '/root/reference'):
        if src and os.path.isfile(os.path.join(src, 'reconstruction.py')):
            return src
    return None


def copy_callers(src=None):
    """copy the caller files from `src` (default: upstream()); returns the destination, or None without a source"""
    src = src or upstream()
    if src is None:
        return None
    rel = list(FILES) + sorted(os.path.relpath(p, src) for p in glob.glob(os.path.join(src, 'common', '*.py'))
                               if os.path.basename(p) not in SHADOWED)
    tmp = DEST + '.tmp'
    shutil.rmtree(tmp, ignore_errors=True)
    for r in rel:
        os.makedirs(os.path.dirname(os.path.join(tmp, r)), exist_ok=True)
        shutil.copyfile(os.path.join(src, r), os.path.join(tmp, r))     # contents only: the copy stays writable
    shutil.rmtree(DEST, ignore_errors=True)
    os.replace(tmp, DEST)
    return DEST


if __name__ == '__main__':
    print('reference callers ->', copy_callers(sys.argv[1] if len(sys.argv) > 1 else None))
