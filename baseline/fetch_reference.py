"""Recipe for baseline/_ref: an UNMODIFIED copy of the reference's `code/` tree (plus LICENSE.md).

    python baseline/fetch_reference.py            # in the build container, where /root/reference exists

The reference (NVlabs/neuralrgbd) is pure Python with no setup.py / pyproject.toml, so there is nothing to
`pip install --target`: the "install" is a verbatim copy of its source tree (0.6 MB). baseline/_ref/ is git-ignored
(never part of this repo's history) but NOT gpurun-ignored, so it travels to the GPU box, where /root/reference
does not exist. It is used only by
  * bench.py --impl reference / --impl reference-gpu   (the reference's own KVNET.forward, timed beside the engine).
A MANIFEST with the sha256 of every copied file is written next to it so a reader can check nothing was edited.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get('NRGBD_REFERENCE', '/root/reference')
DST = os.path.join(HERE, '_ref')


def fetch(verbose=True):
    if not os.path.isdir(os.path.join(SRC, 'code')):
        if verbose:
            print('fetch_reference: %s not present (GPU box?) - keeping whatever is in %s' % (SRC, DST))
        return os.path.isdir(os.path.join(DST, 'code'))
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    os.makedirs(DST)
    shutil.copytree(os.path.join(SRC, 'code'), os.path.join(DST, 'code'),
                    ignore=shutil.ignore_patterns('__pycache__', '*.pyc'))
    for f in ('LICENSE.md', 'README.md'):
        if os.path.exists(os.path.join(SRC, f)):
            shutil.copy(os.path.join(SRC, f), os.path.join(DST, f))
    manifest = {}
    for root, _, files in os.walk(DST):
        for f in sorted(files):
            p = os.path.join(root, f)
            manifest[os.path.relpath(p, DST)] = hashlib.sha256(open(p, 'rb').read()).hexdigest()
    with open(os.path.join(DST, 'MANIFEST.json'), 'w') as fh:
        json.dump({'source': SRC, 'files': manifest}, fh, indent=1, sort_keys=True)
    if verbose:
        print('fetch_reference: copied %d files to %s' % (len(manifest), DST))
    return True


if __name__ == '__main__':
    sys.exit(0 if fetch() else 1)
