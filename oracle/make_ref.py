#!/usr/bin/env python
"""Recipe: put the UNMODIFIED reference modules of the hot path under ``oracle/_ref/`` (test infrastructure).

``oracle/_ref/`` is git-ignored (reference sources never enter this repository's history) but NOT
gpurun-ignored, so the byte-identical files travel to the GPU box, where ``/root/reference`` does not exist.
``__graft_entry__.build()`` runs this in the build container; on the GPU box the prebuilt directory is used.

What is copied (verbatim, ``shutil.copyfile``; a SHA-256 manifest is written next to them):
  src/NPHM/__init__.py
  src/NPHM/models/{EnsembledDeepSDF,deepSDF,reconstruction,fitting,iterative_root_finding,diff_operators,loss_functions}.py
  src/NPHM/utils/reconstruction.py
  assets/{anchors_39,nphm_lat_mean,nphm_lat_std}.npy
Nothing else of the reference is needed for SURVEY.md section 8's path.  ``oracle/ref_loader.py`` imports them.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get('NPHM_REFERENCE_ROOT', '/root/reference')
DST = os.path.join(HERE, '_ref')

FILES = [
    'src/NPHM/__init__.py',
    'src/NPHM/models/EnsembledDeepSDF.py',
    'src/NPHM/models/deepSDF.py',
    'src/NPHM/models/reconstruction.py',
    'src/NPHM/models/fitting.py',
    'src/NPHM/models/iterative_root_finding.py',
    'src/NPHM/models/diff_operators.py',
    'src/NPHM/models/loss_functions.py',
    'src/NPHM/utils/reconstruction.py',
    'assets/anchors_39.npy',
    'assets/nphm_lat_mean.npy',
    'assets/nphm_lat_std.npy',
]


def main() -> int:
    if not os.path.isdir(REF):
        if os.path.exists(os.path.join(DST, 'MANIFEST.json')):
            print('make_ref: %s absent, keeping the prebuilt %s' % (REF, DST))
        else:
            # the suite compares against stored reference outputs (tests/golden); only bench.py's reference legs
            # and the golden generators need the modules themselves
            print('make_ref: %s not readable, no reference modules under %s' % (REF, DST))
        return 0
    manifest = {}
    for rel in FILES:
        src = os.path.join(REF, rel)
        dst = os.path.join(DST, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(src, dst)
        with open(dst, 'rb') as f:
            manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(DST, 'MANIFEST.json'), 'w') as f:
        json.dump({'source': REF, 'sha256': manifest}, f, indent=1, sort_keys=True)
    print('make_ref: %d reference files -> %s' % (len(FILES), DST))
    return 0


if __name__ == '__main__':
    sys.exit(main())
