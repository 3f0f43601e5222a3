"""Compile the unmodified reference into oracle/_ref/ (git-ignored).

    python oracle/fetch_ref.py [reference checkout]

The reference (RaptorMai/online-continual-learning) is a plain Python tree without a setup.py, so its
build product is its bytecode: every *.py is compiled to a sourceless *.pyc at the same relative path
under oracle/_ref/, which Python imports directly.  No reference source enters the repository or
oracle/_ref/, and oracle/_ref/ never enters git history.  Nothing under oracle/_ref/ is imported by
the product (online-continual-learning_b200/); it is used by
  * bench.py --impl reference      (the reference's own agents on the host cores),
  * bench.py's reference_gpu figure (the same agents on cuda:0),
  * tests/test_gpu_dropin.py        (reference nn.Module + optimizer -> install() -> train_learner).
A manifest with the sha256 of every compiled file is written next to them so that a test can prove
the build is unmodified.  Where the checkout is absent, an existing oracle/_ref/ is kept as it is.
"""
import hashlib
import json
import os
import py_compile
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, '_ref')
SKIP_DIRS = {'.git', '__pycache__', 'config', 'config_CVPR'}


def fetch(src='/root/reference', quiet=False):
    if not os.path.isdir(src):
        if not quiet:
            print('fetch_ref: %s not present -- keeping existing %s' % (src, DST))
        return os.path.isdir(DST)
    manifest = {}
    for root, dirs, files in os.walk(src):
        dirs[:] = [d for d in dirs if d not in SKIP_DIRS]
        rel = os.path.relpath(root, src)
        for f in files:
            if not f.endswith('.py'):
                continue
            s = os.path.join(root, f)
            d = os.path.normpath(os.path.join(DST, rel, f + 'c'))
            os.makedirs(os.path.dirname(d), exist_ok=True)
            py_compile.compile(s, cfile=d, dfile=os.path.normpath(os.path.join(rel, f)), doraise=True,
                               invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
            with open(d, 'rb') as fh:
                manifest[os.path.relpath(d, DST)] = hashlib.sha256(fh.read()).hexdigest()
    with open(os.path.join(DST, 'MANIFEST.json'), 'w') as fh:
        json.dump({'files': manifest}, fh, indent=1, sort_keys=True)
    if not quiet:
        print('fetch_ref: %d files -> %s' % (len(manifest), DST))
    return True


def verify():
    """True when every file listed in the manifest is present and byte-identical to what was compiled."""
    path = os.path.join(DST, 'MANIFEST.json')
    if not os.path.exists(path):
        return False
    with open(path) as fh:
        files = json.load(fh)['files']
    for rel, digest in files.items():
        p = os.path.join(DST, rel)
        if not os.path.exists(p) or hashlib.sha256(open(p, 'rb').read()).hexdigest() != digest:
            return False
    return bool(files)


if __name__ == '__main__':
    ok = fetch(sys.argv[1]) if len(sys.argv) > 1 else fetch()
    sys.exit(0 if ok and verify() else 1)
