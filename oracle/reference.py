"""Install the unmodified reference under ``oracle/_ref`` for bench.py's reference arm.

The reference is pure Python, so installing it is copying its ``spotlight`` package
from a checkout of it; ``__graft_entry__.build()`` does that from ``SLB_REFERENCE_SRC``,
or from ``DEFAULT_SRC`` when that variable is unset.  ``oracle/_ref`` is a build product
and stays out of git.
"""

import os
import shutil

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
DEFAULT_SRC = '/root/reference'


def source():
    """The reference checkout to install from: ``SLB_REFERENCE_SRC``, else ``DEFAULT_SRC``."""
    return os.environ.get('SLB_REFERENCE_SRC') or DEFAULT_SRC


def install(src, dst=REF_DIR):
    """Copy ``src/spotlight`` to ``dst/spotlight`` unless it is already there.  The copies
    are plain user-writable files whatever the modes of the checkout.  Returns whether
    ``dst`` holds the package afterwards: False when ``src`` has no readable package (the
    bench then times the torch restatement, oracle/torch_port.py, and says so)."""
    target = os.path.join(dst, 'spotlight')
    if os.path.isdir(target):
        return True
    pkg = os.path.join(src, 'spotlight')
    if not os.path.isdir(pkg):
        return False
    tmp = target + '.tmp'
    shutil.rmtree(tmp, ignore_errors=True)
    try:
        for dirpath, dirnames, files in os.walk(pkg, onerror=_raise):
            dirnames[:] = [d for d in dirnames if d != '__pycache__']
            out = os.path.join(tmp, os.path.relpath(dirpath, pkg))
            os.makedirs(out, exist_ok=True)
            for f in files:
                if not f.endswith('.pyc'):
                    shutil.copyfile(os.path.join(dirpath, f), os.path.join(out, f))
    except OSError:
        shutil.rmtree(tmp, ignore_errors=True)
        return False
    os.replace(tmp, target)
    return True


def _raise(err):
    raise err
