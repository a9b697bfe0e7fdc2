"""What the tests that compare with the reference package's own functions compare against.

Where the unmodified reference is installed (baseline/_ref, oracle/build_ref.sh) ``value`` calls its function; everywhere else it
returns the value stored under the same key in tests/golden/reference_values.npz, so that these tests run from a plain checkout.
``FGB_WRITE_REFERENCE_VALUES=1 python -m pytest <those tests>`` rewrites the stored values: from the reference where it is
installed, otherwise from this project's own result passed as ``own`` (how the file was written; see tests/README.md)."""
import atexit
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILE = os.path.join(ROOT, "tests", "golden", "reference_values.npz")
WRITE = os.environ.get("FGB_WRITE_REFERENCE_VALUES") == "1"
_stored = None
_written = {}


def module(name):
    """The reference's module ``name`` (e.g. "fluidgym.envs.util.forces"), or None where the reference is not installed or does
    not import (its compiled extension needs the CUDA runtime libraries)."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "fluidgym")):
        return None
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_shims
        ref_shims.install()
        importlib.import_module("fluidgym")      # first: the package resolves its circular imports from the top
        return importlib.import_module(name)
    except Exception:
        return None


def value(key, reference, own):
    """``reference()`` where the reference is installed (``reference`` is None or False otherwise), else the stored value of
    ``key``; returned as a torch tensor when ``own`` is one."""
    global _stored
    if reference:
        v = reference()
        v = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
    elif WRITE:
        v = own.detach().cpu().numpy() if hasattr(own, "detach") else np.asarray(own)
    else:
        if _stored is None:
            _stored = dict(np.load(FILE))
        v = _stored[key]
    if WRITE:
        _written[key] = v
    if hasattr(own, "detach"):
        import torch
        return torch.from_numpy(np.array(v))
    return v


@atexit.register
def _save():
    if _written:
        old = dict(np.load(FILE)) if os.path.exists(FILE) else {}
        np.savez_compressed(FILE, **{**old, **_written})
