"""Make the reference's plugin base classes importable.

``CoreComponent`` / ``CoreConfig`` come from the real ``detectmatelibrary`` when it is
installed; otherwise a minimal stand-in (detectmateservice_b200/shims) is appended to
``sys.path`` -- appended, so a real installation always wins.  The same goes for ``pynng``
(the reference's transport, engine.py:2), whose SP/PAIR0 wire protocol the shim speaks
natively so mixed deployments interoperate.
"""
from __future__ import annotations

import importlib
import os
import sys
import tempfile

SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shims")


def ipc_tempdir(prefix: str = "dm") -> str:
    """A new directory for ``ipc://`` socket files.  An AF_UNIX address holds at most 107 bytes, which a deep
    $TMPDIR can leave no room for, so the directory is made under /tmp where that exists."""
    return tempfile.mkdtemp(prefix=prefix, dir="/tmp" if os.path.isdir("/tmp") else None)


def install_shims() -> dict:
    """Returns {"detectmatelibrary": "real"|"shim", "pynng": "real"|"shim"|"absent"}."""
    state = {}
    for mod, probe in (("detectmatelibrary", "detectmatelibrary.common.core"), ("pynng", "pynng")):
        try:
            m = importlib.import_module(probe)
            top = sys.modules[mod]
            state[mod] = "shim" if getattr(top, "__shim__", False) else "real"
            continue
        except ImportError:
            pass
        if SHIMS not in sys.path:
            sys.path.append(SHIMS)
        importlib.invalidate_caches()
        try:
            importlib.import_module(probe)
            state[mod] = "shim"
        except ImportError:
            state[mod] = "absent"
    return state
