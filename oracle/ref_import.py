"""Import the UNMODIFIED reference (awarebayes/RecNN) from a local checkout.

TEST INFRASTRUCTURE.  Only usable where a checkout of the reference exists
(``RECNN_REFERENCE_ROOT``); used by the generators of ``tests/golden/``
(``oracle/make_*golden.py``).  No test imports it.

Two modules the reference imports at package-import time are not installed
here and are off the hot path (SURVEY.md 8c): ``matplotlib`` (pulled in by
recnn/utils/plot.py:3) and ``torch_optimizer`` (recnn/nn/algo.py:6).  They are
replaced by empty stub modules in ``sys.modules``; no reference file is touched.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("RECNN_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "recnn", "__init__.py"))


def import_reference():
    """Returns the reference ``recnn`` package (imported once)."""
    if not reference_available():
        raise ImportError("reference tree not present at %s" % REFERENCE_ROOT)
    for name in ("matplotlib", "matplotlib.pyplot", "torch_optimizer"):
        if name not in sys.modules:
            try:
                __import__(name)
            except ImportError:
                mod = types.ModuleType(name)
                mod.__dict__["__stub__"] = True
                sys.modules[name] = mod
    if "matplotlib" in sys.modules and getattr(sys.modules["matplotlib"], "__stub__", False):
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    mod = sys.modules.get("recnn")
    if mod is not None and not os.path.abspath(getattr(mod, "__file__", "")).startswith(
            os.path.abspath(REFERENCE_ROOT)):
        raise ImportError("a different 'recnn' is already imported: %r" % mod)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import recnn  # noqa: E402  (the reference)
    return recnn
