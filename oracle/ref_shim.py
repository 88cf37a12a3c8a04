"""Import the live reference (``/root/reference``) read-only under a harness shim.

TEST INFRASTRUCTURE ONLY: used by ``tests/golden/make_golden.py`` to produce the
committed ``tests/golden/live_*`` vectors, which the tests compare against.

The reference does not import as-is here (SURVEY.md section 8c): ``utils.py:1``
needs tkinter (``from turtle import position``), ``utils.py:3-4`` / ``plot.py:2,9``
need matplotlib, and ``truss.py:321`` uses ``np.bool8`` (removed in numpy 2).
The shim registers stub modules and the alias *before* importing; the reference
files themselves are untouched.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("TRUSS_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "slientruss3d"))


def _stub(name: str, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    mod = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(mod, k, v)
    sys.modules[name] = mod
    return mod


def load():
    """Return the reference's modules as a namespace: .truss .type .utils .ga .generate"""
    if not available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    import numpy as np

    if not hasattr(np, "bool8"):
        np.bool8 = np.bool_                      # truss.py:321

    _stub("turtle", position=None)               # utils.py:1
    try:
        import matplotlib  # noqa: F401
    except Exception:
        class _FancyArrowPatch:                  # utils.py:3,12,25
            def __init__(self, *a, **k):
                pass

        class _Style:
            @staticmethod
            def use(*a, **k):
                pass

        mpl = _stub("matplotlib")
        patches = _stub("matplotlib.patches", FancyArrowPatch=_FancyArrowPatch)
        pyplot = _stub("matplotlib.pyplot", style=_Style())   # plot.py:2,9
        mpl.patches, mpl.pyplot = patches, pyplot
        tk = _stub("mpl_toolkits")
        m3d = _stub("mpl_toolkits.mplot3d", proj3d=None)      # utils.py:4
        tk.mplot3d = m3d

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib

    ns = types.SimpleNamespace()
    ns.utils = importlib.import_module("slientruss3d.utils")
    ns.type = importlib.import_module("slientruss3d.type")
    ns.truss = importlib.import_module("slientruss3d.truss")
    ns.ga = importlib.import_module("slientruss3d.ga")
    ns.generate = importlib.import_module("slientruss3d.generate")
    return ns


def dense_results(truss):
    """Densify a solved reference Truss -> dict(u, ext, axial, weight) of lists."""
    import numpy as np

    dim, nj, nm = truss.dim, truss.nJoint, truss.nMember
    u = np.zeros((nj, dim))
    ext = np.zeros((nj, dim))
    ax = np.zeros(nm)
    for j, v in truss.GetDisplacements().items():
        u[j] = v
    for j, v in truss.GetExternalForces().items():
        ext[j] = v
    for m, v in truss.GetInternalForces().items():
        ax[m] = v
    return {"u": u.ravel(), "ext": ext.ravel(), "axial": ax, "weight": float(truss.weight)}
