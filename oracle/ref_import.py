"""Import the reference's own hot-path modules from a checkout of it (SKA_REFERENCE_ROOT).

The viz imports the reference pulls at module import (matplotlib, plotly; triangulation/vis/
pose_visualization.py:9,17-19 and vggt/vis/pose_visualization.py:10-11) may not be installed, so dummy
sys.modules entries are inserted first (SURVEY.md section 8c).  Used by make_golden.py and by tests
that compare with the checkout when one is present; signature_record() needs no checkout.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("SKA_REFERENCE_ROOT", "/root/reference")

_STUBS = [
    "matplotlib", "matplotlib.pyplot", "matplotlib.gridspec", "matplotlib.animation", "matplotlib.patches",
    "matplotlib.lines", "matplotlib.colors", "matplotlib.cm", "matplotlib.figure", "matplotlib.axes",
    "mpl_toolkits", "mpl_toolkits.mplot3d", "mpl_toolkits.mplot3d.art3d",
    "plotly", "plotly.graph_objs", "plotly.graph_objects", "plotly.offline", "plotly.subplots",
]


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "triangulation"))


class _Anything(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        obj = _Anything(f"{self.__name__}.{name}")
        setattr(self, name, obj)
        return obj

    def __call__(self, *a, **k):
        return _Anything(self.__name__ + "()")


def _install_stubs():
    for name in _STUBS:
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = _Anything(name)


def signature_record(fn) -> list:
    """The parameters of `fn` in order, as JSON-ready dicts: {"name"} when it has no default, {"name", "default"} when the
    default is an int / float / str / bool / None, {"name", "default_is_object": True} for any other default."""
    import inspect

    out = []
    for p in inspect.signature(fn).parameters.values():
        d = p.default
        if d is inspect.Parameter.empty:
            out.append({"name": p.name})
        elif isinstance(d, (int, float, str, bool, type(None))):
            out.append({"name": p.name, "default": d})
        else:
            out.append({"name": p.name, "default_is_object": True})
    return out


def load(module: str):
    """e.g. load('triangulation.triangulate') -> the reference module object."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REF_ROOT}")
    _install_stubs()
    sys.dont_write_bytecode = True
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    return importlib.import_module(module)
