"""TEST INFRASTRUCTURE ONLY -- import shim for the *unmodified* RatInABox reference.

Used by ``oracle/gen_golden.py`` (build container, /root/reference) to pin the
oracle restatement against the live reference, and -- through the copy that
``oracle/make_ref.py`` stages into the git-ignored ``oracle/_ref/`` -- by
``bench.py``'s CPU legs and ``tests/test_gpu_reference_binding.py`` on the GPU box.
Nothing in the product path imports this file.

The reference imports matplotlib and shapely at module top
(ratinabox/Environment.py:6-8, Agent.py:7-8, Neurons.py:7-12, utils.py:2-3).
Neither is installed in this image and there is no network, so we inject the
smallest stand-ins that let the hot path run:

* ``matplotlib`` / ``matplotlib.pyplot`` / ``.collections.EllipseCollection`` /
  ``.colors.to_rgba`` / ``.path.Path.contains_point`` / ``.colormaps``
* ``shapely.Polygon(v).contains(shapely.Point(p))`` with strict-interior
  semantics (what GEOS does for points) and ``.area``.

The hot path itself (Agent.update, Neurons.update/get_state, utils geometry)
runs unmodified from /root/reference.
"""
import sys
import types
import importlib

import os

REFERENCE_ROOT = "/root/reference"
STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")      # oracle/make_ref.py (travels to the GPU box)


def _polygon_contains_strict(verts, p):
    """Even-odd ray cast; points on an edge or vertex are NOT inside."""
    x, y = float(p[0]), float(p[1])
    n = len(verts)
    inside = False
    for i in range(n):
        x0, y0 = verts[i]
        x1, y1 = verts[(i + 1) % n]
        # on-edge test (exact): collinear and within the bounding box
        cross = (x1 - x0) * (y - y0) - (y1 - y0) * (x - x0)
        if cross == 0.0 and min(x0, x1) <= x <= max(x0, x1) and min(y0, y1) <= y <= max(y0, y1):
            return False
        if (y0 > y) != (y1 > y):
            xi = x0 + (y - y0) * (x1 - x0) / (y1 - y0)
            if x < xi:
                inside = not inside
    return inside


class _Point:
    def __init__(self, p):
        self.p = (float(p[0]), float(p[1]))


class _Polygon:
    def __init__(self, verts):
        self.verts = [(float(v[0]), float(v[1])) for v in verts]

    def contains(self, point):
        return _polygon_contains_strict(self.verts, point.p)

    @property
    def area(self):
        a = 0.0
        n = len(self.verts)
        for i in range(n):
            x0, y0 = self.verts[i]
            x1, y1 = self.verts[(i + 1) % n]
            a += x0 * y1 - x1 * y0
        return abs(a) / 2


class _Path:
    def __init__(self, verts):
        self.verts = [(float(v[0]), float(v[1])) for v in verts]

    def contains_point(self, p, radius=0.0):
        # radius<0 shrinks the path slightly in matplotlib; strict interior is
        # the behaviour the reference relies on (Environment.py:873).
        return _polygon_contains_strict(self.verts, p)


def _to_rgba(c, alpha=None):
    return (1.0, 0.5, 0.0, 1.0)


def install():
    """Insert the stub modules into sys.modules (idempotent)."""
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        mpl.__path__ = []
        plt = types.ModuleType("matplotlib.pyplot")
        coll = types.ModuleType("matplotlib.collections")
        colors = types.ModuleType("matplotlib.colors")
        path = types.ModuleType("matplotlib.path")
        cm = types.ModuleType("matplotlib.cm")
        coll.EllipseCollection = type("EllipseCollection", (), {})
        colors.to_rgba = _to_rgba
        path.Path = _Path
        mpl.pyplot, mpl.collections, mpl.colors, mpl.path, mpl.cm = plt, coll, colors, path, cm
        class _Colormaps(dict):                     # matplotlib.colormaps[name](x) -> RGBA (plot colours only)
            def __missing__(self, name):
                return lambda x: (0.0, 0.0, 0.0, 1.0)
        mpl.colormaps = _Colormaps()
        mpl.rcParams = {}
        for name, mod in [("matplotlib", mpl), ("matplotlib.pyplot", plt),
                          ("matplotlib.collections", coll), ("matplotlib.colors", colors),
                          ("matplotlib.path", path), ("matplotlib.cm", cm)]:
            sys.modules[name] = mod
    if "shapely" not in sys.modules:
        sh = types.ModuleType("shapely")
        sh.__path__ = []
        geom = types.ModuleType("shapely.geometry")
        sh.Polygon = geom.Polygon = _Polygon
        sh.Point = geom.Point = _Point
        sh.geometry = geom
        sys.modules["shapely"] = sh
        sys.modules["shapely.geometry"] = geom


def reference_root():
    """Where the unmodified reference lives: /root/reference (build container) or the copy staged by oracle/make_ref.py."""
    for root in (REFERENCE_ROOT, STAGED_ROOT):
        if os.path.isdir(os.path.join(root, "ratinabox")):
            return root
    return None


def import_reference():
    """Return the unmodified reference package (``ratinabox``), or None when neither /root/reference nor the staged copy
    (oracle/_ref, git-ignored, shipped by gpurun) is present."""
    root = reference_root()
    if root is None:
        return None
    install()
    if root not in sys.path:
        sys.path.insert(0, root)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return importlib.import_module("ratinabox")
