"""Load the UNMODIFIED reference kernels from /root/reference (this container only).

TEST INFRASTRUCTURE -- never imported by the product path, by bench.py's GPU arm
or by anything that runs on the GPU box (where /root/reference does not exist).
It is used only by oracle/make_golden.py to generate the fixtures under tests/golden/;
the tests read those fixtures and never the reference itself.

`import xrspatial` fails here because xarray / datashader are not installed
(xrspatial/utils.py:6-9), so we register stub modules for those two packages and a
bare ``xrspatial`` package object whose __path__ points at the read-only tree
(skipping xrspatial/__init__.py, which imports every module).  The hot-path
kernels themselves (Numba @ngjit loops / NumPy) then import and run unmodified.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("XRS_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "xrspatial"))


class _StubDataArray:
    """Just enough of xr.DataArray for ArrayTypeFunctionMapping / convolve_2d."""

    def __init__(self, data=None, name=None, coords=None, dims=None, attrs=None):
        self.data = data
        self.name = name
        self.coords = coords if coords is not None else {}
        self.dims = dims if dims is not None else ()
        self.attrs = attrs if attrs is not None else {}

    @property
    def shape(self):
        return self.data.shape

    @property
    def ndim(self):
        return self.data.ndim

    @property
    def values(self):
        return self.data


class _StubDataset(dict):
    pass


_loaded = {}


def load(modname):
    """Return reference module xrspatial.<modname> (e.g. 'slope')."""
    if modname in _loaded:
        return _loaded[modname]
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    if "xarray" not in sys.modules:
        xr = types.ModuleType("xarray")
        xr.DataArray = _StubDataArray
        xr.Dataset = _StubDataset
        xr.concat = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError())
        sys.modules["xarray"] = xr
    if "datashader" not in sys.modules:
        ds = types.ModuleType("datashader")
        ds.Canvas = object
        tf = types.ModuleType("datashader.transfer_functions")
        colors = types.ModuleType("datashader.colors")
        colors.rgb = lambda *a, **k: (0, 0, 0)
        ds.transfer_functions = tf
        ds.colors = colors
        sys.modules["datashader"] = ds
        sys.modules["datashader.transfer_functions"] = tf
        sys.modules["datashader.colors"] = colors
    if "xrspatial" not in sys.modules:
        pkg = types.ModuleType("xrspatial")
        pkg.__path__ = [os.path.join(REF_ROOT, "xrspatial")]
        sys.modules["xrspatial"] = pkg
    mod = importlib.import_module("xrspatial." + modname)
    _loaded[modname] = mod
    return mod
