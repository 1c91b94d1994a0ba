"""CPU-only tests of the Python host layer: resolution, kernels, validation and error types
mirror the reference's tests (test_focal.py:178-197, test_utils.py, test_dataset_support.py)."""
import numpy as np
import pytest

import xrspatial_b200 as xb
from xrspatial_b200 import convolution, focal, utils, zonal
from xrspatial_b200.dataset_support import supports_dataset, supports_dataset_bands


def raster(data, **kw):
    r = xb.DataArray(np.asarray(data), dims=("y", "x"), **kw)
    return r


def test_resolution_from_attrs_and_coords():
    r = raster(np.zeros((4, 5)), attrs={"res": (0.5, 2.0)})
    assert utils.get_dataarray_resolution(r) == (0.5, 2.0)
    r = raster(np.zeros((4, 5)), attrs={"res": 3})
    assert utils.get_dataarray_resolution(r) == (3, 3)
    r = raster(np.zeros((4, 5)))
    r["y"] = np.linspace(30, 0, 4)     # descending y like create_test_raster (general_checks.py:30-52)
    r["x"] = np.linspace(0, 8, 5)
    assert utils.get_dataarray_resolution(r) == (2.0, 10.0)
    r.attrs["res"] = "bogus"           # falls back to the coordinates (utils.py:268-275)
    assert utils.get_dataarray_resolution(r) == (2.0, 10.0)


def test_calc_cellsize_units():
    r = raster(np.ones((100, 200)), attrs={"res": (0.5, 0.5)})
    assert convolution.calc_cellsize(r) == (0.5, 0.5)
    r = raster(np.ones((100, 200)), attrs={"unit": "km"})
    r["y"] = np.linspace(1, 100, 100)
    r["x"] = np.linspace(1, 200, 200)
    cx, cy = convolution.calc_cellsize(r)
    assert cx == 1000.0 and cy == 1000.0


def test_kernels(known):
    # test_focal.py:190-197
    np.testing.assert_array_equal(convolution.circle_kernel(1, 1, 1), known["focal.kernel_circle_1_1_1"])
    np.testing.assert_array_equal(convolution.annulus_kernel(2, 2, 2, 1), known["focal.kernel_annulus_2_2_2_1"])
    k = convolution.circle_kernel(1, 1, "3m")
    assert k.shape == (7, 7) and k[3].sum() == 7 and k[0].sum() == 1
    assert convolution.circle_kernel(10, 10, "0.03km").shape == (7, 7)
    with pytest.raises(ValueError):
        convolution.circle_kernel(1, 1, "3 parsecs")
    with pytest.raises(ValueError):
        convolution.circle_kernel(1, 1, -3)


def test_custom_kernel_validation():
    # test_focal.py:178-187
    with pytest.raises(ValueError):
        convolution.custom_kernel([[1, 0, 0], [0, 1, 0], [0, 0, 1]])
    with pytest.raises(ValueError):
        convolution.custom_kernel(np.ones((4, 6)))
    k = np.ones((3, 5))
    assert convolution.custom_kernel(k) is k


def test_error_types_before_any_device_work():
    r = raster(np.zeros((4, 4), np.float32), attrs={"res": (1, 1)})
    with pytest.raises(ValueError):
        xb.slope(r, method="spherical")                      # slope.py:334-337
    with pytest.raises(ValueError):
        xb.slope(r, method="geodesic")                       # no lat/lon coordinates (utils.py:680-684)
    g = raster(np.zeros((4, 4), np.float32))
    g["y"] = np.linspace(5000.0, 2000.0, 4)                  # projected metres, not degrees
    g["x"] = np.linspace(0.0, 3.0, 4)
    with pytest.raises(ValueError):
        xb.slope(g, method="geodesic")
    g["y"] = np.linspace(46.0, 45.9, 4)
    with pytest.raises(ValueError):
        xb.aspect(g, method="geodesic", z_unit="furlong")
    with pytest.raises(ValueError):
        xb.aspect(r, method="nope")
    with pytest.raises(RuntimeError):
        xb.hillshade(r, shadows=True)                        # hillshade.py:176-178
    with pytest.raises(TypeError):
        focal.apply(np.zeros((4, 4)), np.ones((3, 3)))       # focal.py:447
    with pytest.raises(ValueError):
        focal.apply(xb.DataArray(np.zeros((2, 3, 4))), np.ones((3, 3)))
    with pytest.raises(ValueError):
        focal.apply(r, np.ones((2, 2)))
    with pytest.raises(NotImplementedError):
        focal.apply(r, np.ones((3, 3)), func=lambda x: 0)    # only built-in reducers cross the C ABI
    with pytest.raises(ValueError):
        focal.focal_stats(r, np.ones((3, 3)), stats_funcs=["mean", "median"])   # validated before any launch
    with pytest.raises(TypeError):
        focal.focal_stats(np.zeros((4, 4)), np.ones((3, 3)))
    with pytest.raises(ValueError):
        focal.focal_stats(r, np.ones((3, 4)))
    with pytest.raises(ValueError):
        xb.savi(r, r, soil_factor=1.5)                       # multispectral.py:999-1000
    with pytest.raises(ValueError):
        xb.evi(r, r, r, gain=-1)
    with pytest.raises(ValueError):
        xb.evi(r, r, r, c1="6")
    with pytest.raises(ValueError):
        xb.ndvi(r, raster(np.zeros((4, 5), np.float32)))     # utils.py:155 shapes
    with pytest.raises(ValueError):
        xb.zonal_stats(r, r, stats_funcs=["median"])         # zonal.py:639-642
    with pytest.raises(ValueError):
        xb.zonal_stats(raster(np.zeros((4, 4), dtype=bool)), r)


def test_unsupported_array_type():
    class Odd(object):
        shape = (2, 2)
        dtype = np.dtype("f4")
    mapper = utils.ArrayTypeFunctionMapping(numpy_func=lambda *a: 1, cupy_func=lambda *a: 2)
    assert mapper(raster(np.zeros((2, 2))))() == 1
    holder = type("H", (), {"data": Odd()})()
    with pytest.raises(TypeError):
        mapper(holder)


def test_supports_dataset_decorators():
    # test_dataset_support.py: per-variable call, name injection, attrs kept, band kwargs
    calls = []

    @supports_dataset
    def f(agg, name="f"):
        calls.append(name)
        return xb.DataArray(agg.data + 1, dims=agg.dims, name=name)

    ds = xb.Dataset({"a": raster(np.zeros((2, 2))), "b": raster(np.ones((2, 2)))}, attrs={"k": 1})
    out = f(ds)
    assert isinstance(out, xb.Dataset) and list(out.data_vars) == ["a", "b"] and out.attrs == {"k": 1}
    assert calls == ["a", "b"] and out["b"].data[0, 0] == 2 and out["a"].name == "a"

    @supports_dataset_bands(nir="nir_agg", red="red_agg")
    def g(nir_agg, red_agg, name="g", extra=0):
        return (nir_agg.data - red_agg.data + extra).sum()

    assert g(ds, nir="b", red="a", extra=1) == 8
    with pytest.raises(TypeError):
        g(ds, nir="b")
    with pytest.raises(ValueError):
        g(ds, nir="b", red="zzz")


def test_zonal_finalize_matches_numpy():
    """finalize() turns (count, shifted sums, min, max) partials into the reference's columns."""
    rng = np.random.default_rng(3)
    vals = [rng.normal(1000, 5, 50), rng.normal(-3, 1, 7), np.array([]), np.array([42.0])]
    pivot = np.full(4, 900.0)
    part = dict(count=np.array([len(v) for v in vals], dtype=np.int64),
                s1=np.array([(v - 900.0).sum() for v in vals]),
                s2=np.array([((v - 900.0) ** 2).sum() for v in vals]),
                min=np.array([v.min() if len(v) else np.inf for v in vals]),
                max=np.array([v.max() if len(v) else -np.inf for v in vals]))
    cols = zonal.finalize(part, pivot, ["mean", "max", "min", "sum", "std", "var", "count"])
    for i, v in enumerate(vals):
        if len(v) == 0:
            assert all(np.isnan(cols[c][i]) for c in cols)
            continue
        np.testing.assert_allclose(cols["mean"][i], v.mean(), rtol=1e-13)
        np.testing.assert_allclose(cols["sum"][i], v.sum(), rtol=1e-13)
        np.testing.assert_allclose(cols["var"][i], v.var(), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(cols["std"][i], v.std(), rtol=1e-9, atol=1e-12)
        assert cols["count"][i] == len(v) and cols["min"][i] == v.min() and cols["max"][i] == v.max()


def test_split_rows():
    from xrspatial_b200.stripes import split_rows
    assert split_rows(10, 3) == [(0, 4), (4, 7), (7, 10)]
    assert split_rows(65536, 8)[7] == (57344, 65536)


def test_crosstab_pivot_matches_pair_loop():
    """The vectorised pivot of zonal.crosstab against the obvious loop (incl. a category subset,
    unselected zones and a zone listed twice)."""
    rng = np.random.default_rng(3)
    pz = rng.integers(0, 40, 3000).astype(np.int64)
    pv = rng.integers(0, 12, 3000).astype(np.float64)
    pc = rng.integers(1, 1 << 20, 3000).astype(np.int64)
    for sel, cats in ((np.arange(40), list(range(12))), (np.array([7, 3, 3, 39, 12]), [2.0, 5.0, 11.0]),
                      (np.array([1.5, 2.0]), [0.0]), (np.array([], dtype=np.int64), [1.0])):
        total, counts = zonal._pivot_pairs(sel, cats, pz, pv, pc)
        zpos = {float(z): i for i, z in enumerate(sel)}
        t2 = np.zeros(len(sel), np.float32)
        c2 = np.zeros((len(cats), len(sel)), np.int64)
        bounds = np.asarray(cats, dtype=np.float64)
        for z, v, c in zip(pz.tolist(), pv.tolist(), pc.tolist()):
            i = zpos.get(float(z))
            if i is None:
                continue
            t2[i] += c
            j = int(np.searchsorted(bounds, v, side="left"))
            if j < len(cats):
                c2[j][i] += c
        np.testing.assert_array_equal(total, t2)
        np.testing.assert_array_equal(counts, c2)


def test_public_signatures_equal_the_reference(refsig):
    """Parameter names, order and defaults of every public function on the path: the reference's, read with
    `inspect` from the unmodified reference by oracle/make_golden.py (tests/golden/reference_signatures.json),
    and this package's.  The only allowed difference: a trailing `comm=None` (row-stripe group) on the zonal
    functions."""
    import importlib
    import inspect
    assert sum(len(v) for v in refsig.values()) == 30

    def params(f):
        return [(k, v.default) for k, v in inspect.signature(inspect.unwrap(f)).parameters.items()]

    for mod, funcs in refsig.items():
        mine_mod = importlib.import_module('xrspatial_b200.' + mod)
        for n, rp in funcs.items():
            mp = params(getattr(mine_mod, n))
            if mod == 'zonal':
                assert mp[-1] == ('comm', None), n
                mp = mp[:-1]
            assert [r['name'] for r in rp] == [k for k, _ in mp], (mod, n)
            for r, (k, b) in zip(rp, mp):
                if set(r) == {'name'}:                      # no default
                    assert b is inspect.Parameter.empty, (mod, n, k)
                elif 'callable' in r:
                    assert callable(b) or r['callable'] == getattr(b, '__name__', b), (mod, n, k)
                elif callable(b):
                    assert r.get('repr') == repr(b.__name__), (mod, n, k)
                elif r.get('nan'):
                    assert b != b, (mod, n, k)
                else:
                    assert r['repr'] == repr(b), (mod, n, k, r['repr'], b)


# ----------------------------------------------------------------- the xarray facade (_xr.py)
class _StrictFakeXarray(object):
    """A stand-in for the real xarray module that is as strict as xarray where the ADVICE findings bite:
    DataArray refuses anything np.asarray cannot take (a CUDA tensor), Dataset.data_vars is read-only."""

    class DataArray(object):
        def __init__(self, data=None, coords=None, dims=None, name=None, attrs=None):
            if type(data).__module__.split(".")[0] == "torch":
                raise TypeError("can't convert cuda:0 device type tensor to numpy")
            self.data = np.asarray(data)
            self.dims = tuple(dims) if dims is not None else tuple("dim_%d" % i for i in range(self.data.ndim))
            self.coords = dict(coords or {})
            self.name, self.attrs = name, dict(attrs or {})
            self.shape, self.ndim, self.dtype = self.data.shape, self.data.ndim, self.data.dtype

    class Dataset(object):
        def __init__(self, data_vars=None, coords=None, attrs=None):
            self._v = dict(data_vars or {})
            self.attrs = dict(attrs or {})

        @property
        def data_vars(self):
            import types
            return types.MappingProxyType(self._v)

        def __setitem__(self, k, v):
            self._v[k] = v

        def __getitem__(self, k):
            return self._v[k]

    @staticmethod
    def concat(objs, dim):
        return ("concat", len(objs))


def test_xarray_facade_picks_the_container_by_payload(monkeypatch):
    """With xarray importable: numpy payloads become real xarray objects, device payloads stay in the
    stand-in (xarray cannot hold a torch tensor), isinstance() accepts both families."""
    import importlib
    import sys
    import types
    fake = types.ModuleType("xarray")
    fake.DataArray, fake.Dataset, fake.concat = _StrictFakeXarray.DataArray, _StrictFakeXarray.Dataset, _StrictFakeXarray.concat
    monkeypatch.setitem(sys.modules, "xarray", fake)
    spec = importlib.util.spec_from_file_location("_xr_under_test", xb._xr.__file__)
    xr_mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(xr_mod)
    assert xr_mod.HAVE_XARRAY
    a = xr_mod.DataArray(np.zeros((2, 3)), dims=("y", "x"), attrs={"res": (1, 1)}, name="n")
    assert isinstance(a, fake.DataArray) and isinstance(a, xr_mod.DataArray) and a.attrs == {"res": (1, 1)}

    class FakeTensor(object):      # looks like a torch tensor to the facade (module name + data_ptr)
        shape, dtype = (2, 3), "float32"

        def data_ptr(self):
            return 0
    FakeTensor.__module__ = "torch"
    t = xr_mod.DataArray(FakeTensor(), dims=("y", "x"))
    assert isinstance(t, xr_mod.ShimDataArray) and isinstance(t, xr_mod.DataArray)
    assert not isinstance(np.zeros(3), xr_mod.DataArray)
    ds = xr_mod.Dataset({"a": a})
    assert isinstance(ds, fake.Dataset) and isinstance(ds, xr_mod.Dataset)
    ds["b"] = a
    with pytest.raises(TypeError):
        ds.data_vars["c"] = a
    dsd = xr_mod.Dataset({"t": t})
    assert isinstance(dsd, xr_mod.ShimDataset)
    dsd["u"] = t
    assert list(dsd.data_vars) == ["t", "u"]
    with pytest.raises(TypeError):
        dsd.data_vars["v"] = t
    assert xr_mod.concat([a, a], None) == ("concat", 2)


def test_shim_is_as_strict_as_xarray_where_it_matters():
    from xrspatial_b200._xr import ShimDataArray, ShimDataset
    a = ShimDataArray(np.zeros((4, 5)), dims=("y", "x"))
    np.testing.assert_array_equal(a["y"].data, np.arange(4))       # default integer index
    np.testing.assert_array_equal(a["x"].data, np.arange(5))
    with pytest.raises(KeyError):
        a["nope"]
    with pytest.raises(ValueError):
        ShimDataArray(np.zeros((4, 5)), dims=("y", "x"), coords={"y": np.arange(3)})
    with pytest.raises(ValueError):
        ShimDataArray(np.zeros((4, 5)), dims=("y",))
    ds = ShimDataset({"a": a})
    with pytest.raises(TypeError):
        ds.data_vars["b"] = a
    with pytest.raises(ValueError):
        ds["b"] = ShimDataArray(np.zeros((3, 5)), dims=("y", "x"))
    ds["b"] = a
    assert list(ds) == ["a", "b"]
    # resolution of a bare DataArray: unit cells (utils.py:233-277 through the default index)
    from xrspatial_b200.utils import get_dataarray_resolution
    assert get_dataarray_resolution(a) == (1.0, 1.0)


def test_zonal_stats_argument_checks_without_a_gpu():
    from xrspatial_b200 import zonal
    z = xb.DataArray(np.zeros((2, 2), np.int32), dims=("y", "x"))
    v = xb.DataArray(np.zeros((2, 2), np.float32), dims=("y", "x"))
    with pytest.raises(ValueError, match="Invalid stat name"):
        zonal.stats(z, v, stats_funcs=["mean", "median"])
    with pytest.raises(TypeError):
        zonal.stats(z, v, stats_funcs="mean")
    with pytest.raises(ValueError, match="equal shapes"):
        zonal.stats(xb.DataArray(np.zeros((2, 3), np.int32), dims=("y", "x")), v)


def test_row_segments_are_wave_balanced():
    """pick_seg_rows (stencil3.cuh, through the host-only hook xrs_debug_pick_seg_rows): tasks = tiles x segments
    are dealt round-robin to the resident CTAs, so a kernel lasts ceil(tasks / resident) task-times.  The chosen
    segment height must (a) respect the minimum height and the chunk quantum, (b) never be worse than the
    round-1 rule (round the segment count UP to ~8 tasks per CTA), and (c) stay within 4 % of the ideal
    H * tiles / resident rows per CTA on the benchmark shapes -- the round-1 rule ran the fused suite in 9
    waves instead of 8.03 (1188 tasks on 1184 slots)."""
    import xrspatial_b200
    lib = xrspatial_b200._lib.lib()

    def cost(H, n_tiles, resident, rows, lead):
        segs = -(-H // rows)
        return -(-(segs * n_tiles) // resident) * (rows + lead)

    def round1_rows(H, n_tiles, resident, quantum):
        want = -(-(resident * 8) // n_tiles)
        rows = max(32, -(-H // want))
        rows = min(rows, H)
        return max(1, -(-(rows + 2) // quantum) * quantum - 2)

    cases = [(32768, 32, 296, 4), (32768, 16, 148, 2), (32768, 22, 148, 8), (65536, 64, 296, 4), (8192, 64, 296, 4),
             (10000, 15, 148, 2), (30000, 30, 296, 4), (2048, 2, 296, 4), (100, 1, 296, 4), (3, 1, 296, 4),
             (4321, 7, 148, 8), (16384, 40, 296, 4)]
    for H, n_tiles, resident, quantum in cases:
        rows = lib.xrs_debug_pick_seg_rows(H, n_tiles, resident, 32, 2, quantum, 8)
        assert rows >= 1 and (rows + 2) % quantum == 0, (H, n_tiles, rows)
        assert rows >= min(32, H) - quantum, (H, n_tiles, rows)
        new, old = cost(H, n_tiles, resident, rows, 2), cost(H, n_tiles, resident, round1_rows(H, n_tiles, resident, quantum), 2)
        assert new <= old, (H, n_tiles, resident, rows, new, old)
        ideal = H * n_tiles / resident
        if H * n_tiles >= 64 * resident * 32:          # enough rows for every CTA to get several tasks
            assert new <= 1.04 * ideal + 40, (H, n_tiles, resident, rows, new, ideal)
    # the running box: lead-in rows kh - 1, batches of 4, tall segments
    for kh, n_tiles in ((9, 40), (25, 46), (5, 40)):
        rows = lib.xrs_debug_pick_seg_rows(32768, n_tiles, 296, 12 * kh, kh - 1, 4, 4)
        assert (rows + kh - 1) % 4 == 0 and rows >= 12 * kh
        assert cost(32768, n_tiles, 296, rows, kh - 1) <= 1.06 * 32768 * n_tiles / 296
