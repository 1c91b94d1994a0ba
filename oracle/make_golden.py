"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build container only).

TEST INFRASTRUCTURE.  Three fixture files are produced:

* tests/golden/known_answers.npz -- the literal known-answer arrays that the reference's
  own test-suite holds for the hot path (QGIS / hand-derived tables; SURVEY.md 8c).  They are
  extracted by parsing /root/reference/xrspatial/tests/*.py with `ast` and evaluating the
  fixture functions (no reference source is copied into this repository, only the data).
* tests/golden/reference_outputs.npz -- seeded inputs and the outputs of the reference's
  Numba-CPU / NumPy kernels (loaded through oracle/ref_loader.py) on those inputs, for every
  op on the hot path, including NaN-laden, flat ("water"), integer-valued and odd-shaped cases.
* tests/golden/reference_signatures.json -- parameter names, order and defaults of every public
  function on the path, read with `inspect` from the reference modules.

Usage:  python oracle/make_golden.py         (needs /root/reference)
"""
import ast
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_loader  # noqa: E402

OUT_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")
TESTS = os.path.join(ref_loader.REF_ROOT, "xrspatial", "tests")


# ------------------------------------------------------------------ known answers
def _fixture_funcs(path):
    src = open(path).read()
    tree = ast.parse(src)
    funcs = {}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef):
            node.decorator_list = []
            mod = ast.Module(body=[node], type_ignores=[])
            funcs[node.name] = compile(ast.fix_missing_locations(mod), path, "exec")
    return funcs


def _call(funcs, name, *args, **kw):
    xr = types.SimpleNamespace(DataArray=lambda a, **k: a)
    ns = dict(np=np, xr=xr,
              create_test_raster=lambda data, backend="numpy", **k: np.asarray(data),
              custom_kernel=lambda k: k,
              has_dask_array=lambda: False)
    exec(funcs[name], ns)
    return ns[name](*args, **kw)


def known_answers():
    g = {}
    f = _fixture_funcs(os.path.join(TESTS, "conftest.py"))
    for n in ("elevation_raster", "elevation_raster_no_nans", "raster"):
        g["conftest." + n] = _call(f, n)

    f = _fixture_funcs(os.path.join(TESTS, "test_slope.py"))
    g["slope.qgis_slope"] = _call(f, "qgis_slope")
    f = _fixture_funcs(os.path.join(TESTS, "test_aspect.py"))
    g["aspect.qgis_aspect"] = _call(f, "qgis_aspect")

    f = _fixture_funcs(os.path.join(TESTS, "test_curvature.py"))
    for n in ("convex_surface", "concave_surface"):
        d, e = _call(f, n)
        g["curvature.%s.data" % n] = np.asarray(d)
        g["curvature.%s.expected" % n] = np.asarray(e)

    f = _fixture_funcs(os.path.join(TESTS, "test_focal.py"))
    g["focal.convolve_2d_data"] = _call(f, "convolve_2d_data")
    g["focal.kernel_circle_1_1_1"] = _call(f, "kernel_circle_1_1_1")
    g["focal.kernel_annulus_2_2_2_1"] = _call(f, "kernel_annulus_2_2_2_1")
    g["focal.convolution_kernel_circle_1_1_1"] = _call(f, "convolution_kernel_circle_1_1_1")
    g["focal.convolution_kernel_annulus_2_2_1"] = _call(f, "convolution_kernel_annulus_2_2_1")
    k, e = _call(f, "convolution_custom_kernel")
    g["focal.convolution_custom_kernel.kernel"] = k
    g["focal.convolution_custom_kernel.expected"] = e
    d, k, e = _call(f, "data_apply")
    g["focal.data_apply.data"], g["focal.data_apply.kernel"] = d, k
    d, k, e = _call(f, "data_focal_stats")
    g["focal.data_focal_stats.data"] = d
    g["focal.data_focal_stats.kernel"] = k
    g["focal.data_focal_stats.expected"] = e  # order: mean max min range std var sum

    f = _fixture_funcs(os.path.join(TESTS, "test_multispectral.py"))
    for n in ("blue", "green", "red", "nir", "tir", "swir1", "swir2"):
        g["multispectral.%s_data" % n] = np.asarray(_call(f, n + "_data", "numpy"), dtype=np.float64)
    for n in ("arvi", "evi", "nbr", "nbr2", "ndvi", "ndmi", "savi", "gci", "sipi", "ebbi"):
        g["multispectral.qgis_" + n] = _call(f, "qgis_" + n)
    for n in ("normalized_ratio", "arvi", "evi", "savi", "sipi", "ebbi"):
        vals = _call(f, "data_uint_dtype_" + n, np.uint16)
        for i, v in enumerate(vals):
            g["multispectral.uint_%s.%d" % (n, i)] = np.asarray(v)

    f = _fixture_funcs(os.path.join(TESTS, "test_zonal.py"))
    g["zonal.data_zones"] = _call(f, "data_zones", "numpy")
    g["zonal.data_values_2d"] = _call(f, "data_values_2d", "numpy")
    for n in ("result_default_stats", "qgis_zonal_stats"):
        d = _call(f, n)
        for k2, v in d.items():
            g["zonal.%s.%s" % (n, k2)] = np.asarray(v, dtype=np.float64)
    zid, d = _call(f, "result_zone_ids_stats")
    g["zonal.result_zone_ids_stats.zone_ids"] = np.asarray(zid)
    for k2, v in d.items():
        g["zonal.result_zone_ids_stats.%s" % k2] = np.asarray(v, dtype=np.float64)
    g["zonal.result_default_stats_dataarray"] = _call(f, "result_default_stats_dataarray")
    # custom statistics (test_zonal.py:204-246: double_sum = 2*sum, range = max - min; nodata 0, zones 1, 2)
    nod, zid, d = _call(f, "result_custom_stats")
    g["zonal.result_custom_stats.nodata_values"] = np.asarray(nod)
    g["zonal.result_custom_stats.zone_ids"] = np.asarray(zid)
    for k2, v in d.items():
        g["zonal.result_custom_stats.%s" % k2] = np.asarray(v, dtype=np.float64)
    _, _, arr = _call(f, "result_custom_stats_dataarray")
    g["zonal.result_custom_stats_dataarray"] = np.asarray(arr)
    # 3-D crosstab (test_zonal.py:48-58 data, :266-336 expected): values of ones, categories cat1..cat4
    layer, zid, d = _call(f, "result_crosstab_3d")
    g["zonal.result_crosstab_3d.layer"] = np.asarray(layer)
    for agg, tab in d.items():
        g["zonal.result_crosstab_3d.%s" % agg] = np.asarray([tab[k2] for k2 in ("zone", "cat1", "cat2", "cat3", "cat4")],
                                                            dtype=np.float64)
    nod, layer, zid, tab = _call(f, "result_nodata_values_crosstab_3d")
    g["zonal.result_nodata_values_crosstab_3d"] = np.asarray([tab[k2] for k2 in ("zone", "cat1", "cat2", "cat3", "cat4")],
                                                             dtype=np.float64)
    return g


# ------------------------------------------------------------------ reference outputs
def terrain(rng, h, w, water=False, nans=0.0, integer=False):
    """Small smooth-ish synthetic DEM (double cumulative sum of noise + a ramp)."""
    z = rng.standard_normal((h, w)).cumsum(0).cumsum(1)
    z += np.linspace(0, 30, w)[None, :] + np.linspace(0, 10, h)[:, None]
    z = (z - z.min()) / (z.max() - z.min() + 1e-9) * 4000.0
    if water:
        z[z < 0.3 * z.max()] = 0.0
    if integer:
        z = np.round(z)
    z = z.astype(np.float32)
    if nans:
        m = rng.random((h, w)) < nans
        z[m] = np.nan
    return z


def reference_outputs():
    slope = ref_loader.load("slope")
    aspect = ref_loader.load("aspect")
    curv = ref_loader.load("curvature")
    hill = ref_loader.load("hillshade")
    conv = ref_loader.load("convolution")
    focal = ref_loader.load("focal")
    ms = ref_loader.load("multispectral")
    zonal = ref_loader.load("zonal")

    g = {}
    rng = np.random.default_rng(20260922)
    cases = {
        "smooth": terrain(rng, 37, 53),
        "water": terrain(rng, 41, 36, water=True),
        "nans": terrain(rng, 33, 47, nans=0.03),
        "integer": terrain(rng, 20, 64, integer=True),
        "rough": (rng.random((29, 31)) * 1000).astype(np.float32),
        "tiny": (rng.integers(-100, 100, size=(3, 4))).astype(np.float32),
        "rand_2x4": np.random.default_rng(2841).integers(-100, 100, size=(2, 4)).astype(np.float32),
        "rand_10x15": np.random.default_rng(2841).integers(-100, 100, size=(10, 15)).astype(np.float32),
    }
    for name, z in cases.items():
        g["dem.%s" % name] = z
        g["slope.%s" % name] = slope._cpu(z, 30.0, 30.0)
        g["slope_aniso.%s" % name] = slope._cpu(z, 10.0, 25.5)
        g["aspect.%s" % name] = aspect._run_numpy(z)
        g["curvature.%s" % name] = curv._run_numpy(z, 30.0)
        g["hillshade.%s" % name] = hill._run_numpy(z, 225, 25)
        g["hillshade_az315_alt45.%s" % name] = hill._run_numpy(z, 315, 45)
        g["focal_mean.%s" % name] = focal._mean_numpy(z.astype(float), (np.nan,))
        out = z.astype(float)
        for _ in range(3):
            out = focal._mean_numpy(out, (np.nan,))
        g["focal_mean_p3.%s" % name] = out
        g["focal_mean_ex.%s" % name] = focal._mean_numpy(z.astype(float), (np.nan, 0.0))

    # convolution kernels
    kernels = {
        "box3": np.ones((3, 3)) / 9.0,
        "box9": np.ones((9, 9)) / 81.0,
        "mixed5": rng.standard_normal((5, 5)),
        "mixed3x7": rng.standard_normal((3, 7)),
        "mixed25": rng.standard_normal((25, 25)),
        "int3": np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]]),
    }
    zc = terrain(rng, 61, 75)
    zcn = zc.copy()
    zcn[10, 12] = np.nan
    zcn[40, 70] = np.inf
    g["conv.dem"] = zc
    g["conv.dem_nan"] = zcn
    for kn, k in kernels.items():
        g["conv.kernel.%s" % kn] = np.asarray(k, dtype=np.float64)
        g["conv.out.%s" % kn] = conv._convolve_2d_numpy(zc, k)
        g["conv.out_nan.%s" % kn] = conv._convolve_2d_numpy(zcn, k)

    # focal apply / focal_stats
    masks = {
        "circle3": np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], dtype=float),
        "full3": np.ones((3, 3)),
        "annulus5": np.array([[0, 1, 1, 1, 0], [1, 1, 0, 1, 1], [1, 0, 0, 0, 1],
                              [1, 1, 0, 1, 1], [0, 1, 1, 1, 0]], dtype=float),
        "rect3x5": np.ones((3, 5)),
        "weights3": np.array([[1, 2, 0], [0.5, 1, 0], [0, 0, 1]], dtype=float),
    }
    fn = dict(mean=focal._calc_mean, sum=focal._calc_sum, min=focal._calc_min,
              max=focal._calc_max, std=focal._calc_std, range=focal._calc_range,
              var=focal._calc_var)
    za = terrain(rng, 23, 27, nans=0.05)
    g["apply.dem"] = za
    for mn, m in masks.items():
        g["apply.mask.%s" % mn] = m
        for sn, f in fn.items():
            g["apply.out.%s.%s" % (mn, sn)] = focal._apply_numpy(za, m, f)

    # multispectral
    def band(lo=0.02, hi=0.6):
        b = terrain(rng, 31, 45)
        b = lo + (hi - lo) * b / 4000.0
        return b.astype(np.float32)

    nir, red, blue, green, swir, tir = [band() for _ in range(6)]
    for b in (nir, red, blue, green, swir, tir):
        b[rng.random(b.shape) < 0.02] = 0.0
        b[rng.random(b.shape) < 0.01] = np.nan
    red[5, 5], nir[5, 5] = 0.25, -0.25      # denominator exactly 0
    g.update({"ms.nir": nir, "ms.red": red, "ms.blue": blue, "ms.green": green,
              "ms.swir": swir, "ms.tir": tir})
    g["ms.ndvi"] = ms._normalized_ratio_cpu(nir, red)
    g["ms.savi"] = ms._savi_cpu(nir, red, 1.0)
    g["ms.savi_L05"] = ms._savi_cpu(nir, red, 0.5)
    g["ms.evi"] = ms._evi_cpu(nir, red, blue, 6.0, 7.5, 1.0, 2.5)
    g["ms.arvi"] = ms._arvi_cpu(nir, red, blue)
    g["ms.gci"] = ms._gci_cpu(nir, green)
    g["ms.sipi"] = ms._sipi_cpu(nir, red, blue)
    g["ms.ebbi"] = ms._ebbi_cpu(red, swir, tir)

    # zonal.stats: float32 values / int32 zones, float64 values / float zones with NaN
    stats7 = ["mean", "max", "min", "sum", "std", "var", "count"]
    zv = terrain(rng, 48, 64, nans=0.02)
    zz = ((np.arange(48)[:, None] // 12) * 4 + (np.arange(64)[None, :] // 16)).astype(np.int32)
    zz[rng.random(zz.shape) < 0.1] = 100 + rng.integers(0, 5)
    g["zonal.values_f32"], g["zonal.zones_i32"] = zv, zz
    df = zonal._stats_numpy(zz, zv, None, {s: zonal._DEFAULT_STATS[s] for s in stats7 + ["majority"]},
                            None, return_type="pandas.DataFrame")
    for c in df.columns:
        g["zonal.f32_i32.%s" % c] = np.asarray(df[c])
    df = zonal._stats_numpy(zz, zv, [3, 7, 100, 999], {s: zonal._DEFAULT_STATS[s] for s in stats7},
                            0.0, return_type="pandas.DataFrame")
    for c in df.columns:
        g["zonal.f32_i32_ids_nodata.%s" % c] = np.asarray(df[c])
    zv64 = (zv.astype(np.float64) + 1e6) * 1.000001
    zzf = zz.astype(np.float64)
    zzf[0, :7] = np.nan
    zzf[1, 3] = -2.5
    g["zonal.values_f64"], g["zonal.zones_f64"] = zv64, zzf
    df = zonal._stats_numpy(zzf, zv64, None, {s: zonal._DEFAULT_STATS[s] for s in stats7},
                            None, return_type="pandas.DataFrame")
    for c in df.columns:
        g["zonal.f64_f64.%s" % c] = np.asarray(df[c])
    arr = zonal._stats_numpy(zz, zv, [3, 7], {s: zonal._DEFAULT_STATS[s] for s in ("mean", "count")},
                             None, return_type="xarray.DataArray")
    g["zonal.f32_i32.broadcast_mean_count_3_7"] = arr
    # custom callables through the reference's own per-zone loop (zonal.py:144-163)
    custom = {"double_sum": lambda v: v.sum() * 2, "range": lambda v: v.max() - v.min(),
              "l2norm": lambda v: np.sqrt(np.sum(v.astype(np.float64) * v))}
    df = zonal._stats_numpy(zz, zv, [3, 7, 100, 999], custom, 0.0, return_type="pandas.DataFrame")
    for c in df.columns:
        g["zonal.f32_i32_custom.%s" % c] = np.asarray(df[c])

    # focal.hotspots (focal.py:918-937) on a raster with two bumps, and zonal.crosstab (2-D)
    import types
    hz = terrain(rng, 64, 80)
    hz[20:26, 30:36] += 3000.0
    hz[45:50, 10:16] -= 2500.0
    hk = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], dtype=float)
    g["hotspots.dem"] = hz
    g["hotspots.kernel"] = hk
    g["hotspots.out"] = focal._hotspots_numpy(types.SimpleNamespace(data=hz), hk)
    hk5 = np.ones((5, 5))
    g["hotspots.out_5x5"] = focal._hotspots_numpy(types.SimpleNamespace(data=hz), hk5)
    cz = rng.integers(0, 6, size=(40, 52)).astype(np.int32)
    cv = rng.integers(10, 15, size=(40, 52)).astype(np.float32)
    cv[rng.random(cv.shape) < 0.05] = np.nan
    cv[cz == 4] = np.nan                      # a zone without any valid value
    g["crosstab.zones"], g["crosstab.values"] = cz, cv
    ucats = np.unique(cv[np.isfinite(cv)])
    for agg in ("count", "percentage"):
        df = zonal._crosstab_numpy(cz, cv, None, ucats, ucats, None, agg)
        g["crosstab.%s.columns" % agg] = np.asarray([float(c) for c in df.columns[1:]])
        g["crosstab.%s.table" % agg] = np.asarray(df.values, dtype=np.float64)
    df = zonal._crosstab_numpy(cz, cv, [1, 3, 9], ucats, [11.0, 13.0], 12.0, "count")
    g["crosstab.sub.table"] = np.asarray(df.values, dtype=np.float64)
    # 3-D values (zonal.py:734-745): categories = layers, cell = statistic of the layer over the zone.
    # A separate generator so that the arrays above keep their seeded values.
    rng3 = np.random.default_rng(777)
    c3 = rng3.standard_normal((4, 40, 52)).astype(np.float32) * 30 + 100
    c3[rng3.random(c3.shape) < 0.03] = np.nan
    c3[2, (cz == 1) & (rng3.random(cz.shape) < 0.5)] = 7.0      # nodata cells (a fully-nodata zone makes np.max raise)
    g["crosstab3d.values"] = c3
    cats3 = np.array([2001.0, 2002.0, 2003.0, 2004.0])
    for agg in ("mean", "max", "min", "sum", "std", "var", "count"):
        df = zonal._crosstab_numpy(cz, c3, [0, 1, 2, 3, 5], cats3, [2001.0, 2003.0, 2004.0], 7.0, agg)
        g["crosstab3d.%s" % agg] = np.asarray(df.values, dtype=np.float64)

    # geodesic slope / aspect (geodesic.py) on a lat/lon grid near 46N, with NaNs and a flat patch
    geod = ref_loader.load("geodesic")
    gz = terrain(rng, 40, 52, nans=0.01).astype(np.float64)
    gz[5:12, 5:12] = 1500.0
    glat = np.linspace(46.5, 46.0, 40)
    glon = np.linspace(7.0, 7.8, 52)
    lat2 = np.broadcast_to(glat[:, None], gz.shape).copy()
    lon2 = np.broadcast_to(glon[None, :], gz.shape).copy()
    a2, b2 = geod.WGS84_A2, geod.WGS84_B2
    g["geodesic.dem"], g["geodesic.lat"], g["geodesic.lon"] = gz, glat, glon
    g["geodesic.slope"] = geod._cpu_geodesic_slope(np.stack([gz, lat2, lon2]), a2, b2, 1.0)
    g["geodesic.aspect"] = geod._cpu_geodesic_aspect(np.stack([gz, lat2, lon2]), a2, b2, 1.0)
    g["geodesic.slope_ft"] = geod._cpu_geodesic_slope(np.stack([gz, lat2, lon2]), a2, b2, 0.3048)
    # curvilinear (2-D) coordinates
    lat2c = lat2 + 0.0005 * np.sin(np.arange(52))[None, :]
    lon2c = lon2 + 0.0007 * np.cos(np.arange(40))[:, None]
    g["geodesic.lat2d"], g["geodesic.lon2d"] = lat2c, lon2c
    g["geodesic.slope_2d"] = geod._cpu_geodesic_slope(np.stack([gz, lat2c, lon2c]), a2, b2, 1.0)
    g["geodesic.aspect_2d"] = geod._cpu_geodesic_aspect(np.stack([gz, lat2c, lon2c]), a2, b2, 1.0)

    # focal.apply over all-ones windows: the shapes of the reference's own focal benchmark
    # (benchmarks/benchmarks/focal.py FocalApply: custom_kernel(np.ones((5, 5))) / ((25, 25))) plus a
    # rectangular one, on a raster with NaNs, an all-NaN patch, +-inf and a FLT_MAX-style sentinel.
    # A separate generator so that the arrays above keep their seeded values.
    rng4 = np.random.default_rng(4040)
    zo = terrain(rng4, 70, 96, nans=0.02)
    zo[20:30, 40:52] = np.nan
    zo[5, 3] = np.inf
    zo[60, 90] = -np.inf
    zo[44, 10] = np.float32(3.4028235e38)
    g["apply_ones.dem"] = zo
    for kh, kw in ((5, 5), (25, 25), (3, 7), (9, 3)):
        g["apply_ones.mean.%dx%d" % (kh, kw)] = focal._apply_numpy(zo, np.ones((kh, kw)), focal._calc_mean)
    return g


# ------------------------------------------------------------------ public signatures
SIGNATURES = {'slope': ['slope'], 'aspect': ['aspect'], 'curvature': ['curvature'], 'hillshade': ['hillshade'],
              'focal': ['mean', 'apply', 'focal_stats', 'hotspots'],
              'convolution': ['convolve_2d', 'convolution_2d', 'custom_kernel', 'circle_kernel', 'annulus_kernel',
                              'calc_cellsize'],
              'zonal': ['stats', 'crosstab'], 'analytics': ['summarize_terrain'],
              'multispectral': ['ndvi', 'savi', 'evi', 'arvi', 'gci', 'sipi', 'ebbi', 'nbr', 'nbr2', 'ndmi'],
              'utils': ['get_dataarray_resolution', 'calc_res', 'validate_arrays']}


def _param(name, default):
    """One parameter as JSON: no "default" key when it has none; a callable default by its
    __name__, a NaN default as a flag, any other default by its repr."""
    import inspect
    if default is inspect.Parameter.empty:
        return {"name": name}
    if callable(default):
        return {"name": name, "callable": getattr(default, "__name__", None)}
    if isinstance(default, float) and default != default:
        return {"name": name, "nan": True}
    return {"name": name, "repr": repr(default)}


def reference_signatures():
    import inspect
    sigs = {}
    for mod, names in SIGNATURES.items():
        m = ref_loader.load(mod)
        sigs[mod] = {n: [_param(k, v.default) for k, v in inspect.signature(inspect.unwrap(getattr(m, n))).parameters.items()]
                     for n in names}
    return sigs


def main():
    import json
    os.makedirs(OUT_DIR, exist_ok=True)
    ka = known_answers()
    np.savez_compressed(os.path.join(OUT_DIR, "known_answers.npz"), **ka)
    ro = reference_outputs()
    np.savez_compressed(os.path.join(OUT_DIR, "reference_outputs.npz"), **ro)
    with open(os.path.join(OUT_DIR, "reference_signatures.json"), "w") as f:
        json.dump(reference_signatures(), f, indent=1)
        f.write("\n")
    for n in ("known_answers.npz", "reference_outputs.npz", "reference_signatures.json"):
        print(n, os.path.getsize(os.path.join(OUT_DIR, n)), "bytes")
    print(len(ka), "known-answer arrays;", len(ro), "reference input/output arrays")


if __name__ == "__main__":
    main()
