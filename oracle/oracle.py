"""ctypes front-end of the CPU oracle (oracle/xrs_oracle.c) + the NumPy zonal oracle.

TEST INFRASTRUCTURE ONLY: may be imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs -- never by xarray-spatial_b200/.

Function names mirror the reference's L1/L0 seam (SURVEY.md section 8c):
slope._cpu, aspect._run_numpy, curvature._cpu, hillshade._run_numpy,
convolution._convolve_2d_numpy, focal._mean_numpy / _apply_numpy,
multispectral._*_cpu, zonal._stats_numpy.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libxrs_oracle.so")
_lib = None
_tmp_so = None      # build()'s product when the tree is read-only

STAT_IDS = {"mean": 0, "sum": 1, "min": 2, "max": 3, "std": 4, "range": 5, "var": 6}


def build(force=False):
    """Returns the path of an up-to-date libxrs_oracle.so: the in-tree one, rebuilt if it is older than
    its source; in a temporary directory instead when the tree is read-only (bench.py must run there)."""
    global _tmp_so
    src = os.path.join(_HERE, "xrs_oracle.c")
    stale = force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src)
    if not stale:
        return _SO
    if os.access(_HERE, os.W_OK):
        out_dir = _HERE
    elif _tmp_so is not None and not force:
        return _tmp_so
    else:
        out_dir = tempfile.mkdtemp(prefix="xrs_oracle_")
    subprocess.check_call(["make", "-f", os.path.join(_HERE, "Makefile"), "-C", out_dir, "-B", "VPATH=" + _HERE,
                           "libxrs_oracle.so"], stdout=subprocess.DEVNULL)
    so = os.path.join(out_dir, "libxrs_oracle.so")
    if out_dir != _HERE:
        _tmp_so = so
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def max_threads():
    return int(lib().xo_max_threads())


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


_i64 = ctypes.c_int64
_dbl = ctypes.c_double
_int = ctypes.c_int


def synth_terrain(rows, cols, row0=0, col0=0, seed=1235, zmin=0.0, zmax=4000.0, nthreads=1):
    """Host twin of the product's benchmark-DEM generator (csrc/synth.cu): the same function of
    (seed, global row, global col), so the CPU arms of bench.py get the benchmark DEM without
    mapping the CUDA library."""
    out = np.empty((rows, cols), np.float32)
    lib().xo_synth_terrain_f32(_p(out), _i64(rows), _i64(cols), _i64(row0), _i64(col0),
                               ctypes.c_uint64(seed), ctypes.c_float(zmin), ctypes.c_float(zmax), _int(nthreads))
    return out


def slope(data, cellsize_x, cellsize_y, nthreads=1):
    """slope.py:56-76 `_cpu`."""
    d = _f32(data)
    out = np.empty(d.shape, np.float32)
    lib().xo_slope_f32(_p(d), _p(out), _i64(d.shape[0]), _i64(d.shape[1]),
                       _dbl(cellsize_x), _dbl(cellsize_y), _int(nthreads))
    return out


def aspect(data, nthreads=1):
    """aspect.py:56-90 `_run_numpy`."""
    d = _f32(data)
    out = np.empty(d.shape, np.float32)
    lib().xo_aspect_f32(_p(d), _p(out), _i64(d.shape[0]), _i64(d.shape[1]), _int(nthreads))
    return out


def curvature(data, cellsize, nthreads=1):
    """curvature.py:44-49 `_run_numpy` -> `_cpu` :31-41."""
    d = _f32(data)
    out = np.empty(d.shape, np.float32)
    lib().xo_curvature_f32(_p(d), _p(out), _i64(d.shape[0]), _i64(d.shape[1]),
                           _dbl(cellsize), _int(nthreads))
    return out


def hillshade(data, azimuth=225, angle_altitude=25, nthreads=1):
    """hillshade.py:20-35 `_run_numpy` (returns float64, see xrs_oracle.c)."""
    d = _f32(data)
    out = np.empty(d.shape, np.float64)
    lib().xo_hillshade_f32(_p(d), _p(out), _i64(d.shape[0]), _i64(d.shape[1]),
                           _dbl(azimuth), _dbl(angle_altitude), _int(nthreads))
    return out


def convolve_2d(data, kernel, nthreads=1):
    """convolution.py:285-313 `_convolve_2d_numpy`."""
    d = _f32(data)
    k = np.ascontiguousarray(kernel, dtype=np.float64)
    out = np.empty(d.shape, np.float32)
    lib().xo_convolve2d_f32(_p(d), _p(k), _int(k.shape[0]), _int(k.shape[1]), _p(out),
                            _i64(d.shape[0]), _i64(d.shape[1]), _int(nthreads))
    return out


def focal_mean(data, passes=1, excludes=(np.nan,), nthreads=1):
    """focal.py:257-259 (astype(float) + passes loop) around `_mean_numpy` :44-67."""
    cur = np.ascontiguousarray(data, dtype=np.float64)
    ex = np.ascontiguousarray(np.asarray(excludes, dtype=np.float64))
    for _ in range(passes):
        out = np.empty(cur.shape, np.float64)
        lib().xo_focal_mean_f64(_p(cur), _p(out), _i64(cur.shape[0]), _i64(cur.shape[1]),
                                _p(ex), _int(ex.size), _int(nthreads))
        cur = out
    return cur


def focal_apply(data, kernel, stat="mean", nthreads=1):
    """focal.py:305-326 `_apply_numpy` with the reducer named `stat` (:268-302)."""
    d = _f32(data)
    k = np.ascontiguousarray(kernel, dtype=np.float64)
    out = np.empty(d.shape, np.float32)
    lib().xo_focal_apply_f32(_p(d), _p(k), _int(k.shape[0]), _int(k.shape[1]),
                             _int(STAT_IDS[stat]), _p(out), _i64(d.shape[0]),
                             _i64(d.shape[1]), _int(nthreads))
    return out


def _ew(name, arrays, scalars=(), nthreads=1):
    arrs = [_f32(a) for a in arrays]
    out = np.empty(arrs[0].shape, np.float32)
    args = [_p(a) for a in arrs] + [_dbl(s) for s in scalars] + [_p(out), _i64(out.size),
                                                                _int(nthreads)]
    getattr(lib(), name)(*args)
    return out


def normalized_ratio(a, b, nthreads=1):
    """multispectral.py:825-841 (ndvi / nbr / nbr2 / ndmi)."""
    return _ew("xo_normalized_ratio_f32", (a, b), nthreads=nthreads)


def savi(nir, red, soil_factor=1.0, nthreads=1):
    """multispectral.py:876-890."""
    return _ew("xo_savi_f32", (nir, red), (soil_factor,), nthreads)


def evi(nir, red, blue, c1=6.0, c2=7.5, soil_factor=1.0, gain=2.5, nthreads=1):
    """multispectral.py:175-188."""
    return _ew("xo_evi_f32", (nir, red, blue), (c1, c2, soil_factor, gain), nthreads)


def arvi(nir, red, blue, nthreads=1):
    """multispectral.py:29-43."""
    return _ew("xo_arvi_f32", (nir, red, blue), nthreads=nthreads)


def gci(nir, green, nthreads=1):
    """multispectral.py:350-360."""
    return _ew("xo_gci_f32", (nir, green), nthreads=nthreads)


def sipi(nir, red, blue, nthreads=1):
    """multispectral.py:1017-1030."""
    return _ew("xo_sipi_f32", (nir, red, blue), nthreads=nthreads)


def ebbi(red, swir, tir, nthreads=1):
    """multispectral.py:1160-1173."""
    return _ew("xo_ebbi_f32", (red, swir, tir), nthreads=nthreads)


# --------------------------------------------------------------------------- zonal
# zonal.py:280-332 `_stats_numpy` restated with NumPy (the arithmetic that matters --
# pairwise float32/float64 summation, two-pass var -- lives inside NumPy itself).
_ZONAL_FUNCS = dict(
    mean=lambda z: z.mean(), max=lambda z: z.max(), min=lambda z: z.min(),
    sum=lambda z: z.sum(), std=lambda z: z.std(), var=lambda z: z.var(),
    count=lambda z: np.ma.count(z),
)


def _majority(z):
    vals, counts = np.unique(z, return_counts=True)
    return vals[np.argmax(counts)]


_ZONAL_FUNCS["majority"] = _majority


def zonal_stats(zones, values, zone_ids=None,
                stats_funcs=("mean", "max", "min", "sum", "std", "var", "count"),
                nodata_values=None):
    """Returns dict(zone=..., <stat>=float64 array...) like the DataFrame columns of
    zonal.py:299-311 (`_sort_and_stride` :121-141, `_calc_stats` :144-163)."""
    zones = np.asarray(zones)
    values = np.asarray(values)
    unique_zones = np.unique(zones[np.isfinite(zones)])
    if zone_ids is None:
        sel = unique_zones
    else:
        sel = np.array([z for z in np.unique(zone_ids) if z in unique_zones],
                       dtype=unique_zones.dtype)
    flat = zones.ravel()
    order = np.argsort(flat)  # same (default, unstable) sort as zonal.py:123
    sorted_zones = flat[order]
    vals_by_zone = values.ravel()[order]
    sorted_zones = sorted_zones[np.isfinite(sorted_zones)]
    breaks = np.searchsorted(sorted_zones, unique_zones, side="right")
    res = {"zone": sel}
    keep = np.isin(unique_zones, sel)
    for name in stats_funcs:
        func = _ZONAL_FUNCS[name]
        col = np.full(unique_zones.shape, np.nan)
        start = 0
        for i in range(len(unique_zones)):
            end = breaks[i]
            if keep[i]:
                zv = vals_by_zone[start:end]
                m = np.isfinite(zv)
                if nodata_values is not None:
                    m &= (zv != nodata_values)
                zv = zv[m]
                if len(zv) > 0:
                    col[i] = func(zv)
            start = end
        res[name] = col[keep]
    return res


# --------------------------------------------------------------------------- hotspots / crosstab
def hotspots(data, kernel, nthreads=1):
    """focal.py:918-937 `_hotspots_numpy` + :881-915 `_calc_hotspots_numpy` (int8)."""
    d = np.asarray(data).astype(np.float32)
    k = np.asarray(kernel, dtype=np.float64)
    mean_array = convolve_2d(d, k / k.sum(), nthreads=nthreads)
    global_mean = np.nanmean(d)
    global_std = np.nanstd(d)
    if global_std == 0:
        raise ZeroDivisionError("Standard deviation of the input raster values is 0.")
    z = (mean_array - global_mean) / global_std
    az = np.abs(z)
    with np.errstate(invalid="ignore"):
        p = np.where(az >= 2.33, 0.0099, np.where(az >= 1.65, 0.0495, np.where(az >= 1.29, 0.0985, 1.0)))
        conf = np.where((az > 2.58) & (p < 0.01), 99, np.where((az > 1.96) & (p < 0.05), 95,
                                                             np.where((az > 1.65) & (p < 0.1), 90, 0)))
        hc = np.where(z > 0, 1, np.where(z < 0, -1, 0))
    return (hc * conf).astype(np.int8)


def crosstab(zones, values, zone_ids=None, cat_ids=None, agg="count", nodata_values=None):
    """zonal.py:748-810 `_crosstab_numpy` for 2-D values: dict(zone=..., <cat>=counts|percentages)."""
    zones = np.asarray(zones)
    values = np.asarray(values)
    valid = np.isfinite(values)
    if nodata_values is not None:
        valid &= values != nodata_values
    unique_cats = np.unique(values[valid])
    cats = unique_cats if cat_ids is None else [c for c in cat_ids if c in unique_cats]
    unique_zones = np.unique(zones[np.isfinite(zones)])
    sel = unique_zones if zone_ids is None else [z for z in zone_ids if z in unique_zones]
    res = {"zone": np.asarray(sel)}
    total = np.array([np.count_nonzero(valid & (zones == z)) for z in sel], dtype=np.float32)
    # zonal.py:719-727: `cat_start` only advances at SELECTED categories, so a selected category
    # also collects the cells of the unselected categories just below it (reference behaviour,
    # kept as is).  With cat_ids=None every category is selected and this is the plain count.
    prev = -np.inf
    for c in sorted(cats):
        cnt = np.array([np.count_nonzero(valid & (zones == z) & (values > prev) & (values <= c)) for z in sel])
        prev = c
        if agg == "percentage":
            t = total.copy()
            t[t == 0] = np.nan
            res[c] = cnt / t * 100
        else:
            res[c] = cnt
    return res


# --------------------------------------------------------------------------- geodesic
def geodesic(data, lat_2d, lon_2d, z_factor=1.0, aspect=False, nthreads=1):
    """slope.py:167-173 / aspect.py:170-176 `_run_numpy_geodesic` -> geodesic.py:179-231."""
    d = np.ascontiguousarray(data, dtype=np.float64)
    la = np.ascontiguousarray(lat_2d, dtype=np.float64)
    lo = np.ascontiguousarray(lon_2d, dtype=np.float64)
    out = np.empty(d.shape, np.float32)
    lib().xo_geodesic_f64(_p(d), _p(la), _p(lo), _p(out), _i64(d.shape[0]), _i64(d.shape[1]), _dbl(z_factor),
                          _int(1 if aspect else 0), _int(nthreads))
    return out
