"""CPU-only: the C-ABI library loads and exports every symbol include/xrs_b200.h declares;
the product refuses to run without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "xrs_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(xrs_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_hot_path():
    syms = header_symbols()
    for s in ("xrs_slope_f32", "xrs_aspect_f32", "xrs_curvature_f32", "xrs_hillshade_f32",
              "xrs_surface_suite_f32", "xrs_focal_mean_f32", "xrs_focal_mean_f64", "xrs_convolve2d_f32",
              "xrs_focal_stat_f32", "xrs_normalized_ratio_f32", "xrs_savi_f32", "xrs_evi_f32",
              "xrs_zonal_hash_run", "xrs_zonal_hash_second_pass", "xrs_host_stencil"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    import xrspatial_b200
    lib = xrspatial_b200._lib.lib()
    for s in header_symbols():
        assert hasattr(lib, s), "libxrs_b200.so does not export %s" % s
    assert lib.xrs_abi_version() == 1


def test_ctypes_prototypes_cover_the_header():
    import xrspatial_b200
    xrspatial_b200._lib.lib()
    declared = set(header_symbols()) - {"xrs_last_error_string"}
    assert declared <= set(xrspatial_b200._lib.EXPORTS), declared - set(xrspatial_b200._lib.EXPORTS)


def test_no_cpu_fallback_without_gpu():
    """The host path needs the device and fails loudly without one.  Checked in a fresh interpreter that
    sees no CUDA device, so that GPU hosts check it too."""
    pytest.importorskip("torch")
    code = "\n".join([
        "import numpy as np",
        "import xrspatial_b200 as xb",
        "agg = xb.DataArray(np.zeros((8, 8), np.float32), attrs={'res': (1, 1)})",
        "for name, f in (('slope', lambda: xb.slope(agg)), ('ndvi', lambda: xb.ndvi(agg, agg))):",
        "    try:",
        "        f()",
        "    except RuntimeError:",
        "        continue",
        "    raise SystemExit('%s computed without a CUDA device' % name)",
    ])
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-s", "-c", code], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_argument_errors_do_not_need_a_gpu():
    import xrspatial_b200
    lib = xrspatial_b200._lib.lib()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    k = (ctypes.c_double * 4)(1, 1, 1, 1)
    # even kernel -> XRS_EINVAL before any CUDA call
    rc = lib.xrs_convolve2d_f32(p, 16, ctypes.c_void_p(ctypes.addressof(buf) + 32), 16, 2, 4,
                                ctypes.cast(k, ctypes.c_void_p), 2, 2, None)
    assert rc == -1
    assert b"odd" in lib.xrs_last_error_string()
    rc = lib.xrs_slope_f32(p, 8, p, 16, 2, 4, 1.0, 1.0, None)   # pitch < row bytes
    assert rc == -1
    with pytest.raises(ValueError):
        xrspatial_b200._lib.check(rc)
