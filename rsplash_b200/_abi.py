"""ctypes mirror of include/splash_cuda.h (struct layouts, constants, small helpers).

Kept free of any library loading so that the product binding (rsplash_b200/_lib.py) and test-side
harnesses can share the layouts.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

SPLASH_ABI_VERSION = 7
SPLASH_NSTATE = 7

SPLASH_OK, SPLASH_ERR_BAD_ARG, SPLASH_ERR_CUDA, SPLASH_ERR_NOMEM, SPLASH_ERR_NO_DEVICE = range(5)
SPLASH_MEM_HOST, SPLASH_MEM_DEVICE = 0, 1
SPLASH_F64, SPLASH_F32 = 0, 1

DIAG_NAMES = (
    "SAT", "WP", "FC", "Ksat", "lambda", "depth", "bub_press", "RES", "Wmax_R", "Tt", "AI",
    "spin_passes", "snow_days", "snowfall_days",
)
SPLASH_NDIAG = len(DIAG_NAMES)

# order of the nine output layers: result[1:8] of R/splash.point.R:182 plus sm_lim (:201)
OUTPUT_NAMES = ("wn", "ro", "pet", "aet", "snow", "cond", "bflow", "netr", "sm_lim")
# monthly aggregation rule, R/splash.point.R:210-211
MONTHLY_MEAN = ("wn", "snow", "sm_lim")
STATE_NAMES = ("wn", "snow", "qin", "td", "nd")  # rows 0..4 of state_final; row 5 the aridity index, row 6 Tt

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)


class SplashGridIn(C.Structure):
    _fields_ = [
        ("n_cells", C.c_int64),
        ("n_days", C.c_int64),
        ("cell_stride", C.c_int64),
        ("year", c_int32_p),
        ("doy", c_int32_p),
        ("month", c_int32_p),
        ("sw_in", C.c_void_p),
        ("tc", C.c_void_p),
        ("pn", C.c_void_p),
        ("lat", C.c_void_p),
        ("elev", C.c_void_p),
        ("slop", C.c_void_p),
        ("asp", C.c_void_p),
        ("resolution", C.c_void_p),
        ("soil", C.c_void_p),
        ("au", C.c_void_p),
        ("au_layers", C.c_int32),
        ("mem_kind", C.c_int32),
        ("forcing_dtype", C.c_int32),
        ("reserved", C.c_int32),
        ("attr_stride", C.c_int64),
    ]


class SplashGridOut(C.Structure):
    _fields_ = [
        ("n_out", C.c_int64),
        ("cell_stride", C.c_int64),
        ("wn", C.c_void_p),
        ("ro", C.c_void_p),
        ("pet", C.c_void_p),
        ("aet", C.c_void_p),
        ("snow", C.c_void_p),
        ("cond", C.c_void_p),
        ("bflow", C.c_void_p),
        ("netr", C.c_void_p),
        ("sm_lim", C.c_void_p),
        ("state_final", C.c_void_p),
        ("cell_diag", C.c_void_p),
        ("mem_kind", C.c_int32),
        ("reserved", C.c_int32),
        ("aux_stride", C.c_int64),
    ]


class SplashOpts(C.Structure):
    _fields_ = [
        ("monthly_out", C.c_int32),
        ("max_spin", C.c_int32),
        ("spin_tol_mm", C.c_double),
        ("tile_cells", C.c_int64),
        ("skip_spinup", C.c_int32),
        ("reserved", C.c_int32),
        ("state_init", C.c_void_p),
        ("state_stride", C.c_int64),
    ]


class SplashUnswcIn(C.Structure):
    _fields_ = [
        ("n_cells", C.c_int64), ("n_layers", C.c_int64), ("cell_stride", C.c_int64),
        ("soil", C.c_void_p), ("wn", C.c_void_p), ("uns_depth", C.c_double),
        ("mem_kind", C.c_int32), ("reserved", C.c_int32),
    ]


class SplashUnswcOut(C.Structure):
    _fields_ = [
        ("cell_stride", C.c_int64), ("theta_i", C.c_void_p), ("wtd", C.c_void_p), ("w_z", C.c_void_p), ("se", C.c_void_p),
        ("mem_kind", C.c_int32), ("reserved", C.c_int32),
    ]


class SplashM2dIn(C.Structure):
    _fields_ = [
        ("n_cells", C.c_int64), ("n_months", C.c_int64), ("n_days", C.c_int64), ("in_stride", C.c_int64), ("out_stride", C.c_int64),
        ("month_start", C.c_void_p), ("monthly", C.c_void_p), ("mem_kind", C.c_int32), ("out_f32", C.c_int32),
    ]


class SplashTerrainIn(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64), ("n_cols", C.c_int64), ("elev", C.c_void_p), ("ymax", C.c_double), ("xres", C.c_double),
        ("yres", C.c_double), ("lonlat", C.c_int32), ("mem_kind", C.c_int32),
    ]


class SplashTerrainOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("slope", "aspect", "lat", "resolution", "flowdir", "ncellin", "ncellout")]


class SplashUpslopeIn(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64), ("n_cols", C.c_int64), ("elev", C.c_void_p), ("ymax", C.c_double), ("xres", C.c_double),
        ("yres", C.c_double), ("lonlat", C.c_int32), ("mem_kind", C.c_int32), ("min_slope_deg", C.c_double),
    ]


class SplashUpslopeOut(C.Structure):
    _fields_ = [("area", C.c_void_p), ("filled", C.c_void_p), ("fill_sweeps", C.c_int64), ("accum_rounds", C.c_int64)]


class SplashDinfIn(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64), ("n_cols", C.c_int64), ("elev", C.c_void_p), ("ymax", C.c_double), ("xres", C.c_double),
        ("yres", C.c_double), ("lonlat", C.c_int32), ("mem_kind", C.c_int32),
    ]


class SplashDinfOut(C.Structure):
    _fields_ = [("area", C.c_void_p), ("filled", C.c_void_p), ("angle", C.c_void_p), ("fill_sweeps", C.c_int64),
                ("flat_rounds", C.c_int64), ("accum_rounds", C.c_int64)]


class SplashStats(C.Structure):
    _fields_ = [
        ("h2d_ms", C.c_double),
        ("setup_ms", C.c_double),
        ("first_ms", C.c_double),
        ("rounds_ms", C.c_double),
        ("bulk_ms", C.c_double),
        ("bulk_span_ms", C.c_double),
        ("d2h_ms", C.c_double),
        ("pool_wait_ms", C.c_double),
        ("scatter_ms", C.c_double),
        ("gpu_ms", C.c_double),
        ("total_ms", C.c_double),
        ("h2d_bytes", C.c_int64),
        ("d2h_bytes", C.c_int64),
        ("spin_cell_days", C.c_int64),
        ("main_cell_days", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("unconverged_cells", C.c_int64),
        ("cycle_cells", C.c_int64),
        ("n_tiles", C.c_int64),
        ("tile_cells", C.c_int64),
        ("pool_cells", C.c_int64),
        ("pool_overflow_cells", C.c_int64),
        ("pool_max_passes", C.c_int64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


def time_axes(dates) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """year / day-of-year / month int32 vectors of a datetime64[D] axis.

    Mirrors format(time_index, '%Y' | '%j' | '%m') at R/splash.point.R:57-59,547.
    """
    d = np.asarray(dates, dtype="datetime64[D]")
    y = d.astype("datetime64[Y]")
    m = d.astype("datetime64[M]")
    year = (y.astype(np.int64) + 1970).astype(np.int32)
    doy = ((d - y.astype("datetime64[D]")).astype(np.int64) + 1).astype(np.int32)
    month = ((m - y.astype("datetime64[M]")).astype(np.int64) + 1).astype(np.int32)
    return year, doy, month


def count_months(year: np.ndarray, month: np.ndarray) -> int:
    """Number of (year, month) runs == length(ztime.months), R/splash.grid.R:163,175."""
    if len(year) == 0:
        return 0
    key = year.astype(np.int64) * 16 + month.astype(np.int64)
    return int(1 + np.count_nonzero(key[1:] != key[:-1]))
