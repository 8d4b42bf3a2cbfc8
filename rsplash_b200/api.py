"""Host-side mirror of the reference's R entry points for the hot path.

`splash_point` and `splash_grid` keep the argument names and meaning of the R functions
(reference R/splash.point.R:29, and the mapply() argument set of R/splash.grid.R:291-304) and
return the same nine layers (R/splash.grid.R:449).  They only marshal numpy arrays into the C ABI
(include/splash_cuda.h); all arithmetic happens in libsplash_cuda's CUDA kernels.

What stays outside (as in the survey's scope table): raster I/O (slope, aspect, upslope area, latitude and
resolution are *inputs* of splash_grid, as they are for splash.point; `terrain` and `upslope_area` derive them), and
the random monthly->daily rain disaggregation (the deterministic interpolation of monthly temperature and
radiation is `month2day_linear`).
"""
from __future__ import annotations

import ctypes as C
from typing import Mapping, Sequence

import numpy as np

from . import _abi
from ._lib import Cluster, Context, SplashError  # noqa: F401

_default_ctx: dict = {}


def default_context(device=0) -> Context:
    """The process-wide context of a device (or of a tuple of devices: a multi-GPU context)."""
    key = tuple(device) if isinstance(device, (list, tuple)) else device
    if key not in _default_ctx:
        _default_ctx[key] = Context(list(key) if isinstance(key, tuple) else key)
    return _default_ctx[key]


def _f64(a, shape=None, name=""):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError(f"{name}: expected shape {shape}, got {a.shape}")
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def splash_grid(sw_in, tc, pn, lat, elev, slop, asp, soil_data, Au, resolution, time_index,
                monthly_out: bool = True, ctx: Context | None = None, outputs: Sequence[str] = _abi.OUTPUT_NAMES,
                return_state: bool = False, return_diag: bool = False, state_init=None, tile_cells: int = 0,
                max_spin: int = 0, spin_tol_mm: float = 0.0) -> dict:
    """Run a block of cells: the body of the reference's worker function `clFun`.

    sw_in, tc, pn   [n_days, n_cells] daily forcing (float64, or float32 to use the f32 path)
    lat, elev, slop, asp, resolution   [n_cells]
    soil_data       [6, n_cells]  sand %, clay %, OM %, gravel %, bulk density (NaN = derive), depth m
    Au              [n_cells] upslope area, or [3, n_cells] with the in/out neighbour counts
    time_index      datetime64[D] axis of the forcing (n_days)
    monthly_out     sim.control$monthly_out of splash.grid (default TRUE there)

    Returns {layer: [n_out, n_cells]} for wn, ro, pet, aet, snow, cond, bflow, netr, sm_lim.
    """
    ctx = ctx or default_context()
    sw_in = np.asarray(sw_in)
    f32 = sw_in.dtype == np.float32
    fdt = np.float32 if f32 else np.float64
    sw_in = np.ascontiguousarray(sw_in, dtype=fdt)
    if sw_in.ndim != 2:
        raise ValueError("sw_in must be [n_days, n_cells]")
    n_days, n_cells = sw_in.shape
    tc = np.ascontiguousarray(tc, dtype=fdt)
    pn = np.ascontiguousarray(pn, dtype=fdt)
    if tc.shape != sw_in.shape or pn.shape != sw_in.shape:
        raise ValueError("sw_in, tc and pn must have the same shape")
    year, doy, month = _abi.time_axes(time_index)
    if len(year) != n_days:
        raise ValueError("time_index length does not match the forcing")
    lat = _f64(lat, (n_cells,), "lat")
    elev = _f64(elev, (n_cells,), "elev")
    slop = _f64(slop, (n_cells,), "slop")
    asp = _f64(asp, (n_cells,), "asp")
    resolution = _f64(np.broadcast_to(np.asarray(resolution, dtype=np.float64), (n_cells,)), (n_cells,), "resolution")
    soil = _f64(soil_data, (6, n_cells), "soil_data")
    au = np.asarray(Au, dtype=np.float64)
    if au.ndim == 1:
        au = au[None, :]
    au = _f64(au, name="Au")
    if au.shape not in ((1, n_cells), (3, n_cells)):
        raise ValueError("Au must be [n_cells] or [3, n_cells]")

    n_out = _abi.count_months(year, month) if monthly_out else n_days
    cin = _abi.SplashGridIn()
    cin.n_cells, cin.n_days, cin.cell_stride = n_cells, n_days, n_cells
    cin.year = year.ctypes.data_as(_abi.c_int32_p)
    cin.doy = doy.ctypes.data_as(_abi.c_int32_p)
    cin.month = month.ctypes.data_as(_abi.c_int32_p)
    cin.sw_in, cin.tc, cin.pn = _ptr(sw_in), _ptr(tc), _ptr(pn)
    cin.lat, cin.elev, cin.slop, cin.asp, cin.resolution = _ptr(lat), _ptr(elev), _ptr(slop), _ptr(asp), _ptr(resolution)
    cin.soil, cin.au, cin.au_layers = _ptr(soil), _ptr(au), au.shape[0]
    cin.mem_kind = _abi.SPLASH_MEM_HOST
    cin.forcing_dtype = _abi.SPLASH_F32 if f32 else _abi.SPLASH_F64

    result = {}
    cout = _abi.SplashGridOut()
    cout.n_out, cout.cell_stride, cout.mem_kind = n_out, n_cells, _abi.SPLASH_MEM_HOST
    for k in outputs:
        if k not in _abi.OUTPUT_NAMES:
            raise ValueError(f"unknown output layer {k!r}")
        result[k] = np.empty((n_out, n_cells), dtype=np.float64)
        setattr(cout, k, _ptr(result[k]))
    if return_state:
        result["state_final"] = np.empty((_abi.SPLASH_NSTATE, n_cells))
        cout.state_final = _ptr(result["state_final"])
    if return_diag:
        result["cell_diag"] = np.empty((_abi.SPLASH_NDIAG, n_cells))
        cout.cell_diag = _ptr(result["cell_diag"])

    opts = _abi.SplashOpts()
    opts.monthly_out = int(bool(monthly_out))
    opts.tile_cells = int(tile_cells)
    opts.max_spin = int(max_spin)
    opts.spin_tol_mm = float(spin_tol_mm)
    if state_init is not None:
        st = _f64(state_init, (_abi.SPLASH_NSTATE, n_cells), "state_init")
        opts.skip_spinup, opts.state_init = 1, _ptr(st)
    ctx.grid_run(cin, opts, cout)
    result["stats"] = ctx.stats()
    return result


def splash_point(sw_in, tc, pn, lat, elev, slop=0.0, asp=0.0, soil_data=None, Au=0.0, resolution=250.0,
                 time_index=None, monthly_out: bool = False, ctx: Context | None = None, return_state: bool = False,
                 return_diag: bool = False) -> dict:
    """splash.point(sw_in, tc, pn, lat, elev, slop, asp, soil_data, Au, resolution, time_index, monthly_out).

    One cell through the C entry `splash_point_run`; same defaults as the R function (R/splash.point.R:29).
    Returns {layer: [n_out]}.
    """
    if soil_data is None or time_index is None:
        raise ValueError("soil_data and time_index are required")
    ctx = ctx or default_context()
    au = np.ascontiguousarray(np.atleast_1d(np.asarray(Au, dtype=np.float64)))
    if au.size not in (1, 3):
        raise ValueError("Au must have 1 or 3 elements")
    vec = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))
    sw_in, tc, pn = vec(sw_in), vec(tc), vec(pn)
    soil = vec(soil_data)
    if soil.size != 6:
        raise ValueError("soil_data must have six elements")
    year, doy, month = _abi.time_axes(time_index)
    n_days = len(year)
    if not (len(sw_in) == len(tc) == len(pn) == n_days):
        raise ValueError("sw_in, tc, pn and time_index must have the same length")
    n_out = _abi.count_months(year, month) if monthly_out else n_days
    result = {k: np.empty(n_out) for k in _abi.OUTPUT_NAMES}
    cout = _abi.SplashGridOut()
    cout.n_out, cout.cell_stride, cout.mem_kind = n_out, 1, _abi.SPLASH_MEM_HOST
    for k in _abi.OUTPUT_NAMES:
        setattr(cout, k, _ptr(result[k]))
    if return_state:
        result["state_final"] = np.empty(_abi.SPLASH_NSTATE)
        cout.state_final = _ptr(result["state_final"])
    if return_diag:
        result["cell_diag"] = np.empty(_abi.SPLASH_NDIAG)
        cout.cell_diag = _ptr(result["cell_diag"])
    opts = _abi.SplashOpts()
    opts.monthly_out = int(bool(monthly_out))
    ctx.point_run(n_days, year, doy, month, sw_in, tc, pn, lat, elev, slop, asp, soil, au, resolution, opts, cout)
    result["stats"] = ctx.stats()
    return result


def unSWC_grid(soil_data, uns_depth: float, wn, ctx: Context | None = None) -> dict:
    """unSWC.grid(soil_data, uns_depth, wn) of the reference (R/unsSWC.grid.R:14): unsaturated-zone diagnostics.

    soil_data  [6, n_cells] as for splash_grid;  wn  [n_layers, n_cells] simulated soil water, mm;  uns_depth  m.
    Returns {w_z, wtd, Se} like the R function, plus theta_i (which R writes to the theta_mean file).
    """
    ctx = ctx or default_context()
    wn = np.ascontiguousarray(wn, dtype=np.float64)
    if wn.ndim != 2:
        raise ValueError("wn must be [n_layers, n_cells]")
    n_layers, n_cells = wn.shape
    soil = _f64(soil_data, (6, n_cells), "soil_data")
    cin = _abi.SplashUnswcIn()
    cin.n_cells, cin.n_layers, cin.cell_stride = n_cells, n_layers, n_cells
    cin.soil, cin.wn, cin.uns_depth, cin.mem_kind = _ptr(soil), _ptr(wn), float(uns_depth), _abi.SPLASH_MEM_HOST
    res = {k: np.empty((n_layers, n_cells)) for k in ("theta_i", "wtd", "w_z", "Se")}
    cout = _abi.SplashUnswcOut()
    cout.cell_stride, cout.mem_kind = n_cells, _abi.SPLASH_MEM_HOST
    cout.theta_i, cout.wtd, cout.w_z, cout.se = _ptr(res["theta_i"]), _ptr(res["wtd"]), _ptr(res["w_z"]), _ptr(res["Se"])
    ctx.check(ctx.lib.splash_unswc_grid_run(ctx.handle, C.byref(cin), C.byref(cout)))
    return res


def terrain(elev, ymax: float, xres: float, yres: float, lonlat: bool = True, ctx: Context | None = None) -> dict:
    """What splash.grid derives from the DEM before the hot path (R/splash.grid.R:95-110, R/upslope_area.R:27-29,
    140-165): slope and aspect (degrees, NA of valid cells -> 0), latitude, resolution = sqrt(cell area) in m, D8 flow
    direction and the cells draining in / out.  elev: [n_rows, n_cols], north row first.  Parity unpinned (raster::terrain
    and raster::area are third-party; see include/splash_cuda.h)."""
    ctx = ctx or default_context()
    z = np.ascontiguousarray(elev, dtype=np.float64)
    if z.ndim != 2:
        raise ValueError("elev must be [n_rows, n_cols]")
    cin = _abi.SplashTerrainIn()
    cin.n_rows, cin.n_cols, cin.elev = z.shape[0], z.shape[1], _ptr(z)
    cin.ymax, cin.xres, cin.yres, cin.lonlat, cin.mem_kind = float(ymax), float(xres), float(yres), int(bool(lonlat)), _abi.SPLASH_MEM_HOST
    res = {k: np.empty(z.shape) for k in ("slope", "aspect", "lat", "resolution", "flowdir", "ncellin", "ncellout")}
    cout = _abi.SplashTerrainOut()
    for k, v in res.items():
        setattr(cout, k, _ptr(v))
    ctx.check(ctx.lib.splash_terrain_run(ctx.handle, C.byref(cin), C.byref(cout)))
    return res


def _upslope_au(entry, cin, cout, counters, optional, elev, ymax, xres, yres, lonlat, ctx, in_ptr, out_ptr, shape) -> dict:
    """The marshalling upslope_area and upslope_areav2 share: fill the geometry of `cin` and cout.area, pass the
    optional [n_rows, n_cols] outputs {field: (wanted on the host, device address or None)}, call `entry`, then
    splash_terrain_run for the two count layers of Au."""
    ctx = ctx or default_context()
    if (in_ptr is None) != (out_ptr is None):
        raise ValueError("in_ptr and out_ptr go together")
    device = in_ptr is not None
    if device:
        if shape is None:
            raise ValueError("shape is required with device pointers")
        nr, nc = (int(s) for s in shape)
    else:
        z = np.ascontiguousarray(elev, dtype=np.float64)
        if z.ndim != 2:
            raise ValueError("elev must be [n_rows, n_cols]")
        nr, nc = z.shape
        au = np.empty((3, nr, nc))
        extra = {k: np.empty((nr, nc)) for k, (want, _) in optional.items() if want}
    n = nr * nc
    mem = _abi.SPLASH_MEM_DEVICE if device else _abi.SPLASH_MEM_HOST
    elev_p = C.c_void_p(int(in_ptr)) if device else _ptr(z)
    au_addr = int(out_ptr) if device else au.ctypes.data
    layer = lambda k: C.c_void_p(au_addr + k * n * 8) if n else None

    cin.n_rows, cin.n_cols, cin.elev = nr, nc, elev_p
    cin.ymax, cin.xres, cin.yres, cin.lonlat, cin.mem_kind = float(ymax), float(xres), float(yres), int(bool(lonlat)), mem
    cout.area = layer(0)
    for k, (_, dptr) in optional.items():
        if device:
            setattr(cout, k, None if dptr is None else C.c_void_p(int(dptr)))
        else:
            setattr(cout, k, _ptr(extra.get(k)))
    ctx.check(getattr(ctx.lib, entry)(ctx.handle, C.byref(cin), C.byref(cout)))

    tin = _abi.SplashTerrainIn()
    tin.n_rows, tin.n_cols, tin.elev = nr, nc, elev_p
    tin.ymax, tin.xres, tin.yres, tin.lonlat, tin.mem_kind = cin.ymax, cin.xres, cin.yres, cin.lonlat, mem
    tout = _abi.SplashTerrainOut()
    tout.ncellin, tout.ncellout = layer(1), layer(2)
    ctx.check(ctx.lib.splash_terrain_run(ctx.handle, C.byref(tin), C.byref(tout)))

    res = {k: int(getattr(cout, k)) for k in counters}
    if not device:
        res.update(area=au[0], ncellin=au[1], ncellout=au[2], Au=au, **extra)
    return res


def upslope_area(elev, ymax: float, xres: float, yres: float, lonlat: bool = True, min_slope_deg: float = 0.1,
                 ctx: Context | None = None, return_filled: bool = False, in_ptr: int | None = None,
                 out_ptr: int | None = None, filled_ptr: int | None = None, shape: tuple | None = None) -> dict:
    """upslope_area() of the reference (R/upslope_area.R:12-58, small-grid branch): the contributing area of every cell
    (topmodel::sinkfill, then topidx's multiple-flow-direction area; see include/splash_cuda.h for the definition,
    PARITY UNPINNED) and the in / out neighbour counts of splash_terrain_run.

    elev  [n_rows, n_cols], north row first, NaN = NA;  min_slope_deg  the fill's minimum slope (sinkfill's `degree`).
    Returns {area, ncellin, ncellout, Au, fill_sweeps, accum_rounds[, filled]}: Au is the [3, n_rows, n_cols] stack
    (area m2, ncellin, ncellout) that splash_grid takes per cell, and area / ncellin / ncellout are its layers.
    With in_ptr / out_ptr (device addresses of the [n_rows, n_cols] float64 DEM and of a [3, n_rows, n_cols] float64
    array that receives Au, e.g. torch tensors' data_ptr()) and shape = (n_rows, n_cols), everything stays in HBM
    (filled_ptr: optional [n_rows, n_cols] float64 for the filled DEM) and only the two counters are returned.
    """
    cin = _abi.SplashUpslopeIn()
    cin.min_slope_deg = float(min_slope_deg)
    return _upslope_au("splash_upslope_area_run", cin, _abi.SplashUpslopeOut(), ("fill_sweeps", "accum_rounds"),
                       {"filled": (return_filled, filled_ptr)}, elev, ymax, xres, yres, lonlat, ctx, in_ptr, out_ptr, shape)


def upslope_areav2(elev, ymax: float, xres: float, yres: float, lonlat: bool = True, ctx: Context | None = None,
                   return_filled: bool = False, return_angle: bool = False, in_ptr: int | None = None,
                   out_ptr: int | None = None, filled_ptr: int | None = None, angle_ptr: int | None = None,
                   shape: tuple | None = None) -> dict:
    """upslope_areav2() of the reference (R/upslope_area.R:59-137, the branch for coarse or large grids that calls
    TauDEM): pit removal to flat, D-infinity flow directions with flats resolved (Garbrecht and Martz), and the
    D-infinity contributing area (see include/splash_cuda.h, splash_upslope_dinf_run, PARITY UNPINNED); with the in /
    out neighbour counts of splash_terrain_run.

    Arguments and results as upslope_area (no min_slope_deg: the fill is to flat), plus the counter flat_rounds and,
    with return_angle (or angle_ptr on the device path), `angle`: the flow angle in radians counter-clockwise from
    east in [0, 2 pi), NaN where a cell has no direction (NA cells, boundary cells).
    """
    return _upslope_au("splash_upslope_dinf_run", _abi.SplashDinfIn(), _abi.SplashDinfOut(),
                       ("fill_sweeps", "flat_rounds", "accum_rounds"),
                       {"filled": (return_filled, filled_ptr), "angle": (return_angle, angle_ptr)},
                       elev, ymax, xres, yres, lonlat, ctx, in_ptr, out_ptr, shape)


def month_starts(time_index_month, time_index) -> np.ndarray:
    """0-based position on the daily axis of each month's first day (time_index_month - time_index[1])."""
    tm = np.asarray(time_index_month, dtype="datetime64[D]")
    t0 = np.asarray(time_index, dtype="datetime64[D]")[0]
    return ((tm - t0) / np.timedelta64(1, "D")).astype(np.int32)


def month2day_linear(monthly, time_index_month, time_index, ctx: Context | None = None, dtype=np.float64,
                     out_ptr: int | None = None, in_ptr: int | None = None, n_cells: int | None = None):
    """approx(time_index_month, x, time_index, method = "linear", rule = 2)$y for every cell of a block: what
    splash.point does to monthly tc and sw_in before anything else (R/splash.point.R:74-84).

    monthly  [n_months, n_cells] (NaN = NA);  time_index_month  datetime64 month starts;  time_index  the daily axis.
    Returns [n_days, n_cells] in `dtype` (float64, or float32 = the f32 forcing layout of splash_grid).
    With in_ptr / out_ptr (device addresses of [n_months, n_cells] float64 and [n_days, n_cells] dtype arrays, e.g.
    torch tensors' data_ptr()) the series are produced in HBM and nothing is returned.
    """
    ctx = ctx or default_context()
    xs = np.ascontiguousarray(month_starts(time_index_month, time_index))
    n_days = len(np.asarray(time_index))
    f32 = np.dtype(dtype) == np.float32
    if not f32 and np.dtype(dtype) != np.float64:
        raise ValueError("dtype must be float64 or float32")
    cin = _abi.SplashM2dIn()
    cin.month_start = xs.ctypes.data_as(C.c_void_p)
    cin.out_f32 = int(f32)
    if (in_ptr is None) != (out_ptr is None):
        raise ValueError("in_ptr and out_ptr go together")
    if in_ptr is not None:
        if n_cells is None:
            raise ValueError("n_cells is required with device pointers")
        cin.n_cells, cin.n_months, cin.n_days = int(n_cells), len(xs), n_days
        cin.monthly, cin.mem_kind = C.c_void_p(int(in_ptr)), _abi.SPLASH_MEM_DEVICE
        ctx.check(ctx.lib.splash_month2day_linear(ctx.handle, C.byref(cin), C.c_void_p(int(out_ptr))))
        return None
    monthly = np.ascontiguousarray(monthly, dtype=np.float64)
    if monthly.ndim != 2 or monthly.shape[0] != len(xs):
        raise ValueError("monthly must be [n_months, n_cells] with one row per element of time_index_month")
    cin.n_cells, cin.n_months, cin.n_days = monthly.shape[1], monthly.shape[0], n_days
    cin.monthly, cin.mem_kind = _ptr(monthly), _abi.SPLASH_MEM_HOST
    out = np.empty((n_days, monthly.shape[1]), dtype=dtype)
    ctx.check(ctx.lib.splash_month2day_linear(ctx.handle, C.byref(cin), _ptr(out)))
    return out
