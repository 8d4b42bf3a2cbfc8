"""ctypes loader of libsplash_cuda.so (the C ABI declared in include/splash_cuda.h).

The library is the only compute path of this package.  If it is missing or cannot create a CUDA
context the package raises -- there is deliberately no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _abi
from .build import LIB_PATH

EXPORTS = (
    "splash_abi_version", "splash_ctx_create", "splash_ctx_destroy", "splash_last_error", "splash_count_months",
    "splash_grid_run", "splash_point_run", "splash_last_stats", "splash_debug_math", "splash_unswc_grid_run",
    "splash_month2day_linear", "splash_ctx_create_multi", "splash_ctx_device_count", "splash_cluster_create",
    "splash_terrain_run", "splash_upslope_area_run", "splash_upslope_dinf_run", "splash_cluster_destroy", "splash_cluster_lanes", "splash_cluster_submit", "splash_cluster_wait", "splash_cluster_last_error",
)

_lib = None


class SplashError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libsplash_cuda error {code}: {msg}")
        self.code = code


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m rsplash_b200.build` "
            "(rsplash_b200 has no CPU implementation to fall back to)")
    lib = C.CDLL(LIB_PATH)
    lib.splash_abi_version.restype = C.c_int
    lib.splash_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.splash_ctx_create.restype = C.c_int
    lib.splash_ctx_destroy.argtypes = [C.c_void_p]
    lib.splash_ctx_destroy.restype = None
    lib.splash_last_error.argtypes = [C.c_void_p]
    lib.splash_last_error.restype = C.c_char_p
    lib.splash_count_months.argtypes = [_abi.c_int32_p, _abi.c_int32_p, C.c_int64]
    lib.splash_count_months.restype = C.c_int64
    lib.splash_grid_run.argtypes = [C.c_void_p, C.POINTER(_abi.SplashGridIn), C.POINTER(_abi.SplashOpts),
                                    C.POINTER(_abi.SplashGridOut)]
    lib.splash_grid_run.restype = C.c_int
    dp = _abi.c_double_p
    ip = _abi.c_int32_p
    lib.splash_point_run.argtypes = [C.c_void_p, C.c_int64, ip, ip, ip, dp, dp, dp, C.c_double, C.c_double, C.c_double,
                                     C.c_double, dp, dp, C.c_int32, C.c_double, C.POINTER(_abi.SplashOpts),
                                     C.POINTER(_abi.SplashGridOut)]
    lib.splash_point_run.restype = C.c_int
    lib.splash_last_stats.argtypes = [C.c_void_p, C.POINTER(_abi.SplashStats)]
    lib.splash_last_stats.restype = C.c_int
    lib.splash_unswc_grid_run.argtypes = [C.c_void_p, C.POINTER(_abi.SplashUnswcIn), C.POINTER(_abi.SplashUnswcOut)]
    lib.splash_unswc_grid_run.restype = C.c_int
    lib.splash_month2day_linear.argtypes = [C.c_void_p, C.POINTER(_abi.SplashM2dIn), C.c_void_p]
    lib.splash_month2day_linear.restype = C.c_int
    lib.splash_debug_math.argtypes = [C.c_void_p, C.c_int, C.c_int64, dp, dp]
    lib.splash_debug_math.restype = C.c_int
    lib.splash_terrain_run.argtypes = [C.c_void_p, C.POINTER(_abi.SplashTerrainIn), C.POINTER(_abi.SplashTerrainOut)]
    lib.splash_terrain_run.restype = C.c_int
    lib.splash_upslope_area_run.argtypes = [C.c_void_p, C.POINTER(_abi.SplashUpslopeIn), C.POINTER(_abi.SplashUpslopeOut)]
    lib.splash_upslope_area_run.restype = C.c_int
    lib.splash_upslope_dinf_run.argtypes = [C.c_void_p, C.POINTER(_abi.SplashDinfIn), C.POINTER(_abi.SplashDinfOut)]
    lib.splash_upslope_dinf_run.restype = C.c_int
    lib.splash_ctx_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
    lib.splash_ctx_create_multi.restype = C.c_int
    lib.splash_ctx_device_count.argtypes = [C.c_void_p]
    lib.splash_ctx_device_count.restype = C.c_int
    lib.splash_cluster_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.splash_cluster_create.restype = C.c_int
    lib.splash_cluster_destroy.argtypes = [C.c_void_p]
    lib.splash_cluster_destroy.restype = None
    lib.splash_cluster_lanes.argtypes = [C.c_void_p]
    lib.splash_cluster_lanes.restype = C.c_int
    lib.splash_cluster_submit.argtypes = [C.c_void_p, C.POINTER(_abi.SplashGridIn), C.POINTER(_abi.SplashOpts),
                                          C.POINTER(_abi.SplashGridOut), C.POINTER(C.c_int64)]
    lib.splash_cluster_submit.restype = C.c_int
    lib.splash_cluster_wait.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(_abi.SplashStats)]
    lib.splash_cluster_wait.restype = C.c_int
    lib.splash_cluster_last_error.argtypes = [C.c_void_p]
    lib.splash_cluster_last_error.restype = C.c_char_p
    if lib.splash_abi_version() != _abi.SPLASH_ABI_VERSION:
        raise ImportError("libsplash_cuda ABI version mismatch; rebuild with `python -m rsplash_b200.build`")
    _lib = lib
    return lib


class Context:
    """The reference's worker pool (raster::beginCluster, R/splash.grid.R:32-39): one GPU, or -- with a sequence of
    device ordinals -- several GPUs of the host, over which splash_grid_run schedules the call's row blocks."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            arr = (C.c_int * len(device))(*[int(d) for d in device])
            rc = self.lib.splash_ctx_create_multi(arr, len(device), C.byref(h))
        else:
            rc = self.lib.splash_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise SplashError(rc, self.lib.splash_last_error(None).decode())
        self.handle = h
        self.device = device

    @property
    def n_devices(self) -> int:
        return self.lib.splash_ctx_device_count(self.handle)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.splash_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def check(self, rc: int):
        if rc != 0:
            raise SplashError(rc, self.lib.splash_last_error(self.handle).decode())

    def grid_run(self, cin: _abi.SplashGridIn, opts: _abi.SplashOpts, cout: _abi.SplashGridOut):
        self.check(self.lib.splash_grid_run(self.handle, C.byref(cin), C.byref(opts), C.byref(cout)))

    def point_run(self, n_days, year, doy, month, sw_in, tc, pn, lat, elev, slop, asp, soil_data, au, resolution,
                  opts: _abi.SplashOpts, cout: _abi.SplashGridOut):
        """splash_point_run: splash.point() of the reference (R/splash.point.R:29), one cell, host vectors."""
        p = lambda a: a.ctypes.data_as(_abi.c_double_p)
        ip = lambda a: a.ctypes.data_as(_abi.c_int32_p)
        self.check(self.lib.splash_point_run(self.handle, int(n_days), ip(year), ip(doy), ip(month), p(sw_in), p(tc), p(pn),
                                             float(lat), float(elev), float(slop), float(asp), p(soil_data), p(au), int(au.size),
                                             float(resolution), C.byref(opts), C.byref(cout)))

    def debug_math(self, op: str, x):
        """exp / log / acos / sin of the day step evaluated on the device (diagnostic); the `*_body` ops are the
        guard-free fast-range bodies of the branch-light day step (NaN outside their guards), `sqrt` / `div` the
        compiler's own expansions they must equal (div: second operand x[(7919 i + 13) mod n])."""
        import numpy as np

        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty_like(x)
        self.check(self.lib.splash_debug_math(self.handle, ("exp", "log", "acos", "sin", "acos_body", "sqrt_body", "sqrt", "div_body", "div", "exp_body", "log_body").index(op), x.size,
                                              x.ctypes.data_as(_abi.c_double_p), y.ctypes.data_as(_abi.c_double_p)))
        return y

    def stats(self) -> dict:
        s = _abi.SplashStats()
        self.check(self.lib.splash_last_stats(self.handle, C.byref(s)))
        return s.as_dict()


class Cluster:
    """Block scheduler: the reference's sendCall / recvOneData loop (R/splash.grid.R:312-314, 359-400).
    submit() returns a ticket at once; wait() returns (ticket, stats) of a finished block.  The arrays behind the
    structs must stay alive and untouched until the block has been waited for (keep them in `keep`)."""

    def __init__(self, devices=(0,), lanes_per_device: int = 2):
        self.lib = load()
        h = C.c_void_p()
        arr = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self.lib.splash_cluster_create(arr, len(devices), int(lanes_per_device), C.byref(h))
        if rc != 0:
            raise SplashError(rc, self.lib.splash_last_error(None).decode())
        self.handle = h
        self._keep = {}

    @property
    def lanes(self) -> int:
        return self.lib.splash_cluster_lanes(self.handle)

    def submit(self, cin, opts, cout, keep=None) -> int:
        t = C.c_int64()
        rc = self.lib.splash_cluster_submit(self.handle, C.byref(cin), C.byref(opts), C.byref(cout), C.byref(t))
        if rc != 0:
            raise SplashError(rc, self.lib.splash_cluster_last_error(self.handle).decode())
        self._keep[t.value] = (cin, opts, cout, keep)
        return t.value

    def wait(self, ticket: int = -1):
        done = C.c_int64()
        st = _abi.SplashStats()
        rc = self.lib.splash_cluster_wait(self.handle, int(ticket), C.byref(done), C.byref(st))
        if rc != 0:
            msg = self.lib.splash_cluster_last_error(self.handle).decode()
            self._keep.pop(done.value, None)
            raise SplashError(rc, msg)
        self._keep.pop(done.value, None)
        return done.value, st.as_dict()

    def close(self):
        if getattr(self, "handle", None):
            self.lib.splash_cluster_destroy(self.handle)
            self.handle = None
            self._keep.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
