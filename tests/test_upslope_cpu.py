"""CPU: the numpy restatement of the upslope contributing area (tests/upslope_oracle.py; PARITY UNPINNED, see
include/splash_cuda.h).  Its priority-flood fill equals a brute-force Jacobi fixpoint bit for bit, the filled surface
satisfies the fill condition, the MFD accumulation conserves area and has the closed forms of a ramp and the
symmetries of a cone; the C structs match their ctypes mirror and the new kernels compile for sm_100a without
spills."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from rsplash_b200 import _abi, build
from tests import upslope_oracle as uo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROJ = dict(ymax=0.0, xres=250.0, yres=250.0, lonlat=False)
GEO = dict(ymax=13.5, xres=0.5, yres=0.5, lonlat=True)


def jacobi_fill(z, rows):
    """W(c) = max(Z(c), min_n W(n) + eps(c->n)) iterated from +inf on the non-boundary valid cells until nothing moves."""
    nr, nc = z.shape
    valid = ~np.isnan(z)
    bnd = uo.boundary_mask(z)
    upd = valid & ~bnd
    w = np.where(upd, np.inf, z)
    rr = np.arange(nr)[:, None]
    for _ in range(nr * nc + 1):
        pad = np.full((nr + 2, nc + 2), np.nan)
        pad[1:-1, 1:-1] = w
        m = np.full(z.shape, np.inf)
        for k, (dr, dc) in enumerate(uo.D8):
            v = pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc] + rows[rr, 6 + uo.d8_dist_col(k)]
            m = np.where(v < m, v, m)
        new = np.where(upd, np.where(m > z, m, z), w)
        if np.array_equal(new, w, equal_nan=True):
            return w
        w = new
    raise AssertionError("no fixpoint")


def dem_rounded(nr=23, nc=29, seed=1):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:nr, 0:nc]
    z = np.round(100 + 20 * np.sin(x / 5.0) * np.cos(y / 4.0) + 3 * rng.standard_normal((nr, nc)))
    z[8:12, 10:16] = 95.0          # a flat
    return z


def dem_pit():
    z = np.add.outer(np.arange(15.0), np.arange(17.0)) * 2.0 + 50.0
    z[7, 8] = 10.0                 # one deep pit
    return z


def dem_basin():
    y, x = np.mgrid[0:21, 0:21]
    z = np.full((21, 21), 200.0)   # a rim round a bowl whose bottom is 100 m ...
    z[3:18, 3:18] = 100.0 + np.hypot(y[3:18, 3:18] - 10, x[3:18, 3:18] - 10)
    z[10, 0:3] = 90.0              # ... that spills through one notch in the rim
    return z


def dem_holes():
    z = dem_rounded(19, 24, seed=4)
    rng = np.random.default_rng(9)
    z[rng.random(z.shape) < 0.08] = np.nan
    z[5:9, 6:10] = np.nan
    return z


CASES = {"rounded": dem_rounded, "pit": dem_pit, "basin": dem_basin, "holes": dem_holes}


def check_fill(z, w, rows):
    valid = ~np.isnan(z)
    assert np.array_equal(np.isnan(w), ~valid)
    assert (w[valid] >= z[valid]).all()
    bnd = uo.boundary_mask(z)
    assert np.array_equal(w[bnd], z[bnd])
    nr, nc = z.shape
    pad = np.full((nr + 2, nc + 2), np.nan)
    pad[1:-1, 1:-1] = w
    m = np.full(z.shape, np.inf)
    rr = np.arange(nr)[:, None]
    for k, (dr, dc) in enumerate(uo.D8):
        v = pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc] + rows[rr, 6 + uo.d8_dist_col(k)]
        m = np.where(v < m, v, m)
    inner = valid & ~bnd
    assert (w[inner] >= m[inner]).all()        # some neighbour n with W(c) >= W(n) + eps(c->n)


def sink_mask(w):
    nr, nc = w.shape
    pad = np.full((nr + 2, nc + 2), np.nan)
    pad[1:-1, 1:-1] = w
    lower = np.zeros(w.shape, dtype=bool)
    for dr, dc in uo.D8:
        lower |= pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc] < w
    return ~np.isnan(w) & ~lower


@pytest.mark.parametrize("geo", [False, True], ids=["projected", "lonlat"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_priority_flood_equals_the_jacobi_fixpoint(case, geo):
    z = CASES[case]()
    kw = GEO if geo else PROJ
    rows = uo.upslope_rows(z.shape[0], kw["ymax"], kw["xres"], kw["yres"], kw["lonlat"], 0.1)
    w = uo.fill_priority_flood(z, rows)
    assert np.array_equal(w, jacobi_fill(z, rows), equal_nan=True)
    check_fill(z, w, rows)
    if case == "pit":
        assert w[7, 8] > z[7, 8]
    if case == "basin":
        assert w[10, 10] > z[10, 4] and w[10, 0] == 90.0 and w[10, 1] > 90.0   # filled over the bowl's lip, graded notch


@pytest.mark.parametrize("geo", [False, True], ids=["projected", "lonlat"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_accumulation_conserves_area(case, geo):
    z = CASES[case]()
    kw = GEO if geo else PROJ
    res = uo.upslope_area(z, min_slope_deg=0.1, **kw)
    rows = uo.upslope_rows(z.shape[0], kw["ymax"], kw["xres"], kw["yres"], kw["lonlat"], 0.1)
    valid = ~np.isnan(z)
    a = res["area"]
    assert np.array_equal(np.isnan(a), ~valid)
    cell = np.broadcast_to(rows[:, 3:4], z.shape)
    assert (a[valid] >= cell[valid]).all()
    total = cell[valid].sum()
    out = a[sink_mask(res["filled"])].sum()
    assert abs(out - total) <= 1e-12 * total


def test_eastward_ramp_accumulates_whole_cells():
    n = 40
    z = (n - np.arange(n, dtype=np.float64))[None, :]       # falls to the east
    res = uo.upslope_area(z, ymax=0.0, xres=100.0, yres=100.0, lonlat=False)
    assert np.array_equal(res["filled"], z)
    assert np.array_equal(res["area"][0], (np.arange(n) + 1) * 100.0 * 100.0)


def test_cone_is_symmetric():
    n = 31
    y, x = np.mgrid[0:n, 0:n]
    z = 500.0 - np.hypot(y - 15, x - 15) * 10.0
    a = uo.upslope_area(z, ymax=0.0, xres=30.0, yres=30.0, lonlat=False)["area"]
    for b in (a[::-1], a[:, ::-1], a.T, a[::-1, ::-1].T):
        assert np.allclose(a, b, rtol=1e-12, atol=0)
    assert a[15, 15] == 900.0 and a[0, 0] > 900.0


def test_upslope_structs_match_the_header():
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write('#include <stdio.h>\n#include <stddef.h>\n#include "splash_cuda.h"\nint main(){printf("%zu %zu %zu %zu %d\\n",'
                             "sizeof(splash_upslope_in),sizeof(splash_upslope_out),offsetof(splash_upslope_in,min_slope_deg),"
                             "offsetof(splash_upslope_out,accum_rounds),SPLASH_ABI_VERSION);return 0;}\n")
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = list(map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()))
    assert got == [C.sizeof(_abi.SplashUpslopeIn), C.sizeof(_abi.SplashUpslopeOut), _abi.SplashUpslopeIn.min_slope_deg.offset,
                   _abi.SplashUpslopeOut.accum_rounds.offset, _abi.SPLASH_ABI_VERSION]


def test_upslope_kernels_compile_for_sm100a_without_spills():
    """ptxas's resource report of the library, built into a temporary file: the four kernels exist and spill nothing."""
    with tempfile.TemporaryDirectory() as d:
        lib = os.path.join(d, "libsplash_cuda.so")
        r = subprocess.run([build.nvcc_path(), *build.NVCC_FLAGS, "-o", lib, *build.SOURCES], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
    report = r.stderr
    for k in ("k_fill_init", "k_fill_sweep", "k_flow_prep", "k_accum"):
        m = re.search(r"Compiling entry function '(_ZN7upslope\d+%s\w*)' for 'sm_100a'\n.*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads" % k, report)
        assert m, k
        assert m.group(2) == m.group(3) == m.group(4) == "0", (k, m.group(0))
