"""CPU: the numpy restatement of the D-infinity contributing area (tests/dinf_oracle.py; PARITY UNPINNED, see
include/splash_cuda.h, splash_upslope_dinf_run) on hand-built surfaces with known answers: a tilted plane, a
paraboloid, a closed basin with a notch, a flat floor between walls; area conservation; the C structs against their
ctypes mirror; the new kernels compile for sm_100a without spills."""
import ctypes as C
import math
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from rsplash_b200 import _abi, build
from tests import dinf_oracle as do
from tests import upslope_oracle as uo
from tests.upslope_cases import fractal_dem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROJ = dict(ymax=0.0, xres=30.0, yres=30.0, lonlat=False)
GEO = dict(ymax=13.5, xres=0.5, yres=0.5, lonlat=True)


def inner_mask(z):
    return ~np.isnan(z) & ~uo.boundary_mask(z)


def jacobi_fill_flat(z):
    """W(c) = max(Z(c), min_n W(n)) iterated from +inf on the non-boundary valid cells until nothing moves."""
    nr, nc = z.shape
    upd = inner_mask(z)
    w = np.where(upd, np.inf, z)
    for _ in range(nr * nc + 1):
        m = np.full(z.shape, np.inf)
        for k in range(8):
            v = do._shift(w, k, np.nan)
            m = np.where(v < m, v, m)
        new = np.where(upd, np.where(m > z, m, z), w)
        if np.array_equal(new, w, equal_nan=True):
            return w
        w = new
    raise AssertionError("no fixpoint")


@pytest.mark.parametrize("phi", [0.3, 1.2, 2.0, 2.9, 3.5, 4.4, 5.0, 5.9])
def test_tilted_plane_flows_at_its_azimuth(phi):
    nr, nc, h = 17, 19, 30.0
    y, x = np.mgrid[0:nr, 0:nc]
    z = -(x * h * math.cos(phi) - y * h * math.sin(phi))   # falls towards azimuth phi (north row first)
    res = do.upslope_areav2(z, **PROJ)
    inner = inner_mask(z)
    assert np.array_equal(np.isnan(res["angle"]), ~inner)
    assert np.abs(res["angle"][inner] - phi).max() <= 1e-14
    assert not res["flat"].any()


@pytest.mark.parametrize("phi,axis", [(0.0, 1), (math.pi / 2, 0)], ids=["east", "north"])
def test_cardinal_tilt_accumulates_whole_cells(phi, axis):
    nr, nc, h = 13, 16, 30.0
    y, x = np.mgrid[0:nr, 0:nc]
    z = 500.0 - (x * round(math.cos(phi)) - y * round(math.sin(phi))) * 2.0
    res = do.upslope_areav2(z, **PROJ)
    inner = inner_mask(z)
    assert (res["angle"][inner] == phi).all()
    cell = h * h
    a = res["area"] if axis == 1 else res["area"][::-1].T       # flow along +column
    for r in range(1, a.shape[0] - 1):                          # the edge rows / columns are boundary cells
        assert np.array_equal(a[r], np.r_[1, np.arange(1, a.shape[1])] * cell)
    assert (a[[0, -1]] == cell).all()


def test_paraboloid_has_the_grids_8_fold_symmetry():
    n = 32                                                       # apex between the four middle cells
    y, x = np.mgrid[0:n, 0:n]
    z = 5000.0 - 2.0 * ((y - 15.5) ** 2 + (x - 15.5) ** 2)       # exact in binary: quarters
    a = do.upslope_areav2(z, **PROJ)["area"]
    for b in (a[::-1], a[:, ::-1], a.T, a[::-1, ::-1].T):
        assert np.allclose(a, b, rtol=1e-12, atol=0)
    assert a[15, 15] == 900.0 and a[0, 0] > 900.0


def test_closed_basin_drains_through_its_notch():
    n = 21
    y, x = np.mgrid[0:n, 0:n]
    z = np.full((n, n), 200.0)                                   # a one-cell rim round a bowl ...
    z[1:-1, 1:-1] = 100.0 + np.hypot(y[1:-1, 1:-1] - 10, x[1:-1, 1:-1] - 10)
    z[10, 0] = 90.0                                              # ... with one notch
    res = do.upslope_areav2(z, **PROJ)
    w = res["filled"]
    assert np.array_equal(w, jacobi_fill_flat(z))
    assert w[10, 10] == 109.0 and w[10, 1] == 109.0               # filled to the notch's sill, flat
    assert res["flat"][2:-2, 2:-2].any()
    inner = inner_mask(z)
    assert np.isfinite(res["angle"][inner]).all()
    cell = 900.0
    edge = ~inner
    a = res["area"]
    assert a[10, 0] == pytest.approx((1 + (n - 2) ** 2) * cell, rel=1e-12)
    others = edge.copy()
    others[10, 0] = False
    assert (a[others] == cell).all()                             # nothing leaves anywhere else


def test_flat_floor_between_walls_converges_away_from_them():
    nr, nc = 9, 14
    z = np.full((nr, nc), 20.0)
    z[2:7, 1:] = 10.0                                            # floor rows 2..6, open at the east edge
    res = do.upslope_areav2(z, **PROJ)
    flat = res["flat"]
    expect_flat = np.zeros(z.shape, dtype=bool)
    expect_flat[2:7, 1:13] = True
    assert np.array_equal(flat, expect_flat)
    r, c = np.mgrid[0:nr, 0:nc]
    towards = 13 - c
    away = 1 + np.minimum(np.minimum(r - 2, 6 - r), c - 1)
    m = np.where(expect_flat, 2 * towards + 3 - away, 0)
    assert np.array_equal(res["mask"], m)
    ang = res["angle"]
    assert np.isfinite(ang[flat]).all()
    cols = slice(3, 12)
    assert (np.sin(ang[2, cols]) < 0).all() and (np.sin(ang[6, cols]) > 0).all()   # off the north / south walls
    assert (ang[4, cols] == 0.0).all()
    assert (np.cos(ang[flat]) > 0).all()                         # and on towards the outlet
    cell = 900.0
    valid_area = z.size * cell
    out = res["area"][np.isnan(ang)].sum()
    assert abs(out - valid_area) <= 1e-12 * valid_area


def dem_rounded(nr=23, nc=29, seed=1):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:nr, 0:nc]
    z = np.round(100 + 20 * np.sin(x / 5.0) * np.cos(y / 4.0) + 3 * rng.standard_normal((nr, nc)))
    z[8:12, 10:16] = 95.0
    return z


def dem_holes():
    z = dem_rounded(19, 24, seed=4)
    rng = np.random.default_rng(9)
    z[rng.random(z.shape) < 0.08] = np.nan
    z[5:9, 6:10] = np.nan
    return z


CASES = {"rounded": dem_rounded, "holes": dem_holes, "fractal": lambda: fractal_dem(40, 50, seed=3)}


@pytest.mark.parametrize("geo", [False, True], ids=["projected", "lonlat"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_fill_directions_and_conservation(case, geo):
    z = CASES[case]()
    kw = GEO if geo else PROJ
    res = do.upslope_areav2(z, **kw)
    assert np.array_equal(res["filled"], jacobi_fill_flat(z), equal_nan=True)
    valid = ~np.isnan(z)
    inner = inner_mask(z)
    ang, a = res["angle"], res["area"]
    assert np.array_equal(np.isnan(ang), ~inner)                 # every valid non-boundary cell has a direction
    assert ((ang[inner] >= 0) & (ang[inner] < 2 * math.pi)).all()
    assert np.array_equal(np.isnan(a), ~valid)
    cell = np.broadcast_to(res["rows"][:, 3:4], z.shape)
    assert (a[valid] >= cell[valid]).all()
    total = cell[valid].sum()
    out = a[valid & ~inner].sum()
    assert abs(out - total) <= 1e-12 * total
    # a receiver is strictly lower in W, or at the same W and strictly lower in M
    w, m = res["filled"], res["mask"]
    for key in ("card", "diag"):
        k = res[key]
        for d in range(8):
            sel = k == d
            wn, mn = do._shift(w, d, np.nan)[sel], do._shift(m, d, 0)[sel]
            assert ((wn < w[sel]) | ((wn == w[sel]) & (mn < m[sel]))).all()


def test_dinf_structs_match_the_header():
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write('#include <stdio.h>\n#include <stddef.h>\n#include "splash_cuda.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %d\\n",'
                             "sizeof(splash_dinf_in),sizeof(splash_dinf_out),offsetof(splash_dinf_in,mem_kind),"
                             "offsetof(splash_dinf_out,angle),offsetof(splash_dinf_out,flat_rounds),"
                             "offsetof(splash_dinf_out,accum_rounds),SPLASH_ABI_VERSION);return 0;}\n")
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = list(map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()))
    assert got == [C.sizeof(_abi.SplashDinfIn), C.sizeof(_abi.SplashDinfOut), _abi.SplashDinfIn.mem_kind.offset,
                   _abi.SplashDinfOut.angle.offset, _abi.SplashDinfOut.flat_rounds.offset,
                   _abi.SplashDinfOut.accum_rounds.offset, _abi.SPLASH_ABI_VERSION]


DINF_KERNELS = ("k_flat_mark", "k_flat_label", "k_flat_seed", "k_flat_height", "k_flat_mask", "k_dinf_dir",
                "k_dinf_prep", "k_accumINS_7FlatBfs", "k_accumINS_8DinfRule", "k_accumINS_7MfdRule")


def test_dinf_kernels_compile_for_sm100a_without_spills():
    """ptxas's resource report of the library, built into a temporary file: every D-infinity kernel (and each
    instantiation of the shared frontier-round kernel) exists and spills nothing."""
    with tempfile.TemporaryDirectory() as d:
        lib = os.path.join(d, "libsplash_cuda.so")
        r = subprocess.run([build.nvcc_path(), *build.NVCC_FLAGS, "-o", lib, *build.SOURCES], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
    report = r.stderr
    for k in DINF_KERNELS:
        found = re.findall(r"Compiling entry function '(_ZN7upslope\d+%s\w*)' for 'sm_100a'\n.*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads" % k, report)
        assert found, k
        for m in found:
            assert m[1] == m[2] == m[3] == "0", (k, m)
