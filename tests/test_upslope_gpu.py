"""GPU: splash_upslope_area_run (depression fill + Quinn MFD accumulation) against the numpy restatement, bit for bit
(tests/upslope_oracle.py: priority flood and a descending-elevation sweep, different algorithms from the kernels'
Jacobi sweeps and level-synchronous rounds); repeatability over calls, memory kinds and multi-GPU contexts;
invariants on a 4000 x 4000 DEM; the result fed to splash_grid."""
import numpy as np
import pytest

from oracle import terrain_oracle as to
from rsplash_b200 import _abi, api
from rsplash_b200._lib import Context, SplashError
from tests import upslope_oracle as uo
from tests.synthetic import make_problem
from tests.upslope_cases import fractal_dem

pytestmark = pytest.mark.gpu

GEO = dict(ymax=13.5, xres=0.5, yres=0.5, lonlat=True)         # the terrain test's grid (139 rows: down to 56 S)
GEO5 = dict(ymax=13.5, xres=1 / 12, yres=1 / 12, lonlat=True)  # 5 arc-minutes
PROJ = dict(ymax=0.0, xres=250.0, yres=250.0, lonlat=False)


def terrain_dem(nr=139, nc=159, seed=3):
    """The terrain test's DEM: integer metres (flats, ties), 3 % NA cells and a flat lake."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:nr, 0:nc]
    z = np.round(800 + 300 * np.sin(x / 17.0) * np.cos(y / 11.0) + 40 * rng.standard_normal((nr, nc)))
    z[rng.random((nr, nc)) < 0.03] = np.nan
    z[10:14, 20:30] = 650.0
    return z


@pytest.fixture(scope="module")
def dem300():
    return fractal_dem(300, 300, seed=11)


def assert_matches_oracle(ctx, z, kw, min_slope_deg=0.1):
    got = api.upslope_area(z, ctx=ctx, return_filled=True, min_slope_deg=min_slope_deg, **kw)
    ref = uo.upslope_area(z, min_slope_deg=min_slope_deg, **kw)
    assert np.array_equal(got["filled"], ref["filled"], equal_nan=True)
    assert np.array_equal(got["area"], ref["area"], equal_nan=True)
    return got, ref


@pytest.mark.parametrize("kw", [GEO, PROJ], ids=["lonlat", "projected"])
def test_bit_identical_to_the_oracle_on_the_terrain_dem(ctx, kw):
    z = terrain_dem()
    got, _ = assert_matches_oracle(ctx, z, kw)
    fd = to.terrain(z, **kw)["flowdir"]
    assert np.array_equal(got["ncellin"], to.ncellflow(fd, "in"), equal_nan=True)
    assert np.array_equal(got["ncellout"], to.ncellflow(fd, "out"), equal_nan=True)
    assert got["Au"].shape == (3,) + z.shape and np.shares_memory(got["Au"], got["area"])
    assert got["fill_sweeps"] >= 1 and got["accum_rounds"] >= 1


def test_bit_identical_to_the_oracle_on_a_fractal_dem_with_sea(ctx, dem300):
    got, _ = assert_matches_oracle(ctx, dem300, GEO5)
    assert np.isnan(got["area"][np.isnan(dem300)]).all()
    got2, _ = assert_matches_oracle(ctx, dem300, PROJ, min_slope_deg=2.5)


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (37, 1), (0, 5), (9, 12)], ids=["1x1", "1xN", "Nx1", "0xN", "allNaN"])
def test_edge_shapes(ctx, shape):
    z = np.full(shape, np.nan) if shape == (9, 12) else np.arange(np.prod(shape), dtype=np.float64)[::-1].reshape(shape) % 7.0
    got = api.upslope_area(z, ctx=ctx, return_filled=True, **PROJ)
    assert got["area"].shape == shape
    if z.size:
        ref = uo.upslope_area(z, **PROJ)
        assert np.array_equal(got["filled"], ref["filled"], equal_nan=True)
        assert np.array_equal(got["area"], ref["area"], equal_nan=True)
    if shape == (1, 1):
        assert got["area"][0, 0] == 250.0 * 250.0 and got["accum_rounds"] == 1
    if shape == (9, 12):
        assert np.isnan(got["area"]).all() and got["accum_rounds"] == 0


def test_repeatable_over_calls_memory_kinds_and_contexts(ctx, dem300):
    import torch

    a = api.upslope_area(dem300, ctx=ctx, return_filled=True, **GEO5)
    b = api.upslope_area(dem300, ctx=ctx, return_filled=True, **GEO5)
    for k in ("Au", "filled", "fill_sweeps", "accum_rounds"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    dev = torch.device("cuda", 0)
    zt = torch.from_numpy(dem300).to(dev)
    au = torch.full((3,) + dem300.shape, -1.0, dtype=torch.float64, device=dev)
    wt = torch.empty(dem300.shape, dtype=torch.float64, device=dev)
    d = api.upslope_area(None, ctx=ctx, in_ptr=zt.data_ptr(), out_ptr=au.data_ptr(), filled_ptr=wt.data_ptr(),
                         shape=dem300.shape, **GEO5)
    assert np.array_equal(au.cpu().numpy(), a["Au"], equal_nan=True)
    assert np.array_equal(wt.cpu().numpy(), a["filled"], equal_nan=True)
    assert (d["fill_sweeps"], d["accum_rounds"]) == (a["fill_sweeps"], a["accum_rounds"])
    devs = list(range(min(2, torch.cuda.device_count())))
    with Context(devs) as mctx:
        m = api.upslope_area(dem300, ctx=mctx, return_filled=True, **GEO5)
    for k in ("Au", "filled", "fill_sweeps", "accum_rounds"):
        assert np.array_equal(m[k], a[k], equal_nan=True), k


def test_arguments_are_checked(ctx):
    z = np.ones((4, 4))
    for bad in (0.0, -1.0, 90.0, np.nan, np.inf):
        with pytest.raises(SplashError) as e:
            api.upslope_area(z, ctx=ctx, min_slope_deg=bad, **PROJ)
        assert e.value.code == _abi.SPLASH_ERR_BAD_ARG
    z[2, 2] = np.inf
    with pytest.raises(SplashError) as e:
        api.upslope_area(z, ctx=ctx, **PROJ)
    assert e.value.code == _abi.SPLASH_ERR_BAD_ARG and "inf" in str(e.value)
    with pytest.raises(SplashError):
        api.upslope_area(np.ones((4, 4)), ctx=ctx, ymax=0.0, xres=0.0, yres=1.0, lonlat=False)
    with pytest.raises(SplashError):
        api.upslope_area(np.ones((4, 4)), ctx=ctx, ymax=-88.0, xres=1.0, yres=1.0, lonlat=True)   # rows past the pole


def _shifted(a, dr, dc, fill):
    nr, nc = a.shape
    pad = np.full((nr + 2, nc + 2), fill, dtype=a.dtype)
    pad[1:-1, 1:-1] = a
    return pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc]


def longest_path(w):
    """Cells on the longest strictly descending path of the filled surface: Kahn levels, vectorised per level."""
    nr, nc = w.shape
    nb = [_shifted(w, dr, dc, np.nan) for dr, dc in uo.D8]
    ndon = sum((x > w).astype(np.int64) for x in nb).ravel()
    flat = w.ravel()
    front = np.flatnonzero(~np.isnan(flat) & (ndon == 0))
    levels = 0
    while front.size:
        levels += 1
        r, c = np.divmod(front, nc)
        rec = []
        for dr, dc in uo.D8:
            rr, cc = r + dr, c + dc
            ok = (rr >= 0) & (rr < nr) & (cc >= 0) & (cc < nc)
            n = rr[ok] * nc + cc[ok]
            rec.append(n[flat[n] < flat[front[ok]]])
        rec = np.concatenate(rec)
        np.subtract.at(ndon, rec, 1)
        u = np.unique(rec)
        front = u[ndon[u] == 0]
    return levels


def test_invariants_on_a_4000_square_dem(ctx):
    z = fractal_dem(4000, 4000, seed=5)
    kw = dict(ymax=60.0, xres=1 / 120, yres=1 / 120, lonlat=True)
    got = api.upslope_area(z, ctx=ctx, return_filled=True, **kw)
    w, a = got["filled"], got["area"]
    rows = uo.upslope_rows(z.shape[0], kw["ymax"], kw["xres"], kw["yres"], True, 0.1)
    valid = ~np.isnan(z)
    assert np.array_equal(np.isnan(w), ~valid) and np.array_equal(np.isnan(a), ~valid)
    assert (w[valid] >= z[valid]).all()
    bnd = uo.boundary_mask(z)
    assert np.array_equal(w[bnd], z[bnd])
    rr = np.arange(z.shape[0])[:, None]
    m = np.full(z.shape, np.inf)
    for k, (dr, dc) in enumerate(uo.D8):
        v = _shifted(w, dr, dc, np.nan) + rows[rr, 6 + uo.d8_dist_col(k)]
        m = np.where(v < m, v, m)
    inner = valid & ~bnd
    assert (w[inner] >= m[inner]).all()
    cell = np.broadcast_to(rows[:, 3:4], z.shape)
    assert (a[valid] >= cell[valid]).all()
    lower = np.zeros(z.shape, dtype=bool)
    for dr, dc in uo.D8:
        lower |= _shifted(w, dr, dc, np.nan) < w
    sinks = valid & ~lower
    total = cell[valid].sum()
    assert abs(a[sinks].sum() - total) <= 1e-12 * total
    assert got["accum_rounds"] == longest_path(w)
    assert got["accum_rounds"] > 100 and got["fill_sweeps"] > 1


def test_end_to_end_into_splash_grid(ctx):
    z = fractal_dem(12, 16, seed=2, sea=0.0)
    kw = dict(ymax=-20.0, xres=0.25, yres=0.25, lonlat=True)
    got = api.upslope_area(z, ctx=ctx, **kw)
    ref = uo.upslope_area(z, **kw)
    fd = to.terrain(z, **kw)["flowdir"]
    au_ref = np.stack([ref["area"], to.ncellflow(fd, "in"), to.ncellflow(fd, "out")])
    n = z.size
    prob, dates = make_problem(n_cells=n, n_years=1, seed=8)
    run = lambda au: api.splash_grid(prob.sw_in, prob.tc, prob.pn, prob.lat, prob.elev, prob.slop, prob.asp, prob.soil,
                                     au.reshape(3, n), prob.resolution, dates, monthly_out=False, ctx=ctx)
    a, b = run(got["Au"]), run(au_ref)
    for k in _abi.OUTPUT_NAMES:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert np.isfinite(a["bflow"]).any()
