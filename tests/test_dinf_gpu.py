"""GPU: splash_upslope_dinf_run (fill to flat, flat resolution, D-infinity accumulation) against the numpy restatement
(tests/dinf_oracle.py: priority flood, queue-based flat labelling and searches, a CPU Kahn queue; different algorithms
from the kernels' sweeps and frontier rounds).  The library returns no flat mask, M or receiver codes, so those are
held through the angle, which names the winning facet and its clip: equal bits on every cell with one receiver
(clipped, or a flat cell's steepest descent), a few ulp where atan(s2 / s1) enters; the area within 1e-12 relative
(the device's atan is the only operation that differs).  Also: repeatability over calls, memory kinds and multi-GPU
contexts; argument checks; edge shapes; invariants on a 4000 x 4000 DEM; the result fed to splash_grid."""
import numpy as np
import pytest

from oracle import terrain_oracle as to
from rsplash_b200 import _abi, api
from rsplash_b200._lib import Context, SplashError
from tests import dinf_oracle as do
from tests import upslope_oracle as uo
from tests.synthetic import make_problem
from tests.upslope_cases import fractal_dem

pytestmark = pytest.mark.gpu

GEO = dict(ymax=13.5, xres=0.5, yres=0.5, lonlat=True)
GEO5 = dict(ymax=13.5, xres=1 / 12, yres=1 / 12, lonlat=True)
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


def assert_matches_oracle(ctx, z, kw):
    got = api.upslope_areav2(z, ctx=ctx, return_filled=True, return_angle=True, **kw)
    ref = do.upslope_areav2(z, **kw)
    assert np.array_equal(got["filled"], ref["filled"], equal_nan=True)
    ga, ra = got["angle"], ref["angle"]
    assert np.array_equal(np.isnan(ga), np.isnan(ra))
    one = (ref["card"] >= 0) != (ref["diag"] >= 0)
    two = (ref["card"] >= 0) & (ref["diag"] >= 0)
    assert np.array_equal(ga[one], ra[one])
    assert (np.abs(ga[two] - ra[two]) <= 4 * np.spacing(ra[two])).all()
    valid = ~np.isnan(z)
    assert np.array_equal(np.isnan(got["area"]), ~valid)
    assert np.abs(got["area"][valid] - ref["area"][valid]).max() <= 1e-12 * np.abs(ref["area"][valid]).max()
    assert (np.abs(got["area"][valid] - ref["area"][valid]) <= 1e-12 * ref["area"][valid]).all()
    return got, ref


@pytest.mark.parametrize("kw", [GEO, PROJ], ids=["lonlat", "projected"])
def test_matches_the_oracle_on_the_terrain_dem(ctx, kw):
    z = terrain_dem()
    got, ref = assert_matches_oracle(ctx, z, kw)
    assert ref["flat"].sum() > 40                                   # the lake, filled pits and integer ties
    fd = to.terrain(z, **kw)["flowdir"]
    assert np.array_equal(got["ncellin"], to.ncellflow(fd, "in"), equal_nan=True)
    assert np.array_equal(got["ncellout"], to.ncellflow(fd, "out"), equal_nan=True)
    assert got["Au"].shape == (3,) + z.shape and np.shares_memory(got["Au"], got["area"])
    assert got["fill_sweeps"] >= 1 and got["flat_rounds"] >= 1 and got["accum_rounds"] >= 1


@pytest.mark.parametrize("kw", [GEO5, PROJ], ids=["lonlat", "projected"])
def test_matches_the_oracle_on_a_fractal_dem_with_sea(ctx, dem300, kw):
    got, ref = assert_matches_oracle(ctx, dem300, kw)
    assert np.isnan(got["area"][np.isnan(dem300)]).all()
    assert ref["flat"].any()


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (37, 1), (0, 5), (9, 12), (5, 6)],
                         ids=["1x1", "1xN", "Nx1", "0xN", "allNaN", "one_valid"])
def test_edge_shapes(ctx, shape):
    if shape == (9, 12):
        z = np.full(shape, np.nan)
    elif shape == (5, 6):
        z = np.full(shape, np.nan)
        z[2, 3] = 7.0
    else:
        z = np.arange(np.prod(shape), dtype=np.float64)[::-1].reshape(shape) % 7.0
    got = api.upslope_areav2(z, ctx=ctx, return_filled=True, return_angle=True, **PROJ)
    assert got["area"].shape == shape
    if z.size:
        ref = do.upslope_areav2(z, **PROJ)
        assert np.array_equal(got["filled"], ref["filled"], equal_nan=True)
        assert np.array_equal(got["area"], ref["area"], equal_nan=True)   # no interior cell: nothing through atan
        assert np.isnan(got["angle"]).all()                                # every valid cell is a boundary cell
    if shape == (1, 1):
        assert got["area"][0, 0] == 250.0 * 250.0 and got["accum_rounds"] == 1
    if shape == (9, 12):
        assert np.isnan(got["area"]).all() and got["accum_rounds"] == 0
    if shape == (5, 6):
        assert got["area"][2, 3] == 250.0 * 250.0 and np.isnan(got["area"]).sum() == z.size - 1


def test_repeatable_over_calls_memory_kinds_and_contexts(ctx, dem300):
    import torch

    keys = ("Au", "filled", "angle", "fill_sweeps", "flat_rounds", "accum_rounds")
    a = api.upslope_areav2(dem300, ctx=ctx, return_filled=True, return_angle=True, **GEO5)
    b = api.upslope_areav2(dem300, ctx=ctx, return_filled=True, return_angle=True, **GEO5)
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    dev = torch.device("cuda", 0)
    zt = torch.from_numpy(dem300).to(dev)
    au = torch.full((3,) + dem300.shape, -1.0, dtype=torch.float64, device=dev)
    wt = torch.empty(dem300.shape, dtype=torch.float64, device=dev)
    at = torch.empty(dem300.shape, dtype=torch.float64, device=dev)
    d = api.upslope_areav2(None, ctx=ctx, in_ptr=zt.data_ptr(), out_ptr=au.data_ptr(), filled_ptr=wt.data_ptr(),
                           angle_ptr=at.data_ptr(), shape=dem300.shape, **GEO5)
    assert np.array_equal(au.cpu().numpy(), a["Au"], equal_nan=True)
    assert np.array_equal(wt.cpu().numpy(), a["filled"], equal_nan=True)
    assert np.array_equal(at.cpu().numpy(), a["angle"], equal_nan=True)
    assert all(d[k] == a[k] for k in ("fill_sweeps", "flat_rounds", "accum_rounds"))
    devs = list(range(min(2, torch.cuda.device_count())))
    with Context(devs) as mctx:
        m = api.upslope_areav2(dem300, ctx=mctx, return_filled=True, return_angle=True, **GEO5)
    for k in keys:
        assert np.array_equal(m[k], a[k], equal_nan=True), k


def test_arguments_are_checked(ctx):
    for bad in (np.inf, -np.inf):
        z = np.ones((4, 4))
        z[2, 2] = bad
        with pytest.raises(SplashError) as e:
            api.upslope_areav2(z, ctx=ctx, **PROJ)
        assert e.value.code == _abi.SPLASH_ERR_BAD_ARG and "inf" in str(e.value)
    for xres, yres in ((0.0, 1.0), (1.0, -1.0), (np.nan, 1.0), (1.0, np.inf)):
        with pytest.raises(SplashError) as e:
            api.upslope_areav2(np.ones((4, 4)), ctx=ctx, ymax=0.0, xres=xres, yres=yres, lonlat=False)
        assert e.value.code == _abi.SPLASH_ERR_BAD_ARG
    with pytest.raises(SplashError) as e:
        api.upslope_areav2(None, ctx=ctx, in_ptr=0, out_ptr=0, shape=(-1, 4), **PROJ)
    assert e.value.code == _abi.SPLASH_ERR_BAD_ARG
    with pytest.raises(SplashError) as e:
        api.upslope_areav2(None, ctx=ctx, in_ptr=0, out_ptr=0, shape=(70000, 70000), **PROJ)   # past int32 cells
    assert e.value.code == _abi.SPLASH_ERR_BAD_ARG
    with pytest.raises(SplashError) as e:
        api.upslope_areav2(np.ones((4, 4)), ctx=ctx, ymax=-88.0, xres=1.0, yres=1.0, lonlat=True)   # past the pole
    assert e.value.code == _abi.SPLASH_ERR_BAD_ARG


def test_invariants_on_a_4000_square_dem(ctx):
    z = fractal_dem(4000, 4000, seed=5)
    kw = dict(ymax=60.0, xres=1 / 120, yres=1 / 120, lonlat=True)
    got = api.upslope_areav2(z, ctx=ctx, return_filled=True, return_angle=True, **kw)
    w, a, ang = got["filled"], got["area"], got["angle"]
    valid = ~np.isnan(z)
    inner = valid & ~uo.boundary_mask(z)
    assert np.array_equal(np.isnan(w), ~valid) and np.array_equal(np.isnan(a), ~valid)
    assert (w[valid] >= z[valid]).all()
    assert np.array_equal(np.isnan(ang), ~inner)                   # every valid non-boundary cell has a direction
    assert ((ang[inner] >= 0) & (ang[inner] < 2 * np.pi)).all()
    rows = do.dinf_rows(z.shape[0], kw["ymax"], kw["xres"], kw["yres"], True)
    cell = np.broadcast_to(rows[:, 3:4], z.shape)
    assert (a[valid] >= cell[valid] * (1 - 1e-12)).all()
    total = cell[valid].sum()
    assert abs(a[valid & ~inner].sum() - total) <= 1e-12 * total   # what leaves the grid is all of it
    assert got["accum_rounds"] > 100 and got["fill_sweeps"] > 1 and got["flat_rounds"] > 1


def test_end_to_end_into_splash_grid(ctx):
    z = fractal_dem(12, 16, seed=2, sea=0.0)
    kw = dict(ymax=-20.0, xres=0.25, yres=0.25, lonlat=True)
    got = api.upslope_areav2(z, ctx=ctx, **kw)
    ref = do.upslope_areav2(z, **kw)
    fd = to.terrain(z, **kw)["flowdir"]
    au_ref = np.stack([ref["area"], to.ncellflow(fd, "in"), to.ncellflow(fd, "out")])
    assert np.allclose(got["Au"], au_ref, rtol=1e-12, atol=0)
    n = z.size
    prob, dates = make_problem(n_cells=n, n_years=1, seed=8)
    run = lambda au: api.splash_grid(prob.sw_in, prob.tc, prob.pn, prob.lat, prob.elev, prob.slop, prob.asp, prob.soil,
                                     au.reshape(3, n), prob.resolution, dates, monthly_out=False, ctx=ctx)
    a, b = run(got["Au"]), run(au_ref)
    for k in _abi.OUTPUT_NAMES:
        assert np.allclose(a[k], b[k], rtol=1e-9, atol=1e-12, equal_nan=True), k
    assert np.isfinite(a["bflow"]).any()
