"""GPU: bench.py --dump-outputs writes what the value leg's last timed step computed, for the cells it names."""
import os
import subprocess
import sys

import numpy as np
import pytest

from rsplash_b200 import _abi, api, synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_equal_a_direct_call_on_the_same_cells(ctx, tmp_path):
    import bench

    n_cells, years = 3000, 1
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cells", str(n_cells), "--years", str(years), "--steps", "2",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    names = _abi.OUTPUT_NAMES + ("cell_diag", "cell_index")
    assert sorted(os.listdir(d)) == sorted(f"{k}.npy" for k in names)
    assert sum(os.path.getsize(d / f"{k}.npy") for k in names) <= bench.DUMP_BYTES
    got = {k: np.load(d / f"{k}.npy") for k in names}
    cells = got["cell_index"].astype(np.int64)
    # every cell fits: all of them are written but the few whose checker result is not finite
    assert np.array_equal(cells, got["cell_index"]) and (np.diff(cells) > 0).all() and 0.98 * n_cells <= len(cells) < n_cells + 1
    # the resident f32 path of the bench equals the host f64 path, and cells are independent: the same bits
    prob = bench.host_problem(synthetic.Grid(n_cells, bench.GRID_SEED), cells, years)
    want = api.splash_grid(prob.sw_in, prob.tc, prob.pn, prob.lat, prob.elev, prob.slop, prob.asp, prob.soil, prob.au,
                           prob.resolution, synthetic.daily_dates(bench.FIRST_YEAR, years), monthly_out=True, ctx=ctx,
                           return_diag=True)
    for k in _abi.OUTPUT_NAMES + ("cell_diag",):
        assert got[k].dtype == np.float64 and np.isfinite(got[k]).all(), k
        assert np.array_equal(got[k], want[k]), k
