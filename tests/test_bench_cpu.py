"""CPU suite: the reference arm of bench.py (the one part of the bench that runs without a GPU) keeps the JSON
contract, and the CUDA arm refuses to run without a device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT)


def test_reference_arm_line():
    r = run("--impl", "reference", "--cpu-sample", "48", "--years", "1", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "splash.grid cell-days/sec" and line["unit"] == "cell-days/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["dtype"] == "f64" and line["data"] == "synthetic"
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and "48 cells" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "cell-days/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["gpu_launches"] == 0


def test_dump_sample_is_fixed_and_fits_the_cap():
    """--dump-outputs writes the same cells on every run, only cells the checker calls finite, as many as fit in
    DUMP_BYTES (f64 + the eleven .npy headers); it asks the checker about each cell at most once."""
    import numpy as np
    import pytest

    import bench
    from rsplash_b200 import _abi, synthetic

    per_cell = 9 * 120 + _abi.SPLASH_NDIAG + 1  # the 10-year workload's monthly layers, cell_diag and the cell index
    finite = np.ones(synthetic.N_CELLS_5ARCMIN, dtype=bool)
    finite[::173] = False
    asked = []

    def finite_of(sub):
        assert (np.diff(sub) > 0).all()
        asked.extend(sub.tolist())
        return finite[sub]

    a = bench.dump_sample(len(finite), per_cell, finite_of)
    assert len(asked) == len(set(asked)) and len(asked) < 1.05 * len(a) + 200
    assert np.array_equal(a, bench.dump_sample(len(finite), per_cell, lambda s: finite[s])) and (np.diff(a) > 0).all()
    assert finite[a].all() and len(a) * per_cell * 8 + 11 * 128 <= bench.DUMP_BYTES
    assert len(a) == (bench.DUMP_BYTES - 64 * 1024) // (8 * per_cell)
    assert np.array_equal(bench.dump_sample(1000, per_cell, lambda s: finite[s]), np.flatnonzero(finite[:1000]))
    with pytest.raises(SystemExit):
        bench.parse_args(["--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args(["--impl", "reference", "--dump-outputs", "x"])


def test_cuda_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        return  # (this test is about the GPU-less container)
    r = run("--steps", "1", "--warmup", "0", "--cells", "1024", "--years", "1")
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
