"""Measurement of splash_upslope_area_run: fill and accumulation kernel time, sweeps and rounds, host-fed wall time.

usage: python tools/upslope_bench.py [--sizes 2160x4320,10800x10800] [--reps 3] [--seed 7]

DEMs: tests/upslope_cases.fractal_dem (spectral fractal + large-scale tilt, lowest 20 % NaN sea) from a seed.  The
2160 x 4320 grid is the 5-arc-minute global grid of bench.py (lon/lat, 90 N to 90 S); 10800 x 10800 is a projected
grid of 90 m cells.  Kernel times: CUDA events around calls on device pointers (after a warm-up call), and per-kernel
sums from torch.profiler in one separate profiled call; the arrays (>= 5 x 8 B per cell) exceed the 126 MB L2 at both
sizes.  Prints the GPU's name and power limit (read-only nvidia-smi query) and one JSON line per size.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rsplash_b200 import api  # noqa: E402
from rsplash_b200._lib import Context  # noqa: E402
from tests.upslope_cases import fractal_dem  # noqa: E402

FILL_KERNELS = ("k_fill_init", "k_fill_sweep")
ACCUM_KERNELS = ("k_flow_prep", "k_accum")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def grid_kw(nr, nc):
    if (nr, nc) == (2160, 4320):
        return dict(ymax=90.0, xres=1 / 12, yres=1 / 12, lonlat=True)
    return dict(ymax=0.0, xres=90.0, yres=90.0, lonlat=False)


def kernel_ms(prof):
    fill = accum = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if any(k in e.key for k in FILL_KERNELS):
            fill += t / 1e3
        elif any(k in e.key for k in ACCUM_KERNELS):
            accum += t / 1e3
    return fill, accum


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2160x4320,10800x10800")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("upslope_bench: no CUDA device (there is nothing to measure on the host)")
    print("gpu:", gpu_info(), flush=True)
    ctx = Context(0)
    dev = torch.device("cuda", 0)
    for size in a.sizes.split(","):
        nr, nc = (int(v) for v in size.split("x"))
        kw = grid_kw(nr, nc)
        t0 = time.perf_counter()
        z = fractal_dem(nr, nc, seed=a.seed)
        gen_s = time.perf_counter() - t0
        zt = torch.from_numpy(z).to(dev)
        au = torch.empty((3, nr, nc), dtype=torch.float64, device=dev)
        run = lambda: api.upslope_area(None, ctx=ctx, in_ptr=zt.data_ptr(), out_ptr=au.data_ptr(), shape=(nr, nc), **kw)
        counters = run()  # warm-up (module load, first allocations)
        ts = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            c = run()  # synchronous; the library works on its own stream, so bracket with device-wide syncs
            torch.cuda.synchronize()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
            assert c == counters, (c, counters)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            run()
            torch.cuda.synchronize()
        fill_ms, accum_ms = kernel_ms(prof)
        t0 = time.perf_counter()
        host = api.upslope_area(z, ctx=ctx, **kw)
        host_s = time.perf_counter() - t0
        assert np.array_equal(host["Au"], au.cpu().numpy(), equal_nan=True)
        n_valid = int(np.count_nonzero(~np.isnan(z)))
        print(json.dumps({
            "size": [nr, nc], "grid": kw, "seed": a.seed, "valid_cells": n_valid, "dem_gen_s": round(gen_s, 2),
            "fill_sweeps": counters["fill_sweeps"], "accum_rounds": counters["accum_rounds"],
            "device_call_ms": {"median": float(np.median(ts)), "min": float(np.min(ts)), "max": float(np.max(ts)), "reps": a.reps},
            "fill_kernel_ms": fill_ms, "accum_kernel_ms": accum_ms,
            "fill_cells_per_s": nr * nc / (fill_ms / 1e3) if fill_ms else None,
            "accum_cells_per_s": n_valid / (accum_ms / 1e3) if accum_ms else None,
            "host_fed_wall_s": host_s,
        }), flush=True)
        del zt, au
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
