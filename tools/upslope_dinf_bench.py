"""Measurement of splash_upslope_dinf_run next to splash_upslope_area_run on the same DEMs: time per device-pointer
call of each, and the D-infinity kernel time split into fill, flats, directions and accumulation, with sweep and
round counts.

usage: python tools/upslope_dinf_bench.py [--sizes 2160x4320,10800x10800] [--reps 3] [--seed 7]

DEMs and grids as tools/upslope_bench.py (fractal surface with 20 % NaN sea; 5' lon/lat global grid, 90 m projected
grid).  Call times: CUDA events around device-pointer calls after a warm-up call of each method, the two methods
alternating; kernel splits: torch.profiler over one separate call of each.  Prints the GPU's name, power limit and
maximum SM clock (read-only nvidia-smi query) and one JSON line per size.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rsplash_b200 import api  # noqa: E402
from rsplash_b200._lib import Context  # noqa: E402
from tests.upslope_cases import fractal_dem  # noqa: E402
from tools.upslope_bench import gpu_info, grid_kw  # noqa: E402

# kernel-name substrings of each stage, matched in this order (k_accum is one template for three stages)
STAGES = (
    ("fill", ("k_fill_init", "k_fill_sweep")),
    ("flats", ("FlatBfs", "k_flat_")),
    ("directions", ("k_dinf_dir",)),
    ("accum", ("DinfRule", "MfdRule", "k_flow_prep", "k_dinf_prep")),
)


def stage_ms(prof):
    out = {name: 0.0 for name, _ in STAGES}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        for name, keys in STAGES:
            if any(k in e.key for k in keys):
                out[name] += t / 1e3
                break
    return out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    c = fn()  # synchronous; the library works on its own stream, so bracket with device-wide syncs
    torch.cuda.synchronize()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2160x4320,10800x10800")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("upslope_dinf_bench: no CUDA device (there is nothing to measure on the host)")
    print("gpu:", gpu_info(), flush=True)
    ctx = Context(0)
    dev = torch.device("cuda", 0)
    for size in a.sizes.split(","):
        nr, nc = (int(v) for v in size.split("x"))
        kw = grid_kw(nr, nc)
        z = fractal_dem(nr, nc, seed=a.seed)
        zt = torch.from_numpy(z).to(dev)
        au = torch.empty((3, nr, nc), dtype=torch.float64, device=dev)
        runs = {
            "mfd": lambda: api.upslope_area(None, ctx=ctx, in_ptr=zt.data_ptr(), out_ptr=au.data_ptr(), shape=(nr, nc), **kw),
            "dinf": lambda: api.upslope_areav2(None, ctx=ctx, in_ptr=zt.data_ptr(), out_ptr=au.data_ptr(), shape=(nr, nc), **kw),
        }
        counters = {k: f() for k, f in runs.items()}  # warm-up
        ts = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, f in runs.items():
                t, c = timed(f)
                assert c == counters[k], (k, c, counters[k])
                ts[k].append(t)
        stages = {}
        for k, f in runs.items():
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                f()
                torch.cuda.synchronize()
            stages[k] = stage_ms(prof)
        host = api.upslope_areav2(z, ctx=ctx, **kw)
        runs["dinf"]()
        assert np.array_equal(host["Au"], au.cpu().numpy(), equal_nan=True)
        line = {"size": [nr, nc], "grid": kw, "seed": a.seed, "valid_cells": int(np.count_nonzero(~np.isnan(z)))}
        for k in runs:
            line[k] = {
                "call_ms": {"median": float(np.median(ts[k])), "min": float(np.min(ts[k])), "max": float(np.max(ts[k])), "reps": a.reps},
                "kernel_ms": {s: round(v, 3) for s, v in stages[k].items() if v or k == "dinf"},
                **counters[k],
            }
        print(json.dumps(line), flush=True)
        del zt, au
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
