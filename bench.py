#!/usr/bin/env python
"""bench.py -- splash.grid cell-days/s on B200 (BASELINE.json metric), one JSON line on rank 0.

Workload (BASELINE.json configs[3], the configuration the metric is quoted on):
    synthetic 5-arcmin global grid, 2 332 800 land cells x 10 years daily (3652 days) incl. spin-up,
    monthly outputs (splash.grid's default sim.control).  The grid is counter-based
    (rsplash_b200/synthetic.py: Grid; every value a function of seed, global cell, day, field), so every
    rank's shard, every row block and the CPU baseline's sample are subsets of the same grid.
Multi-GPU (cells are independent: no data-path collective, only the max-time / sum-job-size all-reduce):
    --scaling strong (default)  ONE grid; blocks of 8 grid rows are dealt round-robin to the ranks, as the
                                reference's scheduler deals row blocks to its workers
                                (R/splash.grid.R:264-268, 312-314).  `config.weak_value` reports, beside it,
                                the throughput with one whole grid per rank.
    --scaling weak              every rank integrates one whole grid (its own forcing realisation).
A step is one whole-job pass of the hot path over the rank's shard:
    value  inputs resident in HBM (forcing stored as f32 -- lossless, the rasters are FLT4S -- all
           arithmetic f64), outputs written to HBM; timed around splash_grid_run(DEVICE pointers)
    e2e    the same job through the C ABI with HOST buffers (pinned, f64 like R's REAL()): the shard is fed
           block of rows by block of rows as the reference's clFun scheduler does (R/splash.grid.R:264-268),
           host->device and device->host copies inside the timed region.  At most 3 timed passes (`e2e.steps`);
           each pinned block is staged once and run for all of them.
The numerator is the job size as the reference defines it: n_cells * n_days plus the spin-up cell-days its
algorithm requires (365 for the aridity pass + passes * 366 per cell); `config.executed_*` quote the
cell-days the GPU actually simulated (exact cycle skipping removes work).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--cells C] [--years Y] [--dump-outputs DIR]
N > 1 is launched by torchrun (one rank per GPU, NCCL); RANK/LOCAL_RANK/WORLD_SIZE come from the env.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from rsplash_b200 import _abi, synthetic  # noqa: E402

METRIC = "splash.grid cell-days/sec"
UNIT = "cell-days/s"
FIRST_YEAR = 2001
GRID_SEED = 20240
ROW_BLOCK = 8        # grid rows per scheduling block of the strong-scaling shards
E2E_MAX_STEPS = 3    # timed passes of the host-fed leg (each moves ~220 GB over PCIe at N = 1)
ROOFLINE_MAX_STEPS = 3
DUMP_BYTES = 64 * 10**6   # --dump-outputs: at most this much in all
DUMP_SEED = 20241


def fp64_work_per_cell_day():
    """FP64 instructions (DFMA/DMUL/DADD thread-instructions) and flops per cell-day of the daily kernel,
    counted by ncu on the shipped kernel (profiles/fp64_work.json, see profiles/README.md)."""
    p = os.path.join(ROOT, "profiles", "fp64_work.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["fp64_inst_per_cell_day"]), float(d["flops_per_cell_day"]), d.get("source", "profiles/fp64_work.json")
    return 0.0, 0.0, "no ncu count committed"


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--cells", type=int, default=synthetic.N_CELLS_5ARCMIN)
    ap.add_argument("--years", type=int, default=10)
    ap.add_argument("--e2e-blocks", type=int, default=0, help="row blocks per rank for the e2e leg (0 = auto)")
    ap.add_argument("--cpu-sample", type=int, default=4096, help="cells of the CPU baseline / parity sample")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling figure at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (the 9 monthly layers and cell_diag, f64) "
                         "as DIR/<name>.npy: the columns of a fixed, seeded sample of the cells whose result on the host "
                         "checker is finite (rank 0's cells at N > 1), and their grid indices as cell_index.npy; "
                         f"at most {DUMP_BYTES // 10**6} MB in all; not with --impl reference")
    args = ap.parse_args(argv)
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed: it has no meaning with --impl reference")
    return args


def plan_seconds(args, world: int) -> dict:
    """Rough wall-clock plan of one bench.py run (seconds), so that a CPU test can hold it under the driver's per-N limit.
    Rates measured in round 2 on the pool's B200 boxes (profiles/README.md): resident pass 2.6 s at N = 1, host-fed pass 4.5 s."""
    frac = (args.cells / synthetic.N_CELLS_5ARCMIN) * (args.years / 10.0)
    pass_s = max(0.9, 2.8 * frac / (world if args.scaling == "strong" else 1))   # chain-bound below ~0.9 s
    e2e_s = max(1.2, 5.0 * frac / (world if args.scaling == "strong" else 1))
    p = {"startup": 75.0, "generate": 6.0 * frac + 4.0,
         "value": (args.warmup + args.steps) * pass_s,
         "roofline": (2 + min(args.steps, ROOFLINE_MAX_STEPS)) * pass_s,
         "e2e": 0.0 if args.no_e2e else 70.0 * frac + (1 + min(args.steps, E2E_MAX_STEPS)) * e2e_s + 8.0 * frac,
         "weak": 0.0 if (world == 1 or args.no_weak or args.scaling == "weak") else 6.0 * frac + 3 * 2.8 * frac,
         "cpu": 0.0 if (world > 1 or args.no_cpu) else 25.0 * (args.cpu_sample / 4096.0) * (args.years / 10.0) + 10.0}
    p["total"] = sum(p.values())
    return p


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp64_peak():
    p = os.path.join(ROOT, "profiles", "r01_fp64_microbench.json")
    if os.path.exists(p):
        return float(json.load(open(p))["dfma_per_s"]), "measured (tools/fp64_peak.cu, profiles/r01_fp64_microbench.json)"
    return 1.86e13, "nominal 148 SM x 64 DFMA/clk x 1.965 GHz"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def required_spin_days(passes) -> int:
    """Spin-up cell-days of the reference algorithm: aridity pass + passes x (365 + check day)."""
    p = passes.to("cpu").double().numpy() if hasattr(passes, "to") else np.asarray(passes, dtype=np.float64)
    return int((365 + p * 366).sum())


# --------------------------------------------------------------------------------------------------
# workload: which cells a rank owns
# --------------------------------------------------------------------------------------------------
def rank_cells(grid: synthetic.Grid, world: int, rank: int, strong: bool):
    """-> list of (c0, c1) contiguous global cell ranges of this rank, ascending.  Strong scaling: blocks of
    ROW_BLOCK grid rows dealt round-robin (block b -> rank b % world); weak: the whole grid."""
    if not strong or world == 1:
        return [(0, grid.n_cells)]
    rs = grid.row_start
    n_rows = len(grid.rows_n)
    segs = []
    for b, r0 in enumerate(range(0, n_rows, ROW_BLOCK)):
        if b % world != rank:
            continue
        c0, c1 = int(rs[r0]), int(rs[min(n_rows, r0 + ROW_BLOCK)])
        if c1 > c0:
            if segs and segs[-1][1] == c0:
                segs[-1] = (segs[-1][0], c1)
            else:
                segs.append((c0, c1))
    return segs


def seg_index(segs) -> np.ndarray:
    return np.concatenate([np.arange(a, b, dtype=np.int64) for a, b in segs]) if segs else np.zeros(0, np.int64)


def dump_sample(n_cells: int, values_per_cell: int, finite_of) -> np.ndarray:
    """Local cell indices written by --dump-outputs, ascending: the first cells, in an order drawn with DUMP_SEED, for
    which finite_of(ascending local indices) -> bool mask says that their result is finite, as many as fit in DUMP_BYTES
    (f64, with room for the .npy headers).  finite_of is the host checker (host_finite), so the choice depends on the
    inputs only and every build writes the same cells.  The reference's own arithmetic overflows to inf in ro / bflow for
    some very sandy soils (about 0.5 % of the grid: pow(x, 1/lambda) underflows, then exp() overflows); such values
    cannot be compared within a tolerance."""
    order = np.random.default_rng(DUMP_SEED).permutation(n_cells)
    k = min(n_cells, (DUMP_BYTES - 64 * 1024) // (8 * values_per_cell))
    chosen, pos = [], 0
    while len(chosen) < k and pos < n_cells:
        batch = order[pos:pos + (k - len(chosen)) * 51 // 50 + 64]  # ~0.5 % of the cells are dropped
        pos += len(batch)
        ok = set(np.sort(batch)[finite_of(np.sort(batch))].tolist())
        chosen += [c for c in batch.tolist() if c in ok]
    return np.sort(np.asarray(chosen[:k], dtype=np.int64))


def host_finite(grid, index, n_years):
    """finite_of for dump_sample: which of the local cells `sub` (global cells index[sub]) have a finite result, all
    monthly layers and cell_diag, on the C restatement of the reference core (tests/oracle_lib.py), on all host cores."""
    from tests import oracle_lib as ol

    def finite_of(sub):
        r = ol.run_cpu(host_problem(grid, index[sub], n_years), monthly=True)
        return np.all([np.isfinite(r[k]).all(0) for k in _abi.OUTPUT_NAMES + ("cell_diag",)], axis=0)
    return finite_of


def grid_in_struct(n_cells, n_days, year, doy, month, sw, tc, pn, cells, mem_kind, f32):
    s = _abi.SplashGridIn()
    s.n_cells, s.n_days, s.cell_stride = n_cells, n_days, n_cells
    s.year = year.ctypes.data_as(_abi.c_int32_p)
    s.doy = doy.ctypes.data_as(_abi.c_int32_p)
    s.month = month.ctypes.data_as(_abi.c_int32_p)
    s.sw_in, s.tc, s.pn = sw, tc, pn
    for k in ("lat", "elev", "slop", "asp", "resolution", "soil", "au"):
        setattr(s, k, cells[k])
    s.au_layers = 3
    s.mem_kind = mem_kind
    s.forcing_dtype = _abi.SPLASH_F32 if f32 else _abi.SPLASH_F64
    return s


def grid_out_struct(n_out, n_cells, ptrs, diag, mem_kind):
    s = _abi.SplashGridOut()
    s.n_out, s.cell_stride, s.mem_kind = n_out, n_cells, mem_kind
    for k, p in zip(_abi.OUTPUT_NAMES, ptrs):
        setattr(s, k, p)
    s.cell_diag = diag
    return s


# --------------------------------------------------------------------------------------------------
# reference / CPU arm
# --------------------------------------------------------------------------------------------------
def sample_indices(n_cells: int, sample_cells: int) -> np.ndarray:
    """Global cell indices of the CPU sample: evenly spread over the grid (every latitude band)."""
    return np.unique(np.linspace(0, n_cells - 1, min(sample_cells, n_cells)).astype(np.int64))


def cpu_sample_problem(sample_cells, n_years, n_cells=synthetic.N_CELLS_5ARCMIN):
    """The CPU legs' bounded sample: a SUBSET of the benchmark grid (same seed, same generator)."""
    grid = synthetic.Grid(n_cells, GRID_SEED)
    pick = sample_indices(n_cells, sample_cells)
    return host_problem(grid, pick, n_years), pick


def host_problem(grid, pick, n_years):
    """Host copy (f64) of the inputs of the grid's cells `pick` (global indices, ascending)."""
    from tests import oracle_lib as ol

    cells = grid.cells(pick)
    dates = synthetic.daily_dates(FIRST_YEAR, n_years)
    year, doy, month = _abi.time_axes(dates)
    sw, tc, pn = grid.forcing(cells, doy)
    return ol.GridProblem(year, doy, month, sw, tc, pn, cells["lat"], cells["elev"], cells["slop"], cells["asp"],
                          cells["resolution"], cells["soil"], cells["au"])


def time_cpu(prob, core, threads):
    from tests import oracle_lib as ol

    t = time.perf_counter()
    r = ol.run_cpu(prob, monthly=True, core=core, n_threads=threads)
    dt = time.perf_counter() - t
    return dt, r


def cpu_leg(sample_cells, n_years, steps=1, warmup=0, n_cells=synthetic.N_CELLS_5ARCMIN):
    """Times the reference's own CPU implementation (unmodified C++ core from oracle/_ref when it
    was compiled, else the C restatement) on all host cores.  Returns (value, seconds, info, problem, pick, result)."""
    from tests import oracle_lib as ol

    ol.oracle()
    kind = "reference" if ol.have_ref() else "port"
    core = "ref" if kind == "reference" else "oracle"
    threads = os.cpu_count() or 1
    prob, pick = cpu_sample_problem(sample_cells, n_years, n_cells)
    # pass counts (hence the job size) from the restated core: it is bit-identical to the reference core
    _, r0 = time_cpu(prob, "oracle", threads)
    job = prob.n_cells * prob.n_days + required_spin_days(r0["cell_diag"][_abi.DIAG_NAMES.index("spin_passes")])
    for _ in range(warmup):
        time_cpu(prob, core, threads)
    times, res = [], None
    for _ in range(max(1, steps)):
        dt, res = time_cpu(prob, core, threads)
        times.append(dt)
    dt = float(np.mean(times))
    res["cell_diag"][_abi.DIAG_NAMES.index("spin_passes")] = r0["cell_diag"][_abi.DIAG_NAMES.index("spin_passes")]
    info = {"value": job / dt, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{prob.n_cells} cells x {prob.n_days} days (+ spin-up), a subset of the benchmark grid (same counter-based "
                      f"generator and seed), C++ core only ({'unmodified reference sources' if kind == 'reference' else 'C restatement'}; "
                      f"R-side prep restated in C), {threads} threads, {dt:.2f} s per pass"}
    return job / dt, dt, info, prob, pick, res


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    value, dt, info, _, _, _ = cpu_leg(args.cpu_sample, args.years, steps=args.steps, warmup=args.warmup, n_cells=args.cells)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"synthetic 5-arcmin global grid x {args.years} years daily incl. spin-up, monthly outputs; "
                               f"CPU sample of {args.cpu_sample} cells of that grid", "cells": args.cpu_sample, "days_per_cell": None},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def parity_block(prob, ref, got_layers, got_passes) -> dict:
    """GPU results of the sample cells (monthly layers, [n_out, n]) against the reference run of the same cells:
    NaN masks, the north_star gates on monthly values, and -- for the cells outside them -- whether the reference
    itself is ill-conditioned there (tests/conditioning.py: its own result moves under a 1-ulp libm change)."""
    from tests import parity

    n = prob.n_cells
    mask_equal = True
    off = np.zeros(n, dtype=bool)
    worst, per_cell = {}, {}
    for k in _abi.OUTPUT_NAMES:
        g, r = got_layers[k], ref[k]
        gm, rm = np.isnan(g), np.isnan(r)
        if not np.array_equal(gm, rm):
            mask_equal = False
            off |= (gm != rm).any(0)
        ok = ~gm & ~rm & np.isfinite(g) & np.isfinite(r)
        d = np.where(ok, np.abs(g - r), 0.0)
        if k in parity.FLUX:
            lim = parity.REL_FLUX * np.abs(np.where(ok, r, 0.0)) + parity.ABS_GUARD * 31
            bad = d > lim
            w = float((d / np.maximum(np.abs(np.where(ok, r, 1.0)), 1e-3)).max()) if ok.any() else 0.0
        else:
            lim = 1e-8 if k == "sm_lim" else parity.ABS_STATE_MM * (31 if k in ("ro", "bflow") else 1)
            bad = d > lim
            w = float(d.max()) if ok.any() else 0.0
        off |= bad.any(0)
        worst[k] = w
        worst_per_cell = d.max(0) if k not in parity.FLUX else (d / np.maximum(np.abs(np.where(ok, r, 1.0)), 1e-3)).max(0)
        per_cell[k] = worst_per_cell
    passes_equal = int((got_passes == ref["cell_diag"][_abi.DIAG_NAMES.index("spin_passes")]).sum())
    out = {"cells_compared": int(n), "layers": "9 monthly layers", "nan_masks_equal": bool(mask_equal),
           "cells_outside_gates": int(off.sum()), "spin_passes_equal_cells": passes_equal,
           "worst_error_inside_gates": {k: float(v[~off].max()) if (~off).any() else 0.0 for k, v in per_cell.items()},
           "worst_error_all_cells": worst,
           "gates": "<= 1e-9 relative on pet/netr/aet/cond, <= 1e-6 mm on wn/snow (x31 on monthly sums ro/bflow), 1e-8 on sm_lim",
           "against": "oracle/_ref (unmodified reference C++ core) run in this process on the same cells"}
    if off.any():
        try:
            from tests import conditioning
            sub = prob.subset(np.flatnonzero(off))
            sparse, _ = conditioning.stable_cells(sub, None, conditioning.SPARSE)
            dense, _ = conditioning.stable_cells(sub, None, conditioning.DENSE)
            out["outside_of_which_reference_stable_sparse"] = int(sparse.sum())
            out["outside_of_which_reference_stable_dense"] = int((sparse & dense).sum())
        except Exception as e:  # the screen needs the perturbed oracle builds (make -C oracle sens)
            out["conditioning_screen"] = f"unavailable: {e}"
    return out


# --------------------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------------------
class Shard:
    """A rank's cells of one grid, resident on the device: per-cell attributes (f64) and f32 forcing."""

    def __init__(self, torch, device, grid, segs, doy, filler=None):
        self.segs = segs
        self.index = seg_index(segs)
        self.nc = len(self.index)
        nd = len(doy)
        self.cells_np = grid.cells(self.index)
        dev = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=device)
        self.cells = {k: dev(self.cells_np[k]) for k in ("lat", "elev", "slop", "asp", "resolution", "soil", "au")}
        self.filler = filler or synthetic.DeviceFiller(grid, doy, device)
        self.f = [torch.empty((nd, self.nc), dtype=torch.float32, device=device) for _ in range(3)]
        o = 0
        for a, b in segs:  # the generator fills contiguous cell ranges
            sub = {k: (v[..., o:o + (b - a)] if isinstance(v, np.ndarray) else v) for k, v in self.cells_np.items()}
            self.filler.fill(sub, self.f[0][:, o:], self.f[1][:, o:], self.f[2][:, o:])
            o += b - a

    def ptrs(self):
        return {k: v.data_ptr() for k, v in self.cells.items()}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from rsplash_b200 import build
    from rsplash_b200._lib import Context

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libsplash_cuda has no CPU path (use --impl reference for the CPU arm)")
    t_start = time.perf_counter()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    build.build()
    if not os.path.exists(os.path.join(ROOT, "tools", "synth", "libsplash_synth.so")):
        subprocess.run(["make", "-C", os.path.join(ROOT, "tools", "synth")], check=True, capture_output=True)
    ctx = Context(local_rank)

    strong = args.scaling == "strong"
    grid = synthetic.Grid(args.cells, GRID_SEED)
    dates = synthetic.daily_dates(FIRST_YEAR, args.years)
    year, doy, month = _abi.time_axes(dates)
    nd = len(dates)
    n_out = _abi.count_months(year, month)
    phases = {}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def allreduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op={"max": dist.ReduceOp.MAX, "sum": dist.ReduceOp.SUM}[op])
        return float(t.item())

    # ---- resident workload (value leg) -------------------------------------------------------------
    t0 = time.perf_counter()
    segs = rank_cells(grid, world, rank, strong)
    if not strong and world > 1:
        grid = synthetic.Grid(args.cells, GRID_SEED + rank)  # weak: every rank its own forcing realisation
    shard = Shard(torch, device, grid, segs, doy)
    nc = shard.nc
    outs = [torch.empty((n_out, nc), dtype=torch.float64, device=device) for _ in range(9)]
    diag = torch.empty((_abi.SPLASH_NDIAG, nc), dtype=torch.float64, device=device)
    cin = grid_in_struct(nc, nd, year, doy, month, shard.f[0].data_ptr(), shard.f[1].data_ptr(), shard.f[2].data_ptr(),
                         shard.ptrs(), _abi.SPLASH_MEM_DEVICE, f32=True)
    cout = grid_out_struct(n_out, nc, [o.data_ptr() for o in outs], diag.data_ptr(), _abi.SPLASH_MEM_DEVICE)
    opts = _abi.SplashOpts()
    opts.monthly_out = 1
    torch.cuda.synchronize()
    phases["generate_s"] = time.perf_counter() - t0

    # ---- value: W warm-up + K timed steps, inputs resident -------------------------------------------
    t0 = time.perf_counter()
    stats_steps = []
    for _ in range(args.warmup):
        ctx.grid_run(cin, opts, cout)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    tv = time.perf_counter()
    for _ in range(args.steps):
        ctx.grid_run(cin, opts, cout)  # synchronous: returns after its streams are drained
        stats_steps.append(ctx.stats())
    barrier()
    t_value = time.perf_counter() - tv
    clocks = sampler.stop()
    t_value = allreduce(t_value, "max")
    passes = diag[_abi.DIAG_NAMES.index("spin_passes")]
    job_rank = nc * nd + required_spin_days(passes)
    job_total = allreduce(float(job_rank), "sum")
    executed_rank = nc * nd + float(np.mean([s["spin_cell_days"] for s in stats_steps]))
    executed_total = allreduce(executed_rank, "sum")
    cells_all = allreduce(float(nc), "sum")
    ms_per_step = t_value / args.steps * 1e3
    value = job_total / (t_value / args.steps)
    launches = int(sum(s["kernel_launches"] for s in stats_steps))
    finite_frac = float(torch.isfinite(outs[0]).double().mean().item())
    phases["value_s"] = time.perf_counter() - t0

    # what the last timed step computed, before the roofline leg below writes into the same buffers
    if args.dump_outputs and rank == 0:
        pick = dump_sample(nc, len(outs) * n_out + _abi.SPLASH_NDIAG + 1, host_finite(grid, shard.index, args.years))
        pt = torch.as_tensor(pick, device=device)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, o in zip(_abi.OUTPUT_NAMES + ("cell_diag",), outs + [diag]):
            np.save(os.path.join(args.dump_outputs, f"{k}.npy"), o[:, pt].cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "cell_index.npy"), shard.index[pick].astype(np.float64))  # global grid cells

    # GPU results of the parity sample (rank 0, N == 1: the CPU leg runs the same cells on the reference)
    sample_got = None
    if rank == 0 and world == 1 and not args.no_cpu:
        pick = sample_indices(args.cells, args.cpu_sample)  # at N == 1 local index == global index
        pt = torch.as_tensor(pick, device=device)
        sample_got = {k: o[:, pt].cpu().numpy() for k, o in zip(_abi.OUTPUT_NAMES, outs)}
        sample_passes = passes[pt].cpu().numpy()

    # ---- roofline of the dominant kernel: the bulk daily-integration kernel (k_run_bulk) run ALONE over the whole
    #      shard -- a resume call (skip_spinup) launches nothing else of weight -- and timed with CUDA events on its
    #      streams inside the library (splash_stats.bulk_span_ms) ---------------------------------------------------
    t0 = time.perf_counter()
    hbm_peak, hbm_src = peaks()
    dfma_peak, dfma_src = fp64_peak()
    st_dev = torch.empty((_abi.SPLASH_NSTATE, nc), dtype=torch.float64, device=device)
    cout_st = grid_out_struct(n_out, nc, [o.data_ptr() for o in outs], diag.data_ptr(), _abi.SPLASH_MEM_DEVICE)
    cout_st.state_final = st_dev.data_ptr()
    ctx.grid_run(cin, opts, cout_st)                      # spun-up state of every cell
    st_host = st_dev.cpu().numpy().copy()
    ropts = _abi.SplashOpts()
    ropts.monthly_out, ropts.skip_spinup = 1, 1
    ropts.state_init = st_host.ctypes.data_as(C.c_void_p)
    spans = []
    n_roof = min(max(1, args.steps), ROOFLINE_MAX_STEPS)
    for i in range(1 + n_roof):
        ctx.grid_run(cin, ropts, cout)
        if i:
            spans.append(ctx.stats()["bulk_span_ms"])
            launches += ctx.stats()["kernel_launches"]
    bulk_ms = float(np.mean(spans))
    bulk_launches = int(ctx.stats()["n_tiles"])
    bulk_cell_days = nc * nd
    alg_bytes_per_cd = 3 * 4 + 9 * 8 * n_out / nd  # f32 forcing read + monthly layers written
    hbm_achieved = bulk_cell_days * alg_bytes_per_cd / (bulk_ms * 1e-3) / 1e9
    inst_cd, flops_cd, work_src = fp64_work_per_cell_day()
    hbm_part = {"achieved": hbm_achieved, "peak": hbm_peak, "frac": hbm_achieved / hbm_peak, "unit": "GB/s",
                "peak_source": hbm_src, "algorithmic_bytes_per_cell_day": alg_bytes_per_cd}
    roofline = {
        "bound": "fp64", "kernel": "k_run_bulk (daily integration of every cell of the shard), timed alone", "steps": n_roof,
        "unit": "TFLOP/s", "achieved": None, "peak": 2 * dfma_peak / 1e12, "frac": None, "traffic": None,
        "peak_source": dfma_src, "fp64_inst_per_cell_day": inst_cd, "flops_per_cell_day": flops_cd, "work_source": work_src,
        "kernel_ms_per_launch": bulk_ms / bulk_launches, "launches_per_pass": bulk_launches,
        "cell_days_per_launch": bulk_cell_days / bulk_launches, "cell_days_per_s": bulk_cell_days / (bulk_ms * 1e-3),
        "note": "the path is bound by the FP64 pipe (transcendentals), not by HBM and not by tensor cores; "
                "the HBM figures are given beside it",
        "hbm": hbm_part,
    }
    if flops_cd:
        roofline["achieved"] = bulk_cell_days * flops_cd / (bulk_ms * 1e-3) / 1e12
        roofline["frac"] = roofline["achieved"] / roofline["peak"]
        roofline["fp64_pipe_frac"] = bulk_cell_days * inst_cd / (bulk_ms * 1e-3) / dfma_peak
    tr = os.path.join(ROOT, "profiles", "fp64_work.json")
    if os.path.exists(tr):
        roofline["traffic"] = json.load(open(tr)).get("dram_bytes_per_cell_day")
        if roofline["traffic"] is not None:
            roofline["traffic"] = roofline["traffic"] * bulk_cell_days / bulk_launches
            roofline["traffic_source"] = ("dram__bytes_read + dram__bytes_write per cell-day of the ncu capture named in work_source (a "
                                          "ONE-year launch: the per-cell constants, read once per launch, weigh 10x more in it than in "
                                          "the 10-year launches timed here), scaled to this launch's cell-days")
    shard_index, shard_cells_np, filler = shard.index, shard.cells_np, shard.filler
    del st_dev, cout, cout_st, outs, diag, shard, cin   # the resident forcing is not needed any more
    torch.cuda.empty_cache()
    phases["roofline_s"] = time.perf_counter() - t0

    # ---- e2e: the same job through the C ABI with pinned HOST buffers, row blocks through the block scheduler ----
    e2e = None
    if not args.no_e2e:
        t0 = time.perf_counter()
        # pinned f64 forcing: at most ~45 % of what the host has free, shared by the ranks of the box
        pin_budget = 76e9
        try:
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
            pin_budget = min(pin_budget, 0.45 * avail / world)
        except Exception:
            pass
        # One pinned block at a time, as large as the budget allows (fewer calls = fewer exposed straggler tails): the
        # block is staged once, then run for the warm-up and every timed pass; a pass is the sum over the blocks.
        per_cell = nd * 3 * 8 + n_out * 9 * 8 + 14 * 8
        bsz = int(min(nc, max(1024, (pin_budget / per_cell) // 1024 * 1024)))
        if args.e2e_blocks:
            bsz = int(np.ceil(nc / args.e2e_blocks / 1024) * 1024)
        else:  # equal blocks
            bsz = int(np.ceil(nc / np.ceil(nc / bsz) / 1024) * 1024)
        n_blocks = int(np.ceil(nc / bsz))
        pin = lambda *shape: torch.empty(shape, dtype=torch.float64, pin_memory=True)
        buf = {"f": [pin(nd, bsz) for _ in range(3)], "out": [pin(n_out, bsz) for _ in range(9)],
               "cells": {k: np.zeros((v.shape[0], bsz) if v.ndim == 2 else (bsz,)) for k, v in shard_cells_np.items()
                         if k in ("lat", "elev", "slop", "asp", "resolution", "soil", "au")}}
        bufs = [buf]
        chunk_days = max(1, int(2e9 // (bsz * 8 * 3)))
        d_chunk = [torch.empty((chunk_days, bsz), dtype=torch.float64, device=device) for _ in range(3)]
        hopts = _abi.SplashOpts()
        hopts.monthly_out = 1
        phases["e2e_alloc_s"] = time.perf_counter() - t0

        def stage(b):
            """block b's inputs into pinned host memory (untimed: this is the caller's data): generated on the device, copied out"""
            b0, b1 = b * bsz, min(nc, (b + 1) * bsz)
            n = b1 - b0
            idx = shard_index[b0:b1]
            # contiguous runs of global cells inside the block (shard boundaries of the round-robin deal)
            cuts = np.flatnonzero(np.diff(idx) != 1) + 1
            runs = np.split(np.arange(n), cuts)
            for d0 in range(0, nd, chunk_days):
                d1 = min(nd, d0 + chunk_days)
                for r in runs:
                    sub = {k: (v[..., b0 + r[0]:b0 + r[-1] + 1] if isinstance(v, np.ndarray) else v) for k, v in shard_cells_np.items()}
                    filler.fill(sub, d_chunk[0][:, r[0]:], d_chunk[1][:, r[0]:], d_chunk[2][:, r[0]:], day0=d0, n_days=d1 - d0)
                for h, dsrc in zip(buf["f"], d_chunk):
                    h[d0:d1, :n].copy_(dsrc[:d1 - d0, :n])
            for k, v in buf["cells"].items():
                v[..., :n] = shard_cells_np[k][..., b0:b1]
            torch.cuda.synchronize()
            return n

        def structs(n):
            hp = {k: v.ctypes.data for k, v in buf["cells"].items()}
            bin_ = grid_in_struct(n, nd, year, doy, month, buf["f"][0].data_ptr(), buf["f"][1].data_ptr(), buf["f"][2].data_ptr(), hp,
                                  _abi.SPLASH_MEM_HOST, f32=False)
            bin_.cell_stride = bsz
            bin_.attr_stride = bsz
            bout = grid_out_struct(n_out, n, [o.data_ptr() for o in buf["out"]], None, _abi.SPLASH_MEM_HOST)
            bout.cell_stride = bsz
            return bin_, bout

        n_e2e = min(max(1, args.steps), E2E_MAX_STEPS)
        t_steps = np.zeros(n_e2e)
        h2d_b = d2h_b = 0
        block_stats = []
        barrier()  # the ranks start their host-fed passes together (they share the host's memory and PCIe fabric)
        for b in range(n_blocks):
            bin_, bout = structs(stage(b))
            for rep in range((1 if b == 0 else 0) + n_e2e):   # one untimed call of the first block sizes the device buffers
                k = rep - (1 if b == 0 else 0)
                torch.cuda.synchronize()
                t = time.perf_counter()
                ctx.grid_run(bin_, hopts, bout)
                dt = time.perf_counter() - t
                if k >= 0:
                    t_steps[k] += dt
                    s_ = ctx.stats()
                    launches += s_["kernel_launches"]
                    if k == n_e2e - 1:
                        h2d_b += s_["h2d_bytes"]
                        d2h_b += s_["d2h_bytes"]
                        block_stats.append({q: s_[q] for q in ("total_ms", "gpu_ms", "h2d_ms", "d2h_ms", "pool_wait_ms", "first_ms", "rounds_ms",
                                                               "bulk_ms", "n_tiles", "tile_cells", "pool_cells", "pool_max_passes")})
        t_e2e = allreduce(float(t_steps.mean()), "max")
        e2e = {"value": job_total / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d_b), "d2h_bytes_per_step": int(d2h_b),
               "ms_per_step": t_e2e * 1e3, "steps": n_e2e, "row_blocks": n_blocks,
               "host_buffers": "pinned f64 (what R's REAL() holds), day-major; one block of rows per call (splash_grid_run on host "
                               "pointers), each block staged once and run for every timed pass",
               "block_stats_last_step": block_stats}
        del bufs, buf, d_chunk
        torch.cuda.empty_cache()
        phases["e2e_s"] = time.perf_counter() - t0

    # ---- weak-scaling figure beside the strong one (N > 1): one whole grid per rank ------------------------
    weak_value = None
    if world > 1 and strong and not args.no_weak:
        t0 = time.perf_counter()
        wgrid = synthetic.Grid(args.cells, GRID_SEED + 1000 + rank)
        wshard = Shard(torch, device, wgrid, [(0, wgrid.n_cells)], doy)
        wn = wshard.nc
        wouts = [torch.empty((n_out, wn), dtype=torch.float64, device=device) for _ in range(9)]
        wdiag = torch.empty((_abi.SPLASH_NDIAG, wn), dtype=torch.float64, device=device)
        win = grid_in_struct(wn, nd, year, doy, month, wshard.f[0].data_ptr(), wshard.f[1].data_ptr(), wshard.f[2].data_ptr(),
                             wshard.ptrs(), _abi.SPLASH_MEM_DEVICE, f32=True)
        wout = grid_out_struct(n_out, wn, [o.data_ptr() for o in wouts], wdiag.data_ptr(), _abi.SPLASH_MEM_DEVICE)
        ctx.grid_run(win, opts, wout)
        barrier()
        tw = time.perf_counter()
        for _ in range(2):
            ctx.grid_run(win, opts, wout)
        barrier()
        t_weak = allreduce(time.perf_counter() - tw, "max")
        wjob = allreduce(float(wn * nd + required_spin_days(wdiag[_abi.DIAG_NAMES.index("spin_passes")])), "sum")
        weak_value = wjob / (t_weak / 2)
        del wshard, wouts, wdiag
        phases["weak_s"] = time.perf_counter() - t0

    # ---- CPU baseline beside it, and the parity of the benchmark grid's own cells (rank 0, N == 1 only) ----------
    cpu = None
    parity_rep = None
    if rank == 0 and world == 1 and not args.no_cpu:
        t0 = time.perf_counter()
        try:
            _, _, cpu, prob, pick, ref = cpu_leg(args.cpu_sample, args.years, n_cells=args.cells)
            if sample_got is not None:
                parity_rep = parity_block(prob, ref, sample_got, sample_passes)
        except Exception as e:  # the checker is optional for the measurement itself
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
        phases["cpu_s"] = time.perf_counter() - t0

    if rank == 0:
        phases["total_s"] = time.perf_counter() - t_start
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"synthetic 5-arcmin global grid ({args.cells} land cells) x {args.years} years daily "
                            f"({nd} days) incl. spin-up, monthly outputs (BASELINE.json configs[3])",
                "cells_total": int(cells_all), "cells_rank0": nc, "n_days": nd, "n_out_layers": 9, "n_months": n_out,
                "parallelism": (f"one grid, blocks of {ROW_BLOCK} grid rows dealt round-robin to {world} rank(s), no data-path collective"
                                if strong else f"{world} rank(s), one whole grid (own forcing realisation) per rank, no data-path collective"),
                "generator": f"counter-based splitmix64(seed {GRID_SEED}, cell, day, field): shards, row blocks and the CPU sample are subsets of one grid",
                "forcing_hbm_dtype": "f32 (lossless: values are FP32-representable like the FLT4S rasters)",
                "l2": "inputs per step (>= 10 GB per rank) are far larger than the 126 MB L2",
                "job_cell_days": job_total, "executed_cell_days": executed_total,
                "executed_cell_days_per_s": executed_total / (ms_per_step * 1e-3),
                "spin_share_of_job": 1.0 - cells_all * nd / job_total,
                "finite_fraction_wn": finite_frac,
                # SURVEY 8(d): the series days alone over the same wall time, so that spin-up pass counts do not blur it
                "nd_only_cell_days_per_s": cells_all * nd / (ms_per_step * 1e-3),
                "weak_value": weak_value if weak_value is not None else (value if world == 1 or not strong else None),
                "phases_s": {k: round(v, 1) for k, v in phases.items()},
            },
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "parity": parity_rep, "e2e": e2e, "gpu_launches": launches,
            "stats_last_step": stats_steps[-1],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
