"""Development aid: the resident benchmark workload under different runtime knobs of the library
(SPLASH_POOL_STAGE1, SPLASH_ROUNDS_RT, SPLASH_CHAIN_FAST ... are read at context creation) and, with
SPLASH_CUDA_LIB=<path to a variant libsplash_cuda.so> in the environment of the process, under another build of it.
usage: knob_bench.py <cells> <years> "K1=V1,K2=V2" "K1=V3" ...   (one timed call per setting, after one warm-up)"""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import bench  # noqa: E402
from rsplash_b200 import _abi, synthetic  # noqa: E402
from rsplash_b200._lib import Context  # noqa: E402

n_cells, n_years = int(sys.argv[1]), int(sys.argv[2])
device = torch.device("cuda", 0)
grid = synthetic.Grid(n_cells, bench.GRID_SEED)
dates = synthetic.daily_dates(bench.FIRST_YEAR, n_years)
year, doy, month = _abi.time_axes(dates)
nd, n_out = len(dates), _abi.count_months(year, month)
shard = bench.Shard(torch, device, grid, [(0, n_cells)], doy)
nc = shard.nc
outs = [torch.empty((n_out, nc), dtype=torch.float64, device=device) for _ in range(9)]
diag = torch.empty((_abi.SPLASH_NDIAG, nc), dtype=torch.float64, device=device)
st_dev = torch.empty((_abi.SPLASH_NSTATE, nc), dtype=torch.float64, device=device)
cin = bench.grid_in_struct(nc, nd, year, doy, month, shard.f[0].data_ptr(), shard.f[1].data_ptr(), shard.f[2].data_ptr(),
                           shard.ptrs(), _abi.SPLASH_MEM_DEVICE, f32=True)
cout = bench.grid_out_struct(n_out, nc, [o.data_ptr() for o in outs], diag.data_ptr(), _abi.SPLASH_MEM_DEVICE)
cout.state_final = st_dev.data_ptr()
opts = _abi.SplashOpts()
opts.monthly_out = 1
keys = ("gpu_ms", "first_ms", "rounds_ms", "bulk_ms", "bulk_span_ms", "pool_wait_ms", "pool_cells", "pool_overflow_cells",
        "pool_max_passes", "n_tiles", "kernel_launches")
import hashlib
for setting in sys.argv[3:]:
    for kv in filter(None, setting.split(",")):
        k, v = kv.split("=")
        os.environ[k] = v
    ctx = Context(0)
    ctx.grid_run(cin, opts, cout)
    torch.cuda.synchronize()
    t = time.perf_counter()
    ctx.grid_run(cin, opts, cout)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    s = ctx.stats()
    # the bulk kernel alone: a resume call from the spun-up state
    st_host = st_dev.cpu().numpy().copy()
    ropts = _abi.SplashOpts()
    ropts.monthly_out, ropts.skip_spinup = 1, 1
    ropts.state_init = st_host.ctypes.data
    spans = []
    for i in range(3):
        ctx.grid_run(cin, ropts, cout)
        spans.append(ctx.stats()["bulk_span_ms"])
    digest = hashlib.sha1(outs[0].cpu().numpy().tobytes() + outs[3].cpu().numpy().tobytes()).hexdigest()[:12]
    print(setting or "(default)", "wall %.3f s" % dt, "bulk alone %.1f ms = %.3e cd/s" % (min(spans[1:]), nc * nd / (min(spans[1:]) * 1e-3)),
          json.dumps({k: (round(s[k], 1) if isinstance(s[k], float) else s[k]) for k in keys}), "digest", digest, flush=True)
    ctx.close()
    for kv in filter(None, setting.split(",")):
        os.environ.pop(kv.split("=")[0], None)
