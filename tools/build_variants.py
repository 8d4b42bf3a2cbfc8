"""Development aid: builds named variants of libsplash_cuda.so (extra nvcc flags) into build/variants/ in parallel, for
A/B timing on the GPU with SPLASH_CUDA_LIB=<path> (tools/knob_bench.py).  usage: build_variants.py name=flags ..."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, ".")
from rsplash_b200 import build as b

out_dir = os.path.join("build", "variants")
os.makedirs(out_dir, exist_ok=True)


def one(spec):
    name, _, flags = spec.partition("=")
    out = os.path.join(out_dir, f"libsplash_{name}.so")
    cmd = [b.nvcc_path(), *b.NVCC_FLAGS, *flags.split(), "-o", out, *b.SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        return name, "FAILED\n" + r.stderr[-2000:]
    info = [l for l in r.stderr.splitlines() if "k_run_bulkIfLb1" in l or "k_spin_firstIf" in l]
    lines = r.stderr.splitlines()
    rep = []
    for i, l in enumerate(lines):
        if "Compiling entry function" in l and ("k_run_bulkIfLb1" in l or "k_pool_spin" in l):
            rep.append(l.split("'")[1][-40:] + " | " + lines[i + 1].strip() + " | " + lines[i + 2].strip().replace("ptxas info    : ", ""))
    return name, "\n   ".join(rep)


with ThreadPoolExecutor(max_workers=4) as ex:
    for name, rep in ex.map(one, sys.argv[1:]):
        print(name, "\n  ", rep, flush=True)
