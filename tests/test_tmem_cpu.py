"""CPU: the bulk launch keeps its cold constants and monthly sums in tensor memory.  ptxas's resource report and the SASS
of the library, built for sm_100a into a temporary directory: every k_run_bulk instantiation moves data to and from TMEM
(STTM / LDTM) and spills no more than the numbers below, and no other kernel touches TMEM."""
import os
import re
import subprocess
import tempfile

from rsplash_b200 import build

# Spill stores / loads (bytes) of k_run_bulk<FT, kMonthly> with CUDA 12.9.  768 threads x 80 registers is the whole
# register file, and the day step's peak working set is larger than 80 registers: what is left spills in the state
# half, not around the cold constants or the monthly sums (304-624 B of stores with those in registers / L2).
MAX_SPILL = {
    ("f", "0"): (296, 440),
    ("f", "1"): (320, 444),
    ("d", "0"): (364, 464),
    ("d", "1"): (380, 468),
}


def _build():
    with tempfile.TemporaryDirectory() as d:
        lib = os.path.join(d, "libsplash_cuda.so")
        r = subprocess.run([build.nvcc_path(), *build.NVCC_FLAGS, "-o", lib, *build.SOURCES], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        cuobjdump = os.path.join(os.path.dirname(build.nvcc_path()), "cuobjdump")
        s = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True)
        assert s.returncode == 0, s.stderr[-2000:]
    return r.stderr, s.stdout


def _sass_by_function(sass):
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur:
            out[cur].append(line)
    return out


def test_bulk_kernel_uses_tmem_and_no_other_kernel_does():
    report, sass = _build()
    funcs = _sass_by_function(sass)
    bulk = {f: "\n".join(v) for f, v in funcs.items() if "k_run_bulk" in f}
    assert len(bulk) == 4, sorted(bulk)
    for (ft, monthly), (max_st, max_ld) in MAX_SPILL.items():
        name = [f for f in bulk if re.search(r"k_run_bulkI%sLb%sE" % (ft, monthly), f)]
        assert len(name) == 1, (ft, monthly, sorted(bulk))
        body = bulk[name[0]]
        assert re.search(r"\bSTTM\b", body) and re.search(r"\bLDTM\b", body), name[0]
        m = re.search(r"Compiling entry function '%s' for 'sm_100a'\n.*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                      r"(\d+) bytes spill loads" % re.escape(name[0]), report)
        assert m, name[0]
        assert int(m.group(2)) <= max_st and int(m.group(3)) <= max_ld, (name[0], m.group(0))
    for f, lines in funcs.items():
        if "k_run_bulk" in f:
            continue
        body = "\n".join(lines)
        assert not re.search(r"\b(STTM|LDTM|UTCATOMSWS)\b", body), f
