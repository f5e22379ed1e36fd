"""The "rejected_contigs" option on the emulated library of tests/sim against the oracle: a few golden regions, the same
regions with every contig rejected for support and for length, and one call with the "long_regions" option where a
region with 4,500-base reads is routed to the long assembler.  The regions run in a child process with BK_LIB pointing at
the emulator build, as tests/test_simt_region_report.py does; under AddressSanitizer with exact-size allocations when
BK_TEST_ASAN=1."""
import json
import os
import subprocess
import sys

import pytest

import sim_util
from conftest import ROOT

CHILD = r"""
import json, sys
sys.path.insert(0, "tests")
from breakmer_b200 import _lib, batch, shard, synth
from test_gpu_long_regions import LONG_READ_REGIONS
from test_gpu_rejected_contigs import check_regions, forced, golden_regions, packed, run
# g001-g003 accept their contigs; g013 and g021 also reject some (so does C2 region 5)
regions = [golden_regions()[i] for i in (0, 1, 2, 12, 20)]
calls = [(regions, None, False), forced(regions[:2], "support") + (False,), forced(regions[:2], "length") + (False,),
         ([synth.config_region("C2", 5), synth.make_region("lr0", **dict(LONG_READ_REGIONS)["lr0"])], None, True)]
h = _lib.Handle(0)
rows = []
for regs, read_len, long_regions in calls:
    pk = packed(regs, read_len)
    out, rep = run(h, pk, long_regions=long_regions)
    n_rej = check_regions(out, rep, regs, read_len)
    off, _rep = run(h, pk, on=False, long_regions=long_regions)
    rows.append(dict(names=[r.name for r in regs], n_rejected=n_rej, reasons=sorted(set(out.rej_reason.tolist())),
                     n_contigs=out.n_contigs, passes=[row["pass"] for row in rep],
                     same_accepted=shard.region_digests(out, pk) == shard.region_digests(off, pk)))
h.close()
print("RESULT " + json.dumps(rows))
"""


def _run(lib, env_extra=None):
    env = dict(os.environ, BK_LIB=lib, PYTHONPATH=ROOT, **(env_extra or {}))
    out = subprocess.run([sys.executable, "-c", CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=3600)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and line, out.stdout[-2000:] + out.stderr[-4000:]
    assert "AddressSanitizer" not in out.stderr and "runtime error" not in out.stderr, out.stderr[-4000:]
    rows = json.loads(line[0][len("RESULT "):])
    assert len(rows) == 4
    assert all(r["same_accepted"] for r in rows), rows
    assert rows[0]["n_rejected"] > 0 and rows[3]["n_rejected"] > 0
    assert rows[1]["n_contigs"] == rows[2]["n_contigs"] == 0
    assert rows[1]["reasons"] == [1] and 2 in rows[2]["reasons"]           # (support is tested first)
    assert rows[1]["n_rejected"] > 0 and rows[2]["n_rejected"] > 0
    assert rows[3]["passes"] == ["batched", "long"]


def test_rejected_contigs_on_the_emulated_library():
    _run(sim_util.build_simt("libbreakmer_simt_TESTONLY.so", "all.cpp"))


def test_rejected_contigs_under_address_sanitizer():
    if not os.environ.get("BK_TEST_ASAN"):
        pytest.skip("set BK_TEST_ASAN=1 to build and run the AddressSanitizer library")
    lib = sim_util.build_simt("libbreakmer_simt_asan_TESTONLY.so", "all.cpp",
                              extra=["-O1", "-g", "-DSIMT_ARENA_MALLOC", "-fsanitize=address,undefined"])
    # libstdc++ is preloaded behind the runtime so that its __cxa_throw interceptor finds the real one: the getter throws
    # (and catches) internally for every result made with the option off
    rt = [subprocess.run(["g++", "-print-file-name=" + n], capture_output=True, text=True).stdout.strip()
          for n in ("libasan.so", "libstdc++.so.6")]
    _run(lib, {"LD_PRELOAD": " ".join(rt), "ASAN_OPTIONS": "detect_leaks=0:halt_on_error=1",
               "UBSAN_OPTIONS": "print_stacktrace=1:halt_on_error=1"})
