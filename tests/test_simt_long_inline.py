"""The "long_regions" option of bk_compare_kmers_batch on the emulated library of tests/sim against the oracle: one call
with a C2 region, reads of 4,500 and 6,000 bases, a contig that grows past 4,095 bases and a read of 65,536 bases; one
at k = 21; and a region whose assemble_kernel attempt emits contigs before it stops (they must not reach the result).
The regions run in a child process with BK_LIB pointing at the emulator build, as tests/test_simt_long_regions.py
does; under AddressSanitizer with exact-size allocations when BK_TEST_ASAN=1.  route_long_kernel and the device queue
are where an off-by-one would hide."""
import json
import os
import subprocess
import sys

import pytest

import sim_util
from conftest import ROOT

CHILD = r"""
import json, sys
import numpy as np
sys.path.insert(0, "tests")
from breakmer_b200 import _lib, batch, synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only
from test_gpu_long_inline import MIX_READ_LEN, mixed_region
from test_gpu_long_regions import GROWING_REGION, LONG_READ_REGIONS, over_limit_region
lr = dict(LONG_READ_REGIONS)
calls = [[synth.config_region("C2", 1), synth.make_region("lr0", **lr["lr0"]), synth.make_region("lr2", **lr["lr2"]),
          synth.make_region(*GROWING_REGION[:1], **GROWING_REGION[1]), over_limit_region(65536)],
         [synth.make_region("lr1", **lr["lr1"])],
         [mixed_region()]]
h = _lib.Handle(0)
h.set_option("long_regions", 1)
rows = []
for regions in calls:
    pk = batch.PackedBatch(regions)
    mix = regions[0].name == "mix"
    if mix:
        pk.read_len = np.array([MIX_READ_LEN, 0], dtype=np.int32)
    out = batch.run(h, pk)
    for i, r in enumerate(regions):
        row = dict(name=r.name, status=int(out.region_status[i]), n_contigs=int(out.ctg_reg_off[i + 1] - out.ctg_reg_off[i]))
        if r.name != "zz_over":
            _a, _b, _c, only = oracle_sample_only(r)
            exp = assembler_py.init_assembly(only, r.reads, r.k, r.rc_thresh, MIX_READ_LEN if mix else r.read_len)
            got = out.contig_records(i)
            row.update(sample_only_equal=out.sample_only(i) == only, contigs_equal=got == exp,
                       max_contig=max([len(c["seq"]) for c in got] or [0]))
        rows.append(row)
h.close()
print("RESULT " + json.dumps(rows))
"""


def _run(library, extra_env=None):
    env = dict(os.environ, BK_LIB=library, PYTHONPATH=ROOT)
    env.update(extra_env or {})
    out = subprocess.run([sys.executable, "-c", CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=2400)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and line, out.stdout[-2000:] + out.stderr[-4000:]
    return json.loads(line[0][len("RESULT "):]), out.stderr


def _check(rows):
    by = {r["name"]: r for r in rows}
    assert set(by) == {"C2_00001", "lr0", "lr1", "lr2", "grow", "zz_over", "mix"}
    assert by["zz_over"]["status"] == -4 and by["zz_over"]["n_contigs"] == 0
    assert by["grow"]["max_contig"] > 4095
    for r in rows:
        if r["name"] != "zz_over":
            assert r["status"] == 0 and r["sample_only_equal"] and r["contigs_equal"], r


def test_long_regions_inline_on_the_emulated_library():
    _check(_run(sim_util.build_simt("libbreakmer_simt_TESTONLY.so", "all.cpp"))[0])


def test_long_regions_inline_under_address_sanitizer():
    if not os.environ.get("BK_TEST_ASAN"):
        pytest.skip("set BK_TEST_ASAN=1 to build and run the AddressSanitizer library")
    lib = sim_util.build_simt("libbreakmer_simt_asan_TESTONLY.so", "all.cpp",
                              extra=["-O1", "-g", "-DSIMT_ARENA_MALLOC", "-fsanitize=address,undefined"])
    asan_rt = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    rows, err = _run(lib, {"LD_PRELOAD": asan_rt, "ASAN_OPTIONS": "detect_leaks=0:halt_on_error=1",
                           "UBSAN_OPTIONS": "print_stacktrace=1:halt_on_error=1"})
    assert "AddressSanitizer" not in err and "runtime error" not in err, err[-4000:]
    _check(rows)
