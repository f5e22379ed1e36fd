"""bk_compare_kmers_long (assemble_long_kernel) on the emulated library of tests/sim against the oracle: a region with
4,500-base reads and a region whose contig grows past 4,095 bases from 3,000-base reads.  The regions run in a child
process with BK_LIB pointing at the emulator build (as tests/test_simt_library.py does).  The same run under
AddressSanitizer + UBSan, with every arena allocation an exact-size malloc, is opt-in (BK_TEST_ASAN=1): the per-CTA
scratch of the long kernel is sized per call, and that is where an out-of-bounds access would hide."""
import json
import os
import subprocess
import sys

import pytest

import sim_util
from conftest import ROOT

CHILD = r"""
import json, sys
from breakmer_b200 import _lib, batch, synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only
specs = [("lr0", dict(seed=11, L=10000, cov=6, k=15, e=0.003, event=("del", 300, None), rl=4500)),
         ("grow", dict(seed=22, L=7000, cov=60, k=15, e=0.002, event=("del", 300, None), rl=3000))]
h = _lib.Handle(0)
rows = []
for name, kw in specs:
    r = synth.make_region(name, **kw)
    _a, _b, _c, only = oracle_sample_only(r)
    exp = assembler_py.init_assembly(only, r.reads, r.k, r.rc_thresh, r.read_len)
    fast = list(batch.run(h, batch.PackedBatch([r])).region_status)
    out = batch.run(h, batch.PackedBatch([r]), long=True)
    got = out.contig_records(0)
    rows.append(dict(name=name, fast_status=[int(s) for s in fast], status=[int(s) for s in out.region_status],
                     sample_only_equal=out.sample_only(0) == only, contigs_equal=got == exp,
                     max_contig=max([len(c["seq"]) for c in got] or [0]), max_read=max(len(x[1]) for x in r.reads)))
h.close()
print("RESULT " + json.dumps(rows))
"""


def _run(library, extra_env=None):
    env = dict(os.environ, BK_LIB=library, PYTHONPATH=ROOT)
    env.update(extra_env or {})
    out = subprocess.run([sys.executable, "-c", CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and line, out.stdout[-2000:] + out.stderr[-4000:]
    return json.loads(line[0][len("RESULT "):]), out.stderr


def _check(rows):
    by = {r["name"]: r for r in rows}
    assert by["lr0"]["max_read"] > 4095 and by["lr0"]["fast_status"] == [-4]
    assert by["grow"]["max_read"] <= 4095 and by["grow"]["fast_status"] == [-4]      # the fast kernel's growth check
    assert by["grow"]["max_contig"] > 4095
    for r in rows:
        assert r["status"] == [0] and r["sample_only_equal"] and r["contigs_equal"], r


def test_long_regions_on_the_emulated_library():
    _check(_run(sim_util.build_simt("libbreakmer_simt_TESTONLY.so", "all.cpp"))[0])


def test_long_regions_under_address_sanitizer():
    if not os.environ.get("BK_TEST_ASAN"):
        pytest.skip("set BK_TEST_ASAN=1 to build and run the AddressSanitizer library")
    lib = sim_util.build_simt("libbreakmer_simt_asan_TESTONLY.so", "all.cpp",
                              extra=["-O1", "-g", "-DSIMT_ARENA_MALLOC", "-fsanitize=address,undefined"])
    asan_rt = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    rows, err = _run(lib, {"LD_PRELOAD": asan_rt, "ASAN_OPTIONS": "detect_leaks=0:halt_on_error=1",
                           "UBSAN_OPTIONS": "print_stacktrace=1:halt_on_error=1"})
    assert "AddressSanitizer" not in err and "runtime error" not in err, err[-4000:]
    _check(rows)
