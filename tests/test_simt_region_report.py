"""The per-region report on the emulated library of tests/sim against the oracle: the counters of a few golden regions,
and one call with the "long_regions" option where a region with 4,500-base reads is routed to the long assembler.  The
regions run in a child process with BK_LIB pointing at the emulator build, as tests/test_simt_long_inline.py does."""
import json
import os
import subprocess
import sys

import sim_util
from conftest import ROOT

CHILD = r"""
import json, sys
import numpy as np
sys.path.insert(0, "tests")
from conftest import golden
from breakmer_b200 import _lib, batch, synth
from test_gpu_long_regions import LONG_READ_REGIONS
from test_gpu_region_report import COUNTERS, oracle_report
cases = golden("assembly_golden.json")["cases"]
regions = []
for c in cases[:4]:
    kw = dict(c["kwargs"]); kw["event"] = tuple(kw["event"])
    if kw["k"] == 15:
        regions.append(synth.make_region(c["name"], **kw))
import dataclasses
# the same regions with every contig rejected: for support (rc_thresh above any count), for length (read_len 10,000)
calls = [(regions, 0, None), ([dataclasses.replace(r, name=r.name + "_s", rc_thresh=10 ** 6) for r in regions[:2]], 0, None),
         ([dataclasses.replace(r, name=r.name + "_l") for r in regions[:2]], 0, 10000),
         ([synth.config_region("C2", 1), synth.make_region("lr0", **dict(LONG_READ_REGIONS)["lr0"])], 1, None)]
h = _lib.Handle(0)
rows = []
for regs, long_regions, read_len in calls:
    h.set_option("long_regions", long_regions)
    pk = batch.PackedBatch(regs)
    if read_len:
        pk.read_len = np.array([read_len] * len(regs) + [0], dtype=np.int32)
    out = batch.run(h, pk)
    rep = batch.region_report(h)
    for i, (r, row) in enumerate(zip(regs, rep)):
        ctgs, exp = oracle_report(r, read_len)
        rows.append(dict(name=r.name, row=row, expected=exp, n_contigs=int(out.ctg_reg_off[i + 1] - out.ctg_reg_off[i]),
                         oracle_contigs=len(ctgs), contigs_equal=out.contig_records(i) == ctgs))
    assert sum(row["check_align"] for row in rep) == out.n_check_align
h.close()
print("RESULT " + json.dumps(rows))
"""


def test_region_report_on_the_emulated_library():
    env = dict(os.environ, BK_LIB=sim_util.build_simt("libbreakmer_simt_TESTONLY.so", "all.cpp"), PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-c", CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=2400)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and line, out.stdout[-2000:] + out.stderr[-4000:]
    rows = json.loads(line[0][len("RESULT "):])
    assert len(rows) >= 5 and rows[-1]["name"] == "lr0"
    assert all(r["row"]["rejected_support"] > 0 for r in rows if r["name"].endswith("_s"))
    assert all(r["row"]["rejected_length"] > 0 for r in rows if r["name"].endswith("_l"))
    for r in rows:
        row = r["row"]
        assert r["contigs_equal"] and r["n_contigs"] == r["oracle_contigs"], r
        assert {k: row[k] for k in r["expected"]} == r["expected"], r
        assert row["grown"] == r["n_contigs"] + row["rejected_support"] + row["rejected_length"], r
        assert row["reason"] == "ok", r
        long = r["name"] == "lr0"
        assert row["pass"] == ("long" if long else "batched"), r
        assert row["first_reason"] == ("read_too_long" if long else "ok"), r
