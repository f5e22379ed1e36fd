"""bk_kmer_report and the "normal_kmers" option on the emulated library of tests/sim against the oracle breakdown: a few
golden regions (one with soft-clip k-mers no read holds), a region with soft clips and no reads, one without soft
clips, one left out at upload, and two tumour/normal (C3) regions with the option on and off.  The regions run in a
child process with BK_LIB pointing at the emulator build, as tests/test_simt_rejected_contigs.py does."""
import json
import os
import subprocess
import sys

import sim_util
from conftest import ROOT

CHILD = r"""
import dataclasses, json, sys
import numpy as np
sys.path.insert(0, "tests")
from breakmer_b200 import _lib, batch, shard, synth
from test_gpu_kmer_report import check_normal, check_report, golden_kmer_regions, with_foreign_clips
from test_gpu_long_regions import over_limit_region
golden = [r for r in golden_kmer_regions() if r.k == 15][:3]
base = golden[0]
edge = [dataclasses.replace(base, name="no_reads", reads=[]), dataclasses.replace(base, name="no_clips", sc_records=[]),
        over_limit_region(5000)]
c3 = [synth.config_region("C3", i) for i in (0, 1)]
h = _lib.Handle(0)
rows = []
regs = golden + [with_foreign_clips(golden[1])] + edge
pk = batch.PackedBatch(regs)
out = batch.run(h, pk)
rep = check_report(h, regs, pk, out, skipped=(len(regs) - 1,))
rows.append(dict(not_in_reads=rep[3]["not_in_reads"], no_reads=rep[4], no_clips=rep[5]))
pk = batch.PackedBatch(c3)
off = batch.run(h, pk)
rep_off = check_report(h, c3, pk, off)
h.set_option("normal_kmers", 1)
on = batch.run(h, pk)
h.set_option("normal_kmers", 0)
rep_on = check_report(h, c3, pk, on)
n_normal = check_normal(c3, on, pk)
without = batch.run(h, batch.PackedBatch(c3, with_normal=False))
union = all({**on.sample_only(i), **on.normal_kmers(i)} == without.sample_only(i) for i in range(len(c3)))
rows.append(dict(n_normal=n_normal, in_normal=[r["in_normal"] for r in rep_on], same_report=rep_on == rep_off,
                 same_outputs=shard.region_digests(on, pk) == shard.region_digests(off, pk)
                 and np.array_equal(on.so_mers, off.so_mers) and np.array_equal(on.so_counts, off.so_counts),
                 union=union, off_normal=off.normal is None))
h.close()
print("RESULT " + json.dumps(rows))
"""


def test_kmer_report_on_the_emulated_library():
    lib = sim_util.build_simt("libbreakmer_simt_TESTONLY.so", "all.cpp")
    env = dict(os.environ, BK_LIB=lib, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-c", CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=3600)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and line, out.stdout[-2000:] + out.stderr[-4000:]
    edge, c3 = json.loads(line[0][len("RESULT "):])
    assert edge["not_in_reads"] > 0
    assert edge["no_reads"]["soft_clip"] == edge["no_reads"]["not_in_reads"] > 0
    assert not any(edge["no_clips"].values())
    assert c3["n_normal"] == sum(c3["in_normal"]) > 0
    assert c3["same_report"] and c3["same_outputs"] and c3["union"] and c3["off_normal"]
