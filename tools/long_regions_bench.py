"""Device time of the long assembler (bk_compare_kmers_long, assemble_long_kernel) per region, and the rate of the
anti-diagonal sweep both it and bk_nw_batch use for pairs above 4,095 bases.

    python tools/long_regions_bench.py [--reps N] [--out FILE.json]

Per scenario (one region per call, `reps` calls after one warm-up call): the call's device time (CUDA events around the
whole pass, gpu_ms), the assembler kernel's device time (bk_kernel_times, family "assemble"), check_align calls and DP
cells.  Scenarios:
  5 kb reads at 10x and 30x   nearly every pair is above 4,095 bases, i.e. takes the CTA sweep
  3 kb reads, ~5 kb contig    pairs take the warp DP until the contig passes 4,095 bases, the sweep after
The sweep rate itself is measured on bk_nw_batch pairs that are all above 4,095 bases (nw_long_kernel, family
"nw_batch"): cells = 2 * m * n per pair (both directions).  The card's name and power limit are read in the same run.
Results are printed as one JSON document (and written to --out)."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENARIOS = [
    ("5kb_reads_10x", dict(seed=41, L=12000, cov=10, k=15, e=0.003, event=("del", 300, None), rl=5000)),
    ("5kb_reads_30x", dict(seed=42, L=12000, cov=30, k=15, e=0.003, event=("del", 300, None), rl=5000)),
    ("3kb_reads_growing_contig", dict(seed=22, L=7000, cov=60, k=15, e=0.002, event=("del", 300, None), rl=3000)),
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def region_times(h, region, reps):
    from breakmer_b200 import batch
    pk = batch.PackedBatch([region])
    batch.run(h, pk, long=True)                                    # warm-up: module load, arena growth
    gpu, asm = [], []
    out = None
    for _ in range(reps):
        h.kernel_times_reset(True)
        out = batch.run(h, pk, long=True)
        assert list(out.region_status) == [0], out.region_status
        gpu.append(out.gpu_ms)
        asm.append(h.kernel_times()["assemble"][0])
    h.kernel_times_reset(False)
    ctg = out.contig_records(0)
    return {
        "reads": len(region.reads), "read_len": max(len(x[1]) for x in region.reads),
        "contigs": [len(c["seq"]) for c in ctg], "check_align": out.n_check_align, "dp_cells": out.n_dp_cells,
        "gpu_ms_median": statistics.median(gpu), "gpu_ms_min": min(gpu), "gpu_ms_max": max(gpu),
        "assemble_ms_median": statistics.median(asm),
        "assemble_cells_per_s": 2 * out.n_dp_cells / (statistics.median(asm) * 1e-3),
    }


def sweep_rate(h, m, n, pairs, reps):
    rng = random.Random(7)
    seqs = []
    for _ in range(pairs):
        a = "".join(rng.choice("ACGT") for _ in range(m))
        b = a[m // 3:] + "".join(rng.choice("ACGT") for _ in range(n - (m - m // 3)))
        seqs += [a, b[:n]]
    pa = list(range(0, 2 * pairs, 2))
    pb = list(range(1, 2 * pairs, 2))
    h.nw_batch(seqs, pa, pb)                                       # warm-up
    ms = []
    for _ in range(reps):
        h.kernel_times_reset(True)
        h.nw_batch(seqs, pa, pb)
        ms.append(h.kernel_times()["nw_batch"][0])
    h.kernel_times_reset(False)
    t = statistics.median(ms)
    return {"m": m, "n": n, "pairs": pairs, "ctas": 2 * pairs, "nw_batch_ms_median": t,
            "cells_per_s": 2.0 * m * n * pairs / (t * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from breakmer_b200 import _lib, synth
    res = {"card": card(), "scenarios": {}, "sweep": []}
    h = _lib.Handle(0)
    try:
        for name, kw in SCENARIOS:
            res["scenarios"][name] = region_times(h, synth.make_region(name, **kw), a.reps)
        for m, n, pairs in ((5000, 5000, 1), (5000, 5000, 74), (20000, 20000, 74)):
            res["sweep"].append(sweep_rate(h, m, n, pairs, a.reps))
    finally:
        h.close()
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
