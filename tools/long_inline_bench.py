"""Cost of the "long_regions" option of the batched entries (long regions assembled in the same device pass).

    python tools/long_inline_bench.py [--reps 3] [--chunk 50] [--inflight 8] [--out-dir profiles]

Writes <out-dir>/r4_long_inline.md and <out-dir>/r4_long_inline_bench.json.  Three measurements, all in one process:

  nothing_long   the 500-region C2 panel in chunks of --chunk regions through shard.DevicePipeline with --inflight
                 batches in flight, option off and on alternated --reps times: regions/s of the pipelined panel,
                 sequential ms per call (one chunk at a time, submit + wait, median), and a digest of every region's
                 results (shard.region_digests), which must be the same for both settings
  one_vs_two     the same panel plus three long regions (reads of 4,500 and 6,000 bases, and a contig that grows past
                 4,095 bases from 3,000-base reads) spread over the chunks: a default pass followed by
                 bk_compare_kmers_long on the regions it reported (packing them again included), against one pass with
                 the option on; host wall time and the sum of the calls' gpu_ms
  memory         device memory one handle holds after one chunk of the panel, option off and on: the drop of the
                 device's free memory (cudaMemGetInfo, device-wide, so work of other processes on the same device
                 shows up in it), beside the long kernel's scratch computed from its sizes

The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LONG = [("lr0", dict(seed=11, L=10000, cov=6, k=15, e=0.003, event=("del", 300, None), rl=4500)),
        ("lr2", dict(seed=13, L=13000, cov=5, k=15, e=0.003, event=("tdup", 400), rl=6000)),
        ("grow", dict(seed=22, L=7000, cov=60, k=15, e=0.002, event=("del", 300, None), rl=3000))]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def long_scratch_bytes_per_cta(read_cap=4096):
    """long_assembly_scratch (pipeline_impl.cuh) for AsmCapLong: CAP = 65,536"""
    cap, buf, kcap = 65536, 3 * 65536, 2 * 65536
    return (buf + 4 * buf * 4 + 2 * 4 * kcap * 4 + cap * 8 + (cap + 1) * 4 + 2 * 4096 * 8 + 2049 * 8 + 160 * 1024 +
            read_cap + cap + 9 * (cap + 1) * 4)


def pipelined(pipe, packs):
    """all chunks through the pipeline; -> (wall s, [BatchOutput])"""
    outs = []
    t0 = time.perf_counter()
    for pk in packs:
        if pipe.full():
            outs.append(pipe.pop()[0])
        pipe.submit(pk)
    while pipe.pending():
        outs.append(pipe.pop()[0])
    return time.perf_counter() - t0, outs


def sequential_ms(pipe, packs):
    ms = []
    for pk in packs:
        t0 = time.perf_counter()
        pipe.submit(pk)
        pipe.pop()
        ms.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(ms)


def digest(outs, packs):
    from breakmer_b200 import shard
    d = {}
    for out, pk in zip(outs, packs):
        d.update(shard.region_digests(out, pk))
    return shard.digest_of_digests(d)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=50)
    ap.add_argument("--inflight", type=int, default=8)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    import torch
    from breakmer_b200 import _lib, batch, shard, synth
    res = {"card": card(), "chunk": a.chunk, "inflight": a.inflight, "reps": a.reps}
    panel = list(synth.config_regions("C2"))
    chunks = [panel[i:i + a.chunk] for i in range(0, len(panel), a.chunk)]
    packs = [batch.PackedBatch(c) for c in chunks]
    pipes = {on: shard.DevicePipeline(0, inflight=a.inflight, long_regions=on) for on in (False, True)}
    try:
        # ---- nothing long: the option's cost ----
        for on in (False, True):                                      # warm-up: module load, arena growth
            pipelined(pipes[on], packs)
        rows = []
        for rep in range(a.reps):
            for on in (False, True):
                wall, outs = pipelined(pipes[on], packs)
                assert all(not any(o.region_status) for o in outs)
                rows.append({"rep": rep, "long_regions": on, "regions_per_s": len(panel) / wall,
                             "sequential_ms_per_call": sequential_ms(pipes[on], packs), "digest": digest(outs, packs)})
        res["nothing_long"] = rows
        # ---- one pass against two ----
        longs = [synth.make_region(n, **kw) for n, kw in LONG]
        mixed = [c + ([longs[i]] if i < len(longs) else []) for i, c in enumerate(chunks)]
        mpacks = [batch.PackedBatch(c) for c in mixed]
        h = pipes[False].handles[0]
        flows = []
        for rep in range(a.reps + 1):                                  # the first repeat is a warm-up
            t0 = time.perf_counter()
            _wall, outs = pipelined(pipes[False], mpacks)
            redo = [r for c, o in zip(mixed, outs) for i, r in enumerate(c) if o.region_status[i] != 0]
            lo = batch.run(h, batch.PackedBatch(redo), long=True)
            two_wall = time.perf_counter() - t0
            two_gpu = sum(o.gpu_ms for o in outs) + lo.gpu_ms
            assert sorted(r.name for r in redo) == sorted(n for n, _ in LONG) and not any(lo.region_status)
            t0 = time.perf_counter()
            _wall, outs1 = pipelined(pipes[True], mpacks)
            one_wall = time.perf_counter() - t0
            assert all(not any(o.region_status) for o in outs1)
            if rep:
                flows.append({"rep": rep, "two_pass_wall_ms": 1e3 * two_wall, "two_pass_gpu_ms": two_gpu,
                              "one_pass_wall_ms": 1e3 * one_wall, "one_pass_gpu_ms": sum(o.gpu_ms for o in outs1)})
        res["one_vs_two"] = flows
    finally:
        for p in pipes.values():
            p.close()
    # ---- device memory per handle ----
    mem = {}
    for on in (False, True):
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        h = _lib.Handle(0)
        if on:
            h.set_option("long_regions", 1)
        batch.run(h, packs[0])
        free1 = torch.cuda.mem_get_info(0)[0]
        h.close()
        mem["on" if on else "off"] = free0 - free1
    res["memory_bytes_per_handle"] = mem
    res["long_scratch_bytes_per_cta"] = long_scratch_bytes_per_cta()
    res["card_after"] = card()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "r4_long_inline_bench.json"), "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")
    with open(os.path.join(a.out_dir, "r4_long_inline.md"), "w") as f:
        f.write(report(res))
    print(json.dumps(res, indent=1))


def report(res):
    L = ["# The \"long_regions\" option: cost and one pass against two", "",
         "Card: %s (read before the run; after: %s).  Written by `tools/long_inline_bench.py` from one run; the numbers are"
         " in `r4_long_inline_bench.json`." % (res["card"], res["card_after"]), "",
         "## Nothing long: the 500-region C2 panel, chunks of %d, %d in flight" % (res["chunk"], res["inflight"]), "",
         "| repeat | long_regions | regions/s | sequential ms per call | digest |", "|---|---|---|---|---|"]
    for r in res["nothing_long"]:
        L.append("| %d | %d | %.0f | %.2f | `%s` |" % (r["rep"], r["long_regions"], r["regions_per_s"], r["sequential_ms_per_call"],
                                                       r["digest"][:12]))
    for on in (False, True):
        v = [r["regions_per_s"] for r in res["nothing_long"] if r["long_regions"] == on]
        s = [r["sequential_ms_per_call"] for r in res["nothing_long"] if r["long_regions"] == on]
        L.append("")
        L.append("long_regions=%d: regions/s %.0f .. %.0f, sequential ms per call %.2f .. %.2f" % (on, min(v), max(v), min(s), max(s)))
    L += ["", "Digests equal for both settings: %s" % (len({r["digest"] for r in res["nothing_long"]}) == 1), "",
          "## One pass against two: the panel plus three long regions", "",
          "| repeat | two passes wall ms | two passes gpu_ms | one pass wall ms | one pass gpu_ms |", "|---|---|---|---|---|"]
    for r in res["one_vs_two"]:
        L.append("| %d | %.1f | %.1f | %.1f | %.1f |" % (r["rep"], r["two_pass_wall_ms"], r["two_pass_gpu_ms"], r["one_pass_wall_ms"],
                                                     r["one_pass_gpu_ms"]))
    m = res["memory_bytes_per_handle"]
    L += ["", "gpu_ms is the sum of the calls' device time (CUDA events around each pass); the calls overlap, so it is"
          " not a wall time.", "",
          "## Device memory per handle (after one chunk of the panel)", "",
          "option off: %.1f MB, option on: %.1f MB (drop of the device's free memory).  The long kernel's scratch is %.1f MB"
          " per CTA; with nothing routed at upload the grid is 4 CTAs." % (m["off"] / 1e6, m["on"] / 1e6, res["long_scratch_bytes_per_cta"] / 1e6), ""]
    return "\n".join(L)


if __name__ == "__main__":
    main()
