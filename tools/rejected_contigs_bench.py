"""Cost of the "rejected_contigs" option (the contigs the acceptance test drops, returned with the result).

    python tools/rejected_contigs_bench.py [--reps 3] [--chunk 125] [--inflight 4] [--c5-regions 2000] [--out-dir profiles]

Writes <out-dir>/r5_rejected_contigs.md and <out-dir>/r5_rejected_contigs_bench.json.  For each of C2 (500 regions),
C4 (100) and C5 (the first --c5-regions), one step is the whole panel in chunks of --chunk regions through
shard.DevicePipeline with --inflight batches in flight (decoded results, as the Python drop-ins read them).  The option
off and on are alternated --reps times after one warm-up step each, and per setting the table gives:

  regions/s        regions of a step over its host wall time (median of the repeats)
  contigs          accepted contigs per step, and rejected ones (only with the option on)
  result bytes     bytes of the contig payload per step (sequence, kmer_locs, both count vectors, reads, k-mer tuples):
                   accepted, and rejected on top of them
  arena retry      whether the assembler ran again with an 8x larger output arena in any call of a step: the calls'
                   assemble launches (bk_kernel_times, counted in a separate untimed step) above one per call
  digest           shard.region_digests of every region, which must be the same for both settings

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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def step(pipe, packs):
    """the whole panel through the pipeline -> (wall s, [BatchOutput] in chunk order)"""
    outs = []
    t0 = time.perf_counter()
    for pk in packs:
        if pipe.full():
            outs.append(pipe.pop()[0])
        pipe.submit(pk)
    while pipe.pending():
        outs.append(pipe.pop()[0])
    return time.perf_counter() - t0, outs


def payload_bytes(out, c0, c1):
    """bytes of contigs [c0, c1) of a BatchOutput: sequence (1 + 4 per base with kmer_locs), count vectors (2 x 4),
    reads (4), k-mer tuples (8 + 4 x 4)"""
    if c1 <= c0:
        return 0
    return int(5 * out.seq_off[c0:c1, 1].sum() + 8 * out.cnt_off[c0:c1, 1].sum() + 4 * out.reads_off[c0:c1, 1].sum() +
               24 * out.kmers_off[c0:c1, 1].sum())


def summary(outs, packs):
    from breakmer_b200 import shard
    acc = rej = acc_b = rej_b = 0
    digests = {}
    for out, pk in zip(outs, packs):
        assert not out.region_status.any()
        n_rej = 0 if out.rej_reason is None else len(out.rej_reason)
        acc += out.n_contigs
        rej += n_rej
        acc_b += payload_bytes(out, 0, out.n_contigs)
        rej_b += payload_bytes(out, out.n_contigs, out.n_contigs + n_rej)
        digests.update(shard.region_digests(out, pk))
    return dict(accepted=acc, rejected=rej, accepted_bytes=acc_b, rejected_bytes=rej_b,
                digest=shard.digest_of_digests(digests))


def retry_fired(pipe, packs):
    """whether any call of one (untimed) step launched the assembler more than once"""
    for h in pipe.handles:
        h.kernel_times_reset(True)
    step(pipe, packs)
    launches = sum(h.kernel_times()["assemble"][1] for h in pipe.handles)
    for h in pipe.handles:
        h.kernel_times_reset(False)
    return launches > len(packs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=125)
    ap.add_argument("--inflight", type=int, default=4)
    ap.add_argument("--c5-regions", type=int, default=2000)
    ap.add_argument("--configs", default="C2,C4,C5")
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    from breakmer_b200 import batch, shard, synth
    res = {"card": card(), "chunk": a.chunk, "inflight": a.inflight, "reps": a.reps, "configs": {}}
    pipes = {on: shard.DevicePipeline(0, inflight=a.inflight, rejected_contigs=on) for on in (False, True)}
    try:
        for cfg in a.configs.split(","):
            panel = list(synth.config_regions(cfg, n=a.c5_regions if cfg == "C5" else None))
            packs = [batch.PackedBatch(panel[i:i + a.chunk]) for i in range(0, len(panel), a.chunk)]
            for on in (False, True):                                  # warm-up: module load, arena growth
                step(pipes[on], packs)
            rows = {False: [], True: []}
            sums = {}
            for _rep in range(a.reps):
                for on in (False, True):
                    wall, outs = step(pipes[on], packs)
                    rows[on].append(len(panel) / wall)
                    sums[on] = summary(outs, packs)
            assert sums[False]["digest"] == sums[True]["digest"], cfg
            assert sums[False]["rejected"] == 0
            res["configs"][cfg] = {
                "regions": len(panel), "calls": len(packs),
                **{("on" if on else "off"): dict(regions_per_s=statistics.median(rows[on]), regions_per_s_all=rows[on],
                                                 retry=retry_fired(pipes[on], packs), **sums[on]) for on in (False, True)}}
            print(cfg, json.dumps(res["configs"][cfg]), flush=True)
    finally:
        for p in pipes.values():
            p.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "r5_rejected_contigs_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = ["# The \"rejected_contigs\" option: cost on C2, C4 and C5", "",
             "Card: %s.  `python tools/rejected_contigs_bench.py --reps %d --chunk %d --inflight %d`; one step is the "
             "panel in chunks of %d regions through `shard.DevicePipeline` (%d batches in flight, decoded results), option "
             "off and on alternated, median of %d repeats after a warm-up step each." % (res["card"], a.reps, a.chunk, a.inflight,
                                                                                         a.chunk, a.inflight, a.reps), "",
             "| config | regions | regions/s off | regions/s on | on / off | accepted contigs | rejected contigs | "
             "accepted bytes | rejected bytes | arena retry off / on | digests equal |",
             "|---|---|---|---|---|---|---|---|---|---|---|"]
    for cfg, d in res["configs"].items():
        off, on = d["off"], d["on"]
        lines.append("| %s | %d | %.0f | %.0f | %.3f | %d | %d | %d | %d | %s / %s | %s |" % (
            cfg, d["regions"], off["regions_per_s"], on["regions_per_s"], on["regions_per_s"] / off["regions_per_s"],
            on["accepted"], on["rejected"], on["accepted_bytes"], on["rejected_bytes"], off["retry"], on["retry"],
            off["digest"] == on["digest"]))
    with open(os.path.join(a.out_dir, "r5_rejected_contigs.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
