"""Cost of the k-mer stage's report (always computed) and of the "normal_kmers" option.

    python tools/kmer_report_bench.py --base-root DIR [--base-tag parent] [--reps 2] [--steps 3] [--chunk 125]
                                      [--c5-regions 2000] [--out-dir profiles]

Writes <out-dir>/r6_kmer_report.md and <out-dir>/r6_kmer_report_bench.json.  Three arms run in separate processes,
alternated --reps times: another commit's tree DIR (its package, and its library built there with
BK_BUILD_TAG=<base-tag>: DIR/breakmer_b200/lib/libbreakmer_b200_<base-tag>.so) with the option off, this build with the
option off, and this build with the option on.  Each
arm runs C2 (500 regions), C3 (500, tumour/normal), C4 (100) and C5 (the first --c5-regions) in calls of --chunk regions
on one handle (bk_compare_kmers_batch, undecoded results), one warm-up step and then --steps timed steps per config, and
reads per step from bk_kernel_times:

  region_kmers ms   device time of the region_kmers family (region_kmer_kernel and region_compact_kernel)
  scan ms           device time of the scan family (it also holds the read grouping's scans)
  launches          region_kmers + scan launches
  gpu ms            sum of the calls' gpu_ms (the whole device pass)

The sample-only tables and contigs of every arm are digested (shard.region_digests) and must agree.  The card's name
and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CONFIGS = ("C2", "C3", "C4", "C5")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def worker(a):
    """one arm: the package under a.root with the library BK_LIB names, option a.option; prints one JSON line"""
    sys.path.insert(0, a.root)
    from breakmer_b200 import _lib, batch, shard, synth
    h = _lib.Handle(0)
    if a.option:
        h.set_option("normal_kmers", 1)
    out = {}
    for cfg in CONFIGS:
        panel = list(synth.config_regions(cfg, n=a.c5_regions if cfg == "C5" else None))
        packs = [batch.PackedBatch(panel[i:i + a.chunk]) for i in range(0, len(panel), a.chunk)]

        def one_step(digest=False):
            gpu = 0.0
            digests = {}
            for pk in packs:
                res = batch.run(h, pk, decode=digest)
                gpu += res.gpu_ms
                if digest:
                    digests.update(shard.region_digests(res, pk))
            return gpu, digests

        _gpu, digests = one_step(digest=True)                       # warm-up (module load, arena growth) and digest
        rows = []
        for _s in range(a.steps):
            h.kernel_times_reset(True)
            t0 = time.perf_counter()
            gpu, _d = one_step()
            wall = time.perf_counter() - t0
            kt = h.kernel_times()
            rows.append(dict(region_kmers_ms=kt["region_kmers"][0], scan_ms=kt["scan"][0],
                             launches=int(kt["region_kmers"][1] + kt["scan"][1]), gpu_ms=gpu, regions_per_s=len(panel) / wall))
        h.kernel_times_reset(False)
        out[cfg] = dict(regions=len(panel), calls=len(packs), steps=rows, digest=shard.digest_of_digests(digests))
    h.close()
    print("RESULT " + json.dumps(out), flush=True)


def run_arm(root, lib, option, a):
    env = dict(os.environ, BK_LIB=lib)
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--root", root, "--option", str(option), "--steps", str(a.steps),
           "--chunk", str(a.chunk), "--c5-regions", str(a.c5_regions)]
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
    if p.returncode != 0 or not line:
        raise RuntimeError("arm %s option %d failed:\n%s" % (lib, option, p.stdout[-2000:] + p.stderr[-4000:]))
    return json.loads(line[0][len("RESULT "):])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--option", type=int, default=0)
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--base-root", required=False)
    ap.add_argument("--base-tag", default="parent")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=125)
    ap.add_argument("--c5-regions", type=int, default=2000)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    if not a.base_root:
        ap.error("--base-root is required")
    base = os.path.abspath(a.base_root)
    lib = os.path.join(ROOT, "breakmer_b200", "lib", "libbreakmer_b200.so")
    arms = {"base off": (base, os.path.join(base, "breakmer_b200", "lib", "libbreakmer_b200_%s.so" % a.base_tag), 0),
            "this off": (ROOT, lib, 0), "this on": (ROOT, lib, 1)}
    res = {"card": card(), "base_tag": a.base_tag, "reps": a.reps, "steps": a.steps, "chunk": a.chunk, "arms": {}}
    runs = {name: [] for name in arms}
    for _rep in range(a.reps):
        for name, (root, lib, option) in arms.items():
            runs[name].append(run_arm(root, lib, option, a))
            print(name, "done", flush=True)
    table = {}
    for cfg in CONFIGS:
        digests = {runs[name][i][cfg]["digest"] for name in arms for i in range(a.reps)}
        assert len(digests) == 1, (cfg, digests)
        table[cfg] = {}
        for name in arms:
            steps = [s for r in runs[name] for s in r[cfg]["steps"]]
            table[cfg][name] = {key: statistics.median(s[key] for s in steps) for key in steps[0]}
            table[cfg][name]["region_kmers_ms_all"] = [round(s["region_kmers_ms"], 4) for s in steps]
            table[cfg][name]["regions"] = runs[name][0][cfg]["regions"]
    res["configs"] = table
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "r6_kmer_report_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = ["# The k-mer stage's report and the \"normal_kmers\" option: cost on C2, C3, C4 and C5", "",
             "Card: %s.  `python tools/kmer_report_bench.py --base-tag %s --reps %d --steps %d --chunk %d`; arms alternated "
             "in separate processes, median over %d steps per arm (after one warm-up step per process).  `base` is the "
             "build tagged %s; `this` is this build with the option off and on." % (
                 res["card"], a.base_tag, a.reps, a.steps, a.chunk, a.reps * a.steps, a.base_tag), "",
             "| config | arm | region_kmers ms/step | scan ms/step | launches/step (region_kmers + scan) | gpu ms/step | "
             "regions/s |", "|---|---|---|---|---|---|---|"]
    for cfg in CONFIGS:
        for name in arms:
            d = table[cfg][name]
            lines.append("| %s | %s | %.3f | %.3f | %d | %.1f | %.0f |" % (cfg, name, d["region_kmers_ms"], d["scan_ms"],
                                                                          d["launches"], d["gpu_ms"], d["regions_per_s"]))
    lines += ["", "All region_kmers samples (ms/step):", ""]
    for cfg in CONFIGS:
        lines.append("- %s: %s" % (cfg, "; ".join("%s %s" % (n, table[cfg][n]["region_kmers_ms_all"]) for n in arms)))
    with open(os.path.join(a.out_dir, "r6_kmer_report.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
