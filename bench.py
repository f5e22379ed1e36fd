#!/usr/bin/env python
"""Benchmark of the BreaKmer per-target k-mer assembly hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2] [--dump-outputs DIR]

A "step" is one pass of the whole hot path (target.compare_kmers: k-mer counting, sample-only selection, read
grouping, init_assembly) over the workload's regions.  The default workload is BASELINE.json configs[1], the
500-target gene panel (k=15).

Multi-GPU (one process per GPU under torchrun): the workload's regions are PARTITIONED BY REGION --
`shard.assign_lpt` on a static cost model, distinct regions on every rank, no data-path collective -- and the
per-region results are gathered on the host in target-name order (`shard.gather_by_name`) and compared, by digest,
with the same regions run on rank 0's GPU alone.
  * C2 / C3 / C4 scale weakly: N ranks share a panel of N x 500 (N x 100) distinct regions;
  * C5 scales strongly: the 20,000 exome-scale regions are split over the N ranks, in calls of <= 2,500 regions.
The default line also carries `c5_strong` and `c3_sharded`: the same measurement for BASELINE.json configs 5 and 3.

One JSON line is printed by rank 0.  `value` is whole-job regions/s with the inputs already resident in HBM; `e2e`
is the same metric through the C-ABI calls bk_batch_submit / bk_batch_wait with HOST buffers (host->device copies and
the result read-back inside the timed region).  Each rank drives its GPU from ONE host thread.

--dump-outputs DIR writes what the last timed step of `value` returned as DIR/<name>.npy (see result_arrays).  The
inputs are generated from fixed seeds, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name -> (description, regions per GPU (weak) or in total (strong), scaling)
WORKLOADS = {
    "C1": ("C1: single synthetic 20 kb target region, 100 bp reads at 200x, planted 1.5 kb deletion, k=15", 1, "weak"),
    "C2": ("C2: 500-target gene panel, synthetic tumor reads with planted indels/inversions/tandem dups, k=15", 500, "weak"),
    "C3": ("C3: tumor/normal pair, 500 targets with normal-k-mer subtraction, k=15", 500, "weak"),
    "C4": ("C4: 2000x amplicon-depth panel, 100 amplicons, k=21", 100, "weak"),
    "C5": ("C5: exome-scale 20,000 target regions with planted translocations, k=15, region-sharded", 20000, "strong"),
}
METRIC = "target_regions_assembled_per_sec"
UNIT = "regions/s"
CALL_REGIONS = 2500          # regions per C-ABI call
DUMP_LIMIT = 60 << 20        # bytes of --dump-outputs array data; with the .npy headers the files stay under 64 MB


def config_dict(workload, world, regions_override=0):
    """The `config` object of the JSON line -- identical in both arms."""
    desc, n, scaling = WORKLOADS[workload]
    if regions_override:
        n = regions_override
    total = n * world if scaling == "weak" else n
    return {"workload": desc, "regions_total": total, "regions_per_gpu": total / float(world), "scaling": scaling,
            "k": 21 if workload == "C4" else 15, "rc_thresh": 2,
            "sharding": "by region: C-ABI calls of similar static cost (shard.assign_lpt), every call of a step run by exactly one "
                        "rank, host-side gather by target name; no data-path collective"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def _sample(self):
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM))
            mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
            for bit, name in self.REASONS.items():
                if mask & bit and name != "gpu_idle":
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        # NVML queries contend with kernel launches of every process on the box: keep them sparse.  The first two come
        # early so that a short timed region (few --steps) is still sampled under load.
        for pause in (0.03, 0.09):
            if self._stop_evt.wait(pause):
                return
            self._sample()
        while not self._stop_evt.wait(0.25):
            self._sample()

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        late = False
        if self.ok and not self.samples:     # a timed region shorter than 30 ms: one sample right behind it
            self._sample()
            late = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        out = {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if late:
            out["sampled"] = "right after the timed region (it was shorter than the first sampling delay)"
        return out


# ---------------------------------------------------------------------------------
# CPU side (the oracle; used only as the reported baseline / reference arm)
# ---------------------------------------------------------------------------------
def cpu_region(region):
    """The reference's CPU path for one region, as restated by the oracle: pure-Python
    k-mer counting + set algebra + init_assembly with the pure-Python olc.nw loop
    (that loop is what the reference itself executes in CPython)."""
    from oracle import assembler_py, kmers_py, nw_py
    normal = [x[1] for x in region.normal_reads] if region.normal_reads else None
    _r, _c, _s, only = kmers_py.sample_only(region.ref_fwd, [x[1] for x in region.reads],
                                            [x[1] for x in region.sc_records], region.k, normal)
    ctg = assembler_py.init_assembly(only, region.reads, region.k, region.rc_thresh, region.read_len, nw=nw_py.nw)
    return len(only), len(ctg)


def _cpu_region_by_index(args):
    workload, idx = args
    from breakmer_b200 import synth
    t0 = time.time()
    n_only, n_ctg = cpu_region(synth.config_region(workload, idx))
    return n_only, n_ctg, time.time() - t0


def cpu_c_nw_single(regions, max_regions=40):
    """Context only: the same oracle with its C restatement of olc.nw (what a compiled single-core port of the
    reference would roughly do)."""
    from oracle import assembler_py, kmers_py
    t0 = time.time()
    done = 0
    for r in regions[:max_regions]:
        normal = [x[1] for x in r.normal_reads] if r.normal_reads else None
        _r, _c, _s, only = kmers_py.sample_only(r.ref_fwd, [x[1] for x in r.reads], [x[1] for x in r.sc_records], r.k, normal)
        assembler_py.init_assembly(only, r.reads, r.k, r.rc_thresh, r.read_len)
        done += 1
    return done / (time.time() - t0)


def cpu_baseline_single(workload, regions, budget_s=20.0, max_regions=8):
    t0 = time.time()
    done = 0
    kmers = 0
    for r in regions[:max_regions]:
        n_only, _ = cpu_region(r)
        kmers += n_only
        done += 1
        if time.time() - t0 >= budget_s:
            break
    dt = time.time() - t0
    return {"value": done / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "first %d regions of %s, single process, regions serial (as sv_processor.py:185), "
                      "oracle port with the pure-Python olc.nw loop; jellyfish absent so the k-mer stage is the "
                      "oracle's dict counter (under-states the reference)" % (done, workload),
            "seconds": round(dt, 2), "sample_only_kmers_per_s": kmers / dt}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    cfg = config_dict(args.workload, args.gpus, args.regions)
    n_total = cfg["regions_total"]
    per_step = min(2 * cores, n_total)        # two regions per core per step keeps the pool busy past the stragglers
    budget = float(os.environ.get("BK_REF_BUDGET_S", "170"))
    ctx = mp.get_context("fork")
    t_start = time.time()
    timed_regions = 0
    timed_s = 0.0
    timed_kmers = 0
    steps_done = 0
    with ctx.Pool(cores) as pool:
        nxt = 0
        for step in range(args.warmup + args.steps):
            idx = [(args.workload, (nxt + j) % n_total) for j in range(per_step)]
            nxt += per_step
            t0 = time.time()
            res = pool.map(_cpu_region_by_index, idx, chunksize=1)
            dt = time.time() - t0
            if step >= args.warmup:
                timed_regions += len(res)
                timed_s += dt
                timed_kmers += sum(r[0] for r in res)
                steps_done += 1
            if time.time() - t_start > budget and steps_done >= 1:
                break
    value = timed_regions / timed_s if timed_s > 0 else 0.0
    sample = ("each step is a bounded sample of the workload: %d regions (two per host core, dynamic pool), %d of %d timed "
              "steps completed within the %.0f s budget; oracle port of the reference's CPython path over multiprocessing" %
              (per_step, steps_done, args.steps, budget))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * timed_s / max(1, steps_done), "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "sample_only_kmers_per_s": timed_kmers / timed_s if timed_s > 0 else 0.0,
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------
class Dist:
    """torch.distributed plumbing: barrier + scalar reductions (NCCL) and the host-side object gather."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch = torch
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit("WORLD_SIZE (%d) != --gpus (%d)" % (self.world, args.gpus))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            # every rank keeps to its own share of the host cores (its one driving thread, the ingest threads of the
            # from-files leg): ranks do not migrate onto each other's cores
            try:
                cores = sorted(os.sched_getaffinity(0))
                per = max(1, len(cores) // self.world)
                mine = cores[self.local_rank * per:(self.local_rank + 1) * per]
                if mine and not os.environ.get("BK_BENCH_NO_PIN"):
                    os.sched_setaffinity(0, mine)
            except (AttributeError, OSError):
                pass
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _reduce(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX)

    def sum(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM)

    def gather_floats(self, x):
        if self.world == 1:
            return [x]
        t = self.torch.zeros(self.world, dtype=self.torch.float64, device="cuda")
        t[self.rank] = x
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


class ShardRun:
    """One workload, sharded by region over the ranks.

    The regions are cut into calls of at most `call_regions` by `shard.assign_lpt` on the static cost model (calls of
    similar cost; every rank derives the same calls, no communication).  With one rank the calls simply cycle.  With
    several ranks the calls of every pass are handed out through a host-side work queue -- an atomic counter in the
    torch.distributed store, the only cross-rank traffic besides the final host-side gather: a rank takes the next call
    when it has a free slot, so ranks whose calls turn out slower (per-region cost is only weakly predictable, and a
    500-region call's time is not proportional to its DP work) simply take fewer.  `--static-shards` pins call c to
    rank c % N instead (the plain LPT partition)."""

    def __init__(self, D, workload, total, inflight, spec_width=0, call_regions=CALL_REGIONS, replicate=False, static=False):
        from breakmer_b200 import _lib, batch, shard, synth
        self.D = D
        self.workload = workload
        self.total = total
        self.static = static or D.world == 1
        t0 = time.time()
        self.regions = [synth.config_region(workload, i) for i in range(total)]
        self.costs = [shard.region_cost(r) for r in self.regions]
        if total < D.world:
            raise SystemExit("bench.py: %d regions cannot be sharded over %d ranks" % (total, D.world))
        n_calls = max(D.world, (total + call_regions - 1) // call_regions)
        self.calls = [c for c in shard.assign_lpt(self.costs, n_calls) if c]
        if replicate:                               # diagnostic: every call is call 0 (system effects only)
            self.calls = [self.calls[0]] * len(self.calls)
        nc = len(self.calls)
        # static: this rank only ever runs its own calls; dynamic: any call may come its way
        self.mine = [c for c in range(nc) if c % D.world == D.rank] if self.static else list(range(nc))
        self.packed = {c: batch.PackedBatch([self.regions[i] for i in self.calls[c]]).pin() for c in self.mine}
        self.gen_s = time.time() - t0
        nm = max(1, len(self.mine))
        reps = (max(1, inflight) + nm - 1) // nm
        if not self.static:
            reps = max(2, reps)                     # a rank may draw the same call twice in a row
        self.inflight = max(1, inflight)
        self.n_handles = nm * reps                  # every call resident on the same number of handles
        self.handles = [_lib.Handle(D.local_rank) for _ in range(self.n_handles)]
        for h in self.handles:
            h.set_option("blocking_sync", 1)        # the single host thread of this rank sleeps while it waits
            if spec_width:
                h.set_option("spec_width", spec_width)
        self.handle_call = [self.mine[j % nm] for j in range(self.n_handles)] if self.mine else []
        self.k = next(iter(self.packed.values())).k if self.packed else 15
        self.last = {}

    def warm(self, resident, w=3):
        """untimed: every handle runs at least three calls of its own (with host buffers: every call that may come its
        way, so its arenas have their final size), then `w` passes the way the timed region runs them"""
        from breakmer_b200 import batch
        nm = max(1, len(self.mine))
        for rep in range(3 if resident else max(3, nm if not self.static else 3)):
            for j, h in enumerate(self.handles):
                batch.submit(h, None if resident else self.packed[self.mine[(j + rep) % nm]])
            for h in self.handles:
                batch.wait(h, decode=False)
        self.run_pass(max(3, w), resident)

    def upload(self):
        from breakmer_b200 import batch
        for j, h in enumerate(self.handles):
            batch.upload(h, self.packed[self.handle_call[j]])

    def _call_of(self, t):
        """item t -> call: pass t // nc runs every call once; the order rotates by one per pass so that ranks drawing
        items in lockstep do not keep drawing the same call"""
        nc = len(self.calls)
        return (t + t // nc) % nc

    def _items(self, steps):
        """the (pass, call) items of `steps` passes this rank runs, in order: its own calls (static) or whatever the
        cross-rank queue hands out (dynamic)"""
        nc = len(self.calls)
        n_items = steps * nc
        if self.static:
            for t in range(n_items):
                if self._call_of(t) in self.packed:
                    yield t
            return
        from breakmer_b200 import shard
        queue = shard.CallQueue(self.workload, n_items, self.D.world)
        starve = os.environ.get("BK_BENCH_TEST_STARVE_RANK")       # test hook: that rank takes nothing of the last pass
        t = 0
        while True:
            if starve is not None and int(starve) == self.D.rank and t >= n_items - 2 * nc:
                return
            t = queue.take()
            if t is None:
                return
            yield t

    def run_pass(self, steps, resident, flush=None):
        """steps passes over the calls from ONE host thread: bk_batch_submit keeps up to n_handles batches queued on the
        device, bk_batch_wait collects them in submission order.  Keeps the results of the last pass per call."""
        from breakmer_b200 import batch
        nc = len(self.calls)
        if nc == 0:
            return
        n_items = steps * nc
        t_sub = t_wait = 0.0
        fly = []                                    # (handle index, item) in submission order
        busy = set()
        done = 0

        def drain_one():
            nonlocal t_wait, done
            j, t = fly.pop(0)
            t0 = time.perf_counter()
            res = batch.wait(self.handles[j], decode=False)
            t_wait += time.perf_counter() - t0
            busy.discard(j)
            done += 1
            if t >= n_items - nc:                   # the last pass: what the sharding check looks at
                self.last[self._call_of(t)] = (j, res)

        self.last = {}
        for t in self._items(steps):
            c = self._call_of(t)
            cand = [j for j in range(self.n_handles) if (not resident or self.handle_call[j] == c)]
            while len(fly) >= self.inflight:
                drain_one()
            while True:
                free = [j for j in cand if j not in busy]
                if free:
                    break
                drain_one()
            j = free[0]
            if flush is not None and self.n_handles == 1:
                flush.zero_()                       # sequential mode: flush L2 between timed steps
            t0 = time.perf_counter()
            batch.submit(self.handles[j], None if resident else self.packed[c])
            t_sub += time.perf_counter() - t0
            fly.append((j, t))
            busy.add(j)
        while fly:
            drain_one()
        post = [float(r.host_post_ms) for _j, r in self.last.values()]
        self.items_run = done
        self.host_ms = {"submit_ms_per_call": 1000.0 * t_sub / max(1, done), "wait_ms_per_call": 1000.0 * t_wait / max(1, done),
                        "of_which_result_tables_ms": sum(post) / max(1, len(post)), "calls_run_by_this_rank": done,
                        "note": "host thread: time inside bk_batch_submit (copies + launches) and bk_batch_wait (mostly blocked on the device)"}

    def timed(self, steps, resident, flush=None):
        """-> (device seconds by CUDA events, wall seconds), both max over ranks"""
        torch = self.D.torch
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        self.D.barrier()
        t0 = time.time()
        ev0.record()
        self.run_pass(steps, resident, flush)
        torch.cuda.synchronize()
        ev1.record()
        ev1.synchronize()
        wall = time.time() - t0
        self.D.barrier()
        self.last_local_dev_s = ev0.elapsed_time(ev1) / 1000.0
        return self.D.max(self.last_local_dev_s), self.D.max(wall)

    def counters(self):
        """work counters of the calls of the last pass this rank ran (summed over ranks: one whole pass)"""
        tot = {"contigs": 0, "check_align": 0, "dp_cells": 0, "kmer_occ": 0, "sorted": 0, "sample_only": 0}
        for c, (_j, res) in self.last.items():
            tot["contigs"] += int(res.n_contigs); tot["check_align"] += int(res.n_check_align)
            tot["dp_cells"] += int(res.n_dp_cells); tot["kmer_occ"] += int(res.n_kmer_occurrences)
            tot["sorted"] += int(res.n_sorted_keys); tot["sample_only"] += int(res.so_off[res.n_regions])
        return tot

    def check_against_single_gpu(self):
        """Host-side gather of the per-region result digests in target-name order (from whichever rank ran each call of
        the last pass); rank 0 runs ALL regions on its own GPU and compares.  Returns (ok, digest of digests, regions) on
        rank 0, (None, None, n) elsewhere."""
        from breakmer_b200 import batch, shard
        local = {}
        for c, (_j, res) in sorted(self.last.items()):
            out = batch.BatchOutput(res, self.packed[c])
            local.update(shard.region_digests(out, self.packed[c]))
        merged = shard.gather_by_name(local, self.D.rank, self.D.world)
        ok, dig = None, None
        if self.D.rank == 0:
            single = {}
            if self.D.world == 1 and len(self.calls) == 1:
                single.update(local)              # one rank, one call: it IS the single-GPU run
            else:
                for c in shard.chunk_indices(range(self.total), CALL_REGIONS):
                    pk = batch.PackedBatch([self.regions[i] for i in c])
                    single.update(shard.region_digests(batch.run(self.handles[0], pk), pk))
            ok = bool(merged == dict(sorted(single.items())) and list(merged) == sorted(r.name for r in self.regions))
            dig = shard.digest_of_digests(merged)
        return ok, dig, len(local)

    def close(self):
        for h in self.handles:
            h.close()
        self.handles = []


def sharded_summary(D, workload, total, args, steps):
    """value / e2e / sharding check of one more workload (the c5_strong and c3_sharded keys of the line)."""
    # (C5 calls have long tails -- 2 % of the regions carry all the assembly work -- so more of them are kept in flight)
    run = ShardRun(D, workload, total, max(args.inflight, 8) if workload == "C5" else args.inflight, args.spec_width,
                   static=args.static_shards)
    try:
        run.upload()
        run.warm(True)
        dev_s, _ = run.timed(steps, True)
        by_rank = [round(v, 3) for v in D.gather_floats(1000.0 * run.last_local_dev_s / steps)]
        run.warm(False)
        _, e2e_s = run.timed(steps, False)
        cnt = run.counters()
        ok, dig, _n = run.check_against_single_gpu()
        desc, _n0, scaling = WORKLOADS[workload]
        return {"workload": desc, "regions_total": total, "scaling": scaling, "steps": steps,
                "value": total * steps / dev_s, "unit": UNIT, "ms_per_pass": 1000.0 * dev_s / steps,
                "e2e": {"value": total * steps / e2e_s, "unit": UNIT, "ms_per_pass": 1000.0 * e2e_s / steps},
                "sample_only_kmers_per_s": D.sum(float(cnt["sample_only"])) * steps / dev_s,
                "dp_cells_per_pass": int(D.sum(float(cnt["dp_cells"]))),
                "calls_per_pass": len(run.calls), "regions_per_call": [len(c) for c in run.calls][:16],
                "calls_run_by_rank": [int(v) for v in D.gather_floats(float(run.items_run))],
                "assignment": "static (call c on rank c % N)" if run.static else "dynamic (host-side queue over the ranks)",
                "device_ms_per_pass_by_rank": by_rank,
                "equal_to_single_gpu_run": ok, "result_digest": dig, "generate_s": round(run.gen_s, 1)}
    finally:
        run.close()


def _segments(a, start, length):
    """a[start[i]:start[i] + length[i]] for every i, concatenated"""
    length = np.asarray(length, np.int64)
    ends = np.cumsum(length)
    if not len(ends) or not ends[-1]:
        return a[:0]
    return a[np.arange(ends[-1]) - np.repeat(ends - length - np.asarray(start, np.int64), length)]


def result_arrays(outs, calls, packed, limit=DUMP_LIMIT):
    """The results of one step ({call: batch.BatchOutput}) as flat float64 arrays, region by region in workload order.

    Per region: `region` (index in the workload), `region_status`, `so_len` / `uniq_len` / `ctg_len` (its number of
    sample-only k-mers, unique reads and contigs).  Per contig, in acceptance order: `ctg_seq_len`, `ctg_cnt_len`,
    `ctg_reads_len`, `ctg_kmers_len`.  The payloads `so_mers`, `so_counts`, `uniq_rec`, `uniq_mult`, `ctg_seq`,
    `ctg_kmer_locs`, `ctg_indel_only`, `ctg_others`, `ctg_reads`, `ctg_kmer_mer`, `ctg_kmer_pos`, `ctg_kmer_lth`,
    `ctg_kmer_dist`, `ctg_kmer_order` follow in that order.  The library leaves contig payloads in completion order,
    which changes from run to run; gathered in this order they do not.  Read indices count from the region's first
    read, so they do not depend on how regions are packed into calls.  Every value is an integer below 2**53 (k-mer
    codes need k <= 26), so float64 holds it exactly.  Above `limit` bytes, a fixed seeded sample of whole regions is
    kept."""
    items = []                                  # (region in the workload, call, region in the call, elements to write)
    for c in sorted(outs):
        o = outs[c]
        per_ctg = 4 + 2 * o.seq_off[:, 1] + 2 * o.cnt_off[:, 1] + o.reads_off[:, 1] + 5 * o.kmers_off[:, 1]
        cum = np.concatenate([[0], np.cumsum(per_ctg)])
        size = 5 + 2 * np.diff(o.so_off) + 2 * np.diff(o.uniq_reg_off) + cum[o.ctg_reg_off[1:]] - cum[o.ctg_reg_off[:-1]]
        items += [(calls[c][r], c, r, int(size[r])) for r in range(o.n_regions)]
    items.sort()
    elems = np.array([it[3] for it in items], np.int64)
    if 8 * int(elems.sum()) > limit:
        order = np.random.default_rng(0).permutation(len(items))
        items = [items[i] for i in np.sort(order[np.cumsum(elems[order]) <= limit // 8])]
    cols = {}

    def add(name, a):
        cols.setdefault(name, []).append(np.asarray(a))

    for g, c, r, _n in items:
        o, base = outs[c], int(packed[c].read_reg_off[r])
        add("region", [g])
        add("region_status", o.region_status[r:r + 1])
        a, b = o.so_off[r], o.so_off[r + 1]
        add("so_len", [b - a])
        add("so_mers", o.so_mers[a:b])
        add("so_counts", o.so_counts[a:b])
        a, b = o.uniq_reg_off[r], o.uniq_reg_off[r + 1]
        add("uniq_len", [b - a])
        add("uniq_rec", o.uniq_rec[a:b].astype(np.int64) - base)
        add("uniq_mult", o.uniq_mult[a:b])
        cs = slice(o.ctg_reg_off[r], o.ctg_reg_off[r + 1])
        add("ctg_len", [cs.stop - cs.start])
        for name, tab in (("ctg_seq_len", o.seq_off), ("ctg_cnt_len", o.cnt_off), ("ctg_reads_len", o.reads_off),
                          ("ctg_kmers_len", o.kmers_off)):
            add(name, tab[cs, 1])
        for name, arr, tab in (("ctg_seq", o.seq, o.seq_off), ("ctg_kmer_locs", o.kmer_locs, o.seq_off),
                               ("ctg_indel_only", o.indel_only, o.cnt_off), ("ctg_others", o.others, o.cnt_off),
                               ("ctg_reads", o.reads, o.reads_off), ("ctg_kmer_mer", o.kmer_mer, o.kmers_off),
                               ("ctg_kmer_pos", o.kmer_pos, o.kmers_off), ("ctg_kmer_lth", o.kmer_lth, o.kmers_off),
                               ("ctg_kmer_dist", o.kmer_dist, o.kmers_off), ("ctg_kmer_order", o.kmer_order, o.kmers_off)):
            seg = _segments(arr, tab[cs, 0], tab[cs, 1])
            add(name, seg.astype(np.int64) - base if name == "ctg_reads" else seg)
    res = {}
    for name, parts in cols.items():
        a = np.concatenate(parts)
        if a.size and int(a.max()) >= 1 << 53:
            raise ValueError("%s: values from 2**53 up are not exact in float64" % name)
        res[name] = a.astype(np.float64)
    return res


def dump_outputs(out_dir, run, prefix=""):
    """--dump-outputs: the results of the last pass `run` timed, one .npy per array of result_arrays"""
    from breakmer_b200 import batch
    outs = {c: batch.BatchOutput(res, run.packed[c]) for c, (_j, res) in run.last.items()}
    arrays = result_arrays(outs, run.calls, run.packed, DUMP_LIMIT // run.D.world)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def gpu_arm(args):
    D = Dist(args)
    torch = D.torch
    from breakmer_b200 import batch
    desc, n0, scaling = WORKLOADS[args.workload]
    cfg = config_dict(args.workload, D.world, args.regions)
    total = cfg["regions_total"]
    hbm_peak, peak_src = load_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    run = ShardRun(D, args.workload, total, args.inflight, args.spec_width, replicate=args.replicate, static=args.static_shards)
    H = min(run.inflight, run.n_handles)
    h = run.handles[0]

    # ---- resident-input run: `value` -----------------------------------------------------
    # Steps are independent batches; the rank's single host thread keeps `inflight` of them queued on the device
    # (one handle = one stream + its own buffers each), so the tail of one batch -- a few regions with long serial
    # chains -- overlaps the bulk of the next.  inflight=1 is the strictly sequential mode (L2 flushed between steps).
    run.upload()
    run.warm(True, args.warmup)            # >= W untimed warm-up steps, >= 3 calls on every handle (arenas reach steady state)
    # per-kernel device times: a short SEQUENTIAL pass on one handle with the library's CUDA-event timers on
    # (in the pipelined region kernels of different batches share the SMs, so their durations are not comparable)
    lat_ms = []
    h.kernel_times_reset(True)
    kt_steps = 3
    for _ in range(kt_steps):
        flush.zero_()
        torch.cuda.synchronize()
        r = batch.run(h, None, resident=True, decode=False)
        lat_ms.append(float(r.gpu_ms))
    ktimes = h.kernel_times()
    for hh in run.handles:
        hh.kernel_times_reset(False)                # timers off, launch counters zeroed for the timed region
    sampler = ClockSampler(D.local_rank)
    if not args.no_clock_sampler and D.rank == 0:   # the line is rank 0's: its GPU is the one sampled
        sampler.start()
    dev_s, wall_s = run.timed(args.steps, True, flush)
    host_resident = run.host_ms
    clocks = sampler.stop()
    if args.dump_outputs:             # before any other call reuses the handles' result buffers
        dump_outputs(args.dump_outputs, run, "rank%d_" % D.rank if D.world > 1 else "")
    rank_ms = D.gather_floats(1000.0 * run.last_local_dev_s / args.steps)
    calls_by_rank = [int(v) for v in D.gather_floats(float(run.items_run))]
    gpu_launches = 0
    for hh in run.handles:
        gpu_launches += int(sum(v[1] for v in hh.kernel_times().values()))
    value = total * args.steps / dev_s
    cnt = {k: int(D.sum(float(v))) for k, v in sorted(run.counters().items())}     # one whole step, all ranks
    n_cells_rank = cnt["dp_cells"]
    kmers_per_s = float(cnt["sample_only"]) * args.steps / dev_s
    cells_all = float(n_cells_rank)

    # ---- end to end through the C ABI with host buffers: `e2e` ---------------------------------------
    run.warm(False)
    _, e2e_s = run.timed(args.steps, False)
    host_e2e = run.host_ms
    e2e_value = total * args.steps / e2e_s
    pk0 = run.packed[run.mine[0]]
    outs = {c: batch.BatchOutput(res, run.packed[c]) for c, (_j, res) in run.last.items()}
    # bytes of one whole step (all calls): inputs from the packed arrays, results from the calls this rank ran last
    h2d = D.sum(float(sum(run.packed[c].input_bytes + 8 * (len(run.packed[c].read_off) + len(run.packed[c].sc_off) + len(run.packed[c].ref_off)) +
                          len(run.packed[c].read_flags) for c in outs)))
    d2h = 0
    for out in outs.values():
        d2h += int(out.seq.nbytes + out.kmer_locs.nbytes + out.indel_only.nbytes + out.others.nbytes + out.reads.nbytes +
                   out.kmer_mer.nbytes + 2 * out.kmer_pos.nbytes + out.so_mers.nbytes + out.so_counts.nbytes +
                   out.uniq_rec.nbytes + out.uniq_mult.nbytes)
    d2h = D.sum(float(d2h))
    ok, digest, _nl = (None, None, 0) if args.replicate else run.check_against_single_gpu()

    # ---- same steps with the persistent reference k-mer cache (reported beside the headline, not as it) ----
    ref_cache = None
    if not args.no_ref_cache_leg and len(run.calls) == 1:
        regions_mine = [run.regions[i] for i in run.calls[0]]
        pk_nr = batch.PackedBatch(regions_mine, with_ref=False).pin()
        saved = run.packed
        for hh in run.handles:
            hh.ref_cache_build([r.ref_fwd for r in regions_mine], pk0.k)
        run.packed = {0: pk_nr}
        run.upload()
        run.warm(True)
        rc_s, _ = run.timed(args.steps, True)
        ref_cache = {"value": total * args.steps / rc_s, "unit": UNIT, "ms_per_step": 1000.0 * rc_s / args.steps,
                     "note": "reference k-mers of the targets counted once and kept on the device (bk_ref_cache_build), as the "
                             "reference keeps its reference dumps behind marker files (utils.py:157)"}
        for hh in run.handles:
            hh.ref_cache_clear()
        run.packed = saved

    # ---- ingest row (SURVEY.md 8.7 f.1): the same steps starting from FASTA/FASTQ FILES (tmpfs) -------------------
    from_files = None
    if not args.no_ingest_leg:
        from_files = ingest_leg(args, D, run, total)

    # ---- the Python drop-in a BreaKmer user calls (sv_processor.compare_kmers_batch on target objects) -------------
    dropin = None
    if not args.no_dropin_leg and D.rank == 0:
        dropin = dropin_leg(run, D.local_rank)

    # ---- roofline of the dominant kernel (the assembler) and of the k-mer stage kernels -----------------------------
    asm_ms, asm_n = ktimes["assemble"]
    asm_ms_per_launch = asm_ms / max(1, asm_n)
    # (the call the sequential pass above timed: the one resident on this rank's first handle; with the work queue a rank
    # may have run none of the calls of the last pass, so this is a run of its own)
    pk0 = run.packed[run.handle_call[0]]
    out0 = batch.run(run.handles[0], pk0)
    n_only0 = int(out0.so_off[-1])
    NU = int(out0.uniq_reg_off[-1])
    read_lens = pk0.read_off[1:] - pk0.read_off[:-1]
    uniq_bases = int(read_lens[out0.uniq_rec].sum()) if NU else 0
    d2h0 = int(out0.seq.nbytes + out0.kmer_locs.nbytes + out0.indel_only.nbytes + out0.others.nbytes + out0.reads.nbytes +
               out0.kmer_mer.nbytes + 2 * out0.kmer_pos.nbytes)
    # algorithmic bytes of one assemble launch (DESIGN.md "A-stage"): every unique read once, the sample-only
    # table (12 B/mer), and the contigs written
    asm_bytes = uniq_bases + 12 * n_only0 + d2h0
    asm_gbs = asm_bytes / (asm_ms_per_launch * 1e-3) / 1e9 if asm_ms_per_launch > 0 else 0.0
    cells0 = int(out0.n_dp_cells)
    cells_per_s = cells0 * kt_steps / (asm_ms * 1e-3) if asm_ms > 0 else 0.0
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    alu = int_peak(sm_mhz)
    # DRAM traffic per launch from the committed ncu --set full captures; only valid for the default workload on one GPU
    default_shape = args.workload == "C2" and total == 500 and D.world == 1
    roof_k = kstage_rooflines(ktimes, kt_steps, pk0, out0, hbm_peak)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dev_s / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "config": cfg,
        "run": {"batches_in_flight": H, "host_threads_per_rank": 1, "calls_per_step": len(run.calls),
                "regions_per_call": [len(c) for c in run.calls][:16], "calls_run_by_rank": calls_by_rank,
                "assignment": "static (call c on rank c % N)" if run.static else "dynamic (host-side queue over the ranks)",
                "input_bytes_per_step": sum(run.regions[i].input_bases() for c in run.calls for i in c),
                "assembler_spec_width": args.spec_width or 4, "host_cores_per_rank": max(1, (os.cpu_count() or 1) // max(1, D.world)),
                "l2": ("256 MB buffer written between timed steps (flush)" if H == 1 else
                       "%d independent batches in flight on separate buffers; the per-step working set (~1 GB of "
                       "key/value, scratch and state arrays per batch) exceeds the 126 MB L2" % H),
                "timing": "CUDA events bracketing the K steps (barrier + synchronize on both sides), max over ranks",
                "wall_ms_per_step": 1000.0 * wall_s / args.steps, "device_ms_per_step_by_rank": [round(v, 3) for v in rank_ms],
                "replicated_regions_diagnostic": bool(args.replicate),
                "sequential_latency_ms_per_step": (min(lat_ms) if lat_ms else None), "generate_s": round(run.gen_s, 1),
                "host_e2e": host_e2e, "host_resident": host_resident},
        "sharding_check": {"regions": total, "equal_to_single_gpu_run": ok, "result_digest": digest,
                           "what": "per-region digests (sample-only table + every contig) gathered by target name from all ranks "
                                   "vs the same regions run on rank 0's GPU alone"},
        "sample_only_kmers_per_s": kmers_per_s,
        "with_ref_kmer_cache": ref_cache, "from_files": from_files, "e2e_dropin": dropin,
        "per_step": {"contigs": cnt["contigs"], "check_align_calls": cnt["check_align"], "dp_cells": n_cells_rank,
                     "kmer_occurrences": cnt["kmer_occ"], "sorted_keys": cnt["sorted"], "sample_only_kmers": cnt["sample_only"],
                     "note": "one whole step (all calls, all ranks)"},
        "roofline": {"kernel": "assemble_kernel", "bound": "hbm", "achieved": asm_gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": asm_gbs / hbm_peak, "traffic": 225505792 if default_shape else None, "peak_source": peak_src,
                     "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch (profiles/r2_assemble_kernel.md): 52 MB "
                                     "read + 173 MB written; the writes are the per-warp DP score tables (scratch, ~280 MB footprint) "
                                     "being evicted from L2, not re-reads of the inputs",
                     "algorithmic_bytes_per_launch": asm_bytes, "ms_per_launch": asm_ms_per_launch,
                     "share_of_step": asm_ms / sum(lat_ms) if lat_ms else None,
                     "note": "the dominant kernel is an integer-issue/latency bound DP state machine that moves "
                             "O(m+n) bytes per O(m*n) cell updates; its HBM fraction is small by construction, "
                             "see roofline_alu (its real ceiling) and roofline_per_kernel (the HBM-bound k-mer stage)"},
        "roofline_alu": {"kernel": "assemble_kernel", "bound": "int32 issue", "achieved": cells_per_s, "peak": alu["cells_per_s"],
                         "unit": "DP cell updates/s", "frac": cells_per_s / alu["cells_per_s"],
                         "achieved_in_flight": cells_all * args.steps / dev_s,
                         "frac_in_flight": (cells_all * args.steps / dev_s) / (alu["cells_per_s"] * D.world),
                         "note": "`achieved`/`frac`: one launch alone (sequential pass; bounded by the longest region's serial "
                                 "chain); `*_in_flight`: all DP cells of the timed region / its device time with %d batches in "
                                 "flight (other stages included), against the peak of all %d GPUs" % (H, D.world),
                         "peak_source": alu["source"]},
        "roofline_per_kernel": roof_k,
        "kernel_ms_per_step": {k: round(v[0] / kt_steps, 4) for k, v in ktimes.items() if v[1]},
        "kernel_timing": "sequential pass of %d steps with L2 flush, CUDA events per kernel on the library stream" % kt_steps,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1000.0 * e2e_s / args.steps, "bytes_note": "one whole step, all ranks"},
        "gpu_launches": gpu_launches,
        "clocks": clocks,
    }
    regions0 = run.regions
    run.close()
    if not args.no_extra_workloads and args.workload == "C2" and not args.regions:
        if "c5" in args.extra_workloads:
            line["c5_strong"] = sharded_summary(D, "C5", args.c5_regions, args, max(2, args.steps // 6))
        if "c3" in args.extra_workloads:
            line["c3_sharded"] = sharded_summary(D, "C3", 500 * D.world, args, max(2, args.steps // 4))
    if D.rank == 0 and D.world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_single(args.workload, regions0)
        line["cpu_baseline"]["value_with_c_nw_for_context"] = cpu_c_nw_single(regions0)
    elif D.rank == 0:
        line["cpu_baseline"] = None
    if D.rank == 0:
        print(json.dumps(line))
    D.close()
    return 0


def int_peak(sm_mhz):
    """Ceiling of the DP in cell updates/s.  Measured: profiles/r2_int_peak.json holds the rate at which the DP's own
    cell update (the instruction sequence of nw.cuh, registers only, no shuffles) issues on a full B200
    (tools/int_peak.py).  Fallback: the nominal ALU-pipe arithmetic."""
    p = os.path.join(ROOT, "profiles", "r2_int_peak.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return {"cells_per_s": float(d["cells_per_s"]) * sm_mhz / float(d["sm_mhz"]),
                "source": "measured: %s (tools/int_peak.py, profiles/r2_int_peak.json), scaled to the SM clock of this run" % d["what"]}
    return {"cells_per_s": 148 * 4 * 16 * sm_mhz * 1e6 / 8.0,
            "source": "nominal: 148 SM x 4 SMSP x 16 alu lanes/clk x SM clock / 8 alu-pipe instructions per cell"}


def kstage_rooflines(ktimes, kt_steps, pk, out, hbm_peak):
    """HBM roofline of every k-mer stage / prep kernel family: algorithmic bytes per step (SURVEY.md 8.5) over its
    CUDA-event time in the sequential pass."""
    nd = int(pk.read_bases.size); ns = int(pk.sc_bases.size); nr = int(pk.ref_bases.size); nn = int(pk.normal_bases.size)
    n_sorted = nd + ns
    n_only = int(out.so_off[-1])
    NU = int(out.uniq_reg_off[-1])
    n_rec = len(pk.read_off) - 1
    alg = {
        # G1+G2: 1 B/base in (every input; the reference strand counted once), 12 B per sorted window out
        "kmer_emit": nd + ns + nr + nn + 12 * n_sorted,
        # G3 by the survey's definition: one read + one write of (key, value) per occurrence, whatever the pass count
        "sort_count": 8 * n_sorted, "sort_scan": 0, "sort_scatter": 2 * 12 * n_sorted,
        "run_select": 12 * n_sorted + 8 * n_sorted,        # keys + values in, flag + count out
        "run_scatter": 12 * n_only + 8 * n_sorted,
        "scan": 12 * n_sorted,
        "group_reads": nd + 12 * n_rec + 13 * NU,
        "index": nd + 24 * NU,
        "aux_sort": 0,                                     # (radix passes of the read-grouping and index sorts: launch-latency bound,
                                                           #  a few hundred thousand elements; no meaningful HBM figure)
        "prep": 16 * out.n_regions,
        # one CTA per region (region_kmers.cuh): every input base once (reference strand counted once, SURVEY.md 8.5)
        # + (w + 4) B per sample-only k-mer out
        "region_kmers": nd + ns + nr + nn + 12 * n_only,
    }
    res = {}
    whole_sort_ms = 0.0
    for name, (ms, n) in ktimes.items():
        if not n or name in ("assemble", "nw_batch"):
            continue
        per_step_ms = ms / kt_steps
        if name in ("sort_count", "sort_scan", "sort_scatter"):
            whole_sort_ms += per_step_ms
        b = alg.get(name, 0)
        gbs = b / (per_step_ms * 1e-3) / 1e9 if per_step_ms > 0 else 0.0
        res[name] = {"ms_per_step": round(per_step_ms, 4), "launches_per_step": n / kt_steps, "algorithmic_bytes_per_step": int(b),
                     "achieved_GBps": round(gbs, 1), "frac": round(gbs / hbm_peak, 4) if b else None}
    if whole_sort_ms > 0:
        gbs = 2 * 12 * n_sorted / (whole_sort_ms * 1e-3) / 1e9
        res["whole_sort"] = {"ms_per_step": round(whole_sort_ms, 4), "algorithmic_bytes_per_step": 2 * 12 * n_sorted,
                             "achieved_GBps": round(gbs, 1), "frac": round(gbs / hbm_peak, 4),
                             "note": "count + scan + scatter of all passes against one read + one write per occurrence (SURVEY.md 8.5 G3)"}
    return res


def dropin_leg(run, device):
    """`e2e_dropin`: breakmer_b200.sv_processor.compare_kmers_batch on target objects shaped like the reference's
    (what a BreaKmer user calls after extract_bam_reads / clean_reads), files in tmpfs, contigs materialised lazily."""
    import shutil
    import tempfile
    from tools import dropin_profile
    from breakmer_b200 import sv_processor
    root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    d = tempfile.mkdtemp(prefix="bk_dropin_", dir=root)
    try:
        regions = [run.regions[i] for i in run.calls[0]][:500]
        targets = [dropin_profile.Target(r, d) for r in regions]
        best = {}
        for label, kw in (("python_marshalling", dict(ingest="python")), ("native_ingest", dict(ingest="native"))):
            for rep in range(3):
                for t in targets:
                    t.reset()
                t0 = time.time()
                sv_processor.compare_kmers_batch(targets, device=device, **kw)
                dt = time.time() - t0
                best[label] = min(best.get(label, dt), dt)
        # touching what resolve_sv reads from every contig (sv_processor.py:731-746): sequence, counts, reads, k-mers
        t0 = time.time()
        n_ctg = 0
        for t in targets:
            for c in t.kmers["clusters"]:
                n_ctg += 1
                c.get_contig_seq(); c.get_contig_counts().get_total_reads(); len(c.reads); len(c.kmers); c.get_kmer_locs()
        touch_s = time.time() - t0
        n = len(targets)
        return {"value": n / best["native_ingest"], "unit": "targets/s", "targets": n, "contigs": n_ctg,
                "ms_per_batch_native_ingest": 1000.0 * best["native_ingest"],
                "ms_per_batch_python_marshalling": 1000.0 * best["python_marshalling"],
                "ms_to_touch_every_contig_field": 1000.0 * touch_s,
                "what": "sv_processor.compare_kmers_batch(targets) on %d reference-shaped target objects, best of 3" % n}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def ingest_leg(args, D, run, total):
    """Every step = bk_ingest_files (text of the four files of each target -> page-locked arrays, host threads) followed by
    bk_batch_submit / bk_batch_wait.  Files live in tmpfs; writing them is not timed.  Python marshalling of the same
    regions (batch.PackedBatch) is timed beside it for context."""
    import shutil
    import tempfile
    import torch
    from breakmer_b200 import batch, ingest
    own = [c for c in range(len(run.calls)) if c % D.world == D.rank]      # this leg: call c on rank c % N
    regions = [run.regions[i] for c in own for i in run.calls[c]]
    pk = run.packed[own[0]]
    handles = run.handles
    handles = handles[:run.inflight]
    H = len(handles)
    root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    d = tempfile.mkdtemp(prefix="bk_bench_r%d_" % D.rank, dir=root)
    try:
        refs, fqs, scs, nms = [], [], [], []
        any_normal = any(r.normal_reads for r in regions)
        n_bytes = 0
        for i, r in enumerate(regions):
            base = os.path.join(d, "t%05d" % i)
            texts = {
                "_ref.fa": ">%s\n%s\n" % (r.name, "\n".join(r.ref_fwd[a:a + 60] for a in range(0, len(r.ref_fwd), 60))),
                "_reads.fastq": "".join("%s\n%s\n+\n%s\n" % (rec[0], rec[1], rec[2]) for rec in r.reads),
                "_sc.fa": "".join(">%s\n%s\n" % (rec[0], rec[1]) for rec in r.sc_records),
            }
            if any_normal:
                texts["_normal.fastq"] = "".join("@%s\n%s\n+\n%s\n" % (rec[0].lstrip("@"), rec[1], "I" * len(rec[1]))
                                                 for rec in r.normal_reads)
            for suffix, t in texts.items():
                with open(base + suffix, "w", newline="\n") as f:
                    f.write(t)
                n_bytes += len(t)
            refs.append(base + "_ref.fa"); fqs.append(base + "_reads.fastq"); scs.append(base + "_sc.fa")
            nms.append(base + "_normal.fastq" if any_normal else None)
        normal = nms if any_normal else None
        cores = max(1, (os.cpu_count() or 1) // D.world)     # this rank's share of the host
        ings = [ingest.Ingest(n_threads=cores) for _ in range(H)]   # one parse at a time (single host thread), all cores each
        kw = dict(normal=normal, k=pk.k, rc_thresh=pk.rc_thresh)
        solo = ings[0]
        solo.files(refs, fqs, scs, **kw)
        t0 = time.time()
        reps = 5
        for _ in range(reps):
            solo.files(refs, fqs, scs, **kw)
        parse_s = (time.time() - t0) / reps
        t0 = time.time()
        batch.PackedBatch(regions)
        py_s = time.time() - t0

        def one_pass(steps):
            last = None
            for t in range(steps):
                j = t % H
                if t >= H:
                    last = batch.wait(handles[j], decode=False)
                batch.submit(handles[j], ings[j].files(refs, fqs, scs, **kw))
            for t in range(max(0, steps - H), steps):
                last = batch.wait(handles[t % H], decode=False)
            return last

        one_pass(H)
        D.barrier()
        t0 = time.time()
        last = one_pass(args.steps)
        torch.cuda.synchronize()
        local = time.time() - t0
        D.barrier()
        ff_s = D.max(local)
        n_contigs = int(last.n_contigs)
        # contig hand-off (row f.3): the contig.setup files of every contig of one batch result, written to tmpfs
        pk0 = ings[0].files(refs, fqs, scs, **kw)
        res0 = batch.run(handles[0], pk0, decode=False)
        hand_s, n_files = [], 0
        writer = ingest.Ingest(n_threads=cores)
        for rep in range(3):
            out_root = os.path.join(d, "handoff%d" % rep)
            t0 = time.time()
            n_files = writer.write_contigs(res0, pk0, [os.path.join(out_root, "t%05d" % i, "contigs") for i in range(len(regions))],
                                            [os.path.join(out_root, "t%05d_clusters.out" % i) for i in range(len(regions))])
            hand_s.append(time.time() - t0)
        writer.close()
        for g in ings:
            g.close()
        return {"value": total * args.steps / ff_s, "unit": UNIT, "ms_per_step": 1000.0 * ff_s / args.steps,
                "text_bytes_per_step": n_bytes, "n_contigs": n_contigs,
                "parse_only": {"ms_per_batch": 1000.0 * parse_s, "regions_per_s": len(regions) / parse_s,
                               "text_MB_per_s": n_bytes / parse_s / 1e6, "host_threads": cores},
                "python_marshalling_ms_per_batch": 1000.0 * py_s,
                "handoff": {"ms_per_batch": 1000.0 * min(hand_s), "files_per_batch": n_files, "host_threads": cores,
                            "what": "bk_write_contigs: <id>.fq + <id>.fa per contig and the cluster file per target "
                                    "(sv_processor.py:749-782), tmpfs"},
                "note": "each step parses the targets' FASTA/FASTQ files (tmpfs) with bk_ingest_files into page-locked memory "
                        "and runs bk_batch_submit / bk_batch_wait; %d ingest threads, one driving host thread" % cores}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--regions", type=int, default=0, help="override the workload's region count (per GPU if weak; debugging)")
    ap.add_argument("--spec-width", type=int, default=0, help="assembler warps per region (0 = auto)")
    ap.add_argument("--inflight", type=int, default=8,
                    help="independent batches (steps) kept on the device at once (a batch lasts as long as its longest "
                         "region's serial chain, 17-35 ms on the panel: the depth must cover it)")
    ap.add_argument("--c5-regions", type=int, default=20000, help="size of the c5_strong workload")
    ap.add_argument("--replicate", action="store_true", help="diagnostic: every call is call 0 (not the headline)")
    ap.add_argument("--static-shards", action="store_true", help="call c always runs on rank c %% N (plain LPT partition) "
                    "instead of the host-side work queue over the ranks")
    ap.add_argument("--no-clock-sampler", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cache-leg", action="store_true")
    ap.add_argument("--no-ingest-leg", action="store_true")
    ap.add_argument("--no-dropin-leg", action="store_true")
    ap.add_argument("--no-extra-workloads", action="store_true", help="skip the c5_strong / c3_sharded keys")
    ap.add_argument("--extra-workloads", default="c5,c3", help="which of the two extra workloads to run (default both)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args)
    return gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
