"""Region sharding across GPUs.

Target regions are independent (SURVEY.md section 8.6): the reference's region loop
(sv_processor.py:185-201) touches no shared mutable state.  Work is therefore
partitioned BY REGION with no data-path collective; the only cross-rank step is a
host-side gather of per-region results in target-name order (sv_processor.py:175-176
iterates sorted names).

Two ways to run it:

  * one process per GPU (torchrun; what bench.py does): every rank cuts the regions into the
    same calls with `assign_lpt` on the same static costs; the calls are either pinned to ranks
    (call c on rank c % N) or handed out by `CallQueue` -- an atomic counter in the
    torch.distributed key-value store, host side, no device traffic -- so that a rank whose calls
    turn out slow takes fewer of them; `gather_by_name` collects the per-region results on rank 0;
  * one process, several devices: `run_sharded(regions, devices=[0, 1, ...])` and
    `sv_processor.compare_kmers_batch(targets, devices=[...])` -- `plan_chunks` cuts the regions
    into chunks of similar static cost, and `drive_chunks` runs one host thread per device that
    pulls chunks from a shared queue (largest first) and keeps `inflight` batches on its device
    with bk_batch_submit / bk_batch_wait.
"""
import hashlib
import queue
import threading

import numpy as np

# Static cost model (before anything ran on the device), in DP-cell equivalents.  Fitted on the per-region
# `region_dp_cells` of 24,600 synthetic regions (C2 x 4000, C3, C4, C5 x 20000; tools/cost_model_data.py,
# profiles/r2_cost_model.md): DP cells ~ 94 n^2 + 32.6 k n for n read records (corr 0.61 -- the rest is the
# region's own event structure, which nothing known before the pass predicts), and the k-mer stage costs
# about as much device time per input byte as 57 DP cells.
COST_CELLS_PER_READ2 = 94.0
COST_CELLS_PER_READ = 32600.0
COST_CELLS_PER_BYTE = 57.0


def region_cost(region):
    """Static cost estimate of one region (anything with .reads, .sc_records, .ref_fwd, .normal_reads)."""
    n = len(region.reads)
    nbytes = 2 * len(region.ref_fwd) + sum(len(r[1]) for r in region.reads) + sum(len(r[1]) for r in region.sc_records)
    nbytes += sum(len(r[1]) for r in getattr(region, "normal_reads", ()))
    return COST_CELLS_PER_READ2 * n * n + COST_CELLS_PER_READ * n + COST_CELLS_PER_BYTE * nbytes + 1.0


def assign_lpt(costs, world_size):
    """Longest-processing-time-first assignment.  Returns, per rank, the sorted list
    of region indices it owns.  Deterministic: ties broken by index."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    load = [0] * world_size
    owned = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda w: (load[w], w))
        owned[r].append(i)
        load[r] += costs[i]
    return [sorted(o) for o in owned]


def chunk_indices(indices, max_regions):
    """Split a rank's regions into calls of at most max_regions (n_regions <= 65535 per call; a few thousand
    regions per call keep the device arrays at a few GB)."""
    indices = list(indices)
    if not indices:
        return []
    n_chunks = (len(indices) + max_regions - 1) // max_regions
    per = (len(indices) + n_chunks - 1) // n_chunks
    return [indices[a:a + per] for a in range(0, len(indices), per)]


class CallQueue:
    """Work queue over the ranks of a one-process-per-GPU job: `n_items` numbered items, each taken by exactly one rank.
    The queue is one counter in the key-value store torch.distributed already holds for rendezvous (rank 0 serves it
    over TCP on the host; ~50 us per take): no collective, nothing on the device.  Every rank must construct the queues
    of a job in the same order (the key carries a per-name sequence number).  With world_size 1 it is a local counter."""
    _seq = {}

    def __init__(self, name, n_items, world_size=1, store=None):
        self.n_items = int(n_items)
        self._local = 0
        self._store = None
        if world_size > 1:
            if store is None:
                from torch.distributed import distributed_c10d
                store = distributed_c10d._get_default_store()
            self._store = store
            CallQueue._seq[name] = CallQueue._seq.get(name, 0) + 1
            self._key = "bk_call_queue/%s/%d" % (name, CallQueue._seq[name])

    def take(self):
        """-> the next item number, or None when the queue is empty"""
        if self._store is None:
            t = self._local
            self._local += 1
        else:
            t = self._store.add(self._key, 1) - 1
        return t if t < self.n_items else None


def gather_by_name(local_results, rank, world_size, group=None):
    """Host-side gather of {region name: result} dicts onto rank 0, merged and
    ordered by target name.  Uses torch.distributed only as plumbing."""
    if world_size == 1:
        return dict(sorted(local_results.items()))
    import torch.distributed as dist
    gathered = [None] * world_size if rank == 0 else None
    dist.gather_object(local_results, gathered, dst=0, group=group)
    if rank != 0:
        return None
    merged = {}
    for part in gathered:
        overlap = set(merged) & set(part)
        if overlap:
            raise ValueError("region assigned to two ranks: %s" % sorted(overlap)[:3])
        merged.update(part)
    return dict(sorted(merged.items()))


def region_digests(out, packed):
    """{region name: sha1 hex} of everything the hot path returns for a region -- the sample-only (mer, count) table
    and every contig (sequence, kmer_locs, both count vectors, reads, k-mer 5-tuples) -- independent of how the
    regions were batched: read indices are taken relative to the region's first record."""
    res = {}
    rro = packed.read_reg_off
    for r in range(out.n_regions):
        hsh = hashlib.sha1()
        a, b = int(out.so_off[r]), int(out.so_off[r + 1])
        hsh.update(out.so_mers[a:b].tobytes())
        hsh.update(out.so_counts[a:b].tobytes())
        hsh.update(np.int32(out.region_status[r]).tobytes())
        base = np.int32(rro[r])
        for c in range(int(out.ctg_reg_off[r]), int(out.ctg_reg_off[r + 1])):
            so, sl = out.seq_off[c]
            co, cl = out.cnt_off[c]
            ro, nr = out.reads_off[c]
            ko, nk = out.kmers_off[c]
            for arr in (out.seq[so:so + sl], out.kmer_locs[so:so + sl], out.indel_only[co:co + cl], out.others[co:co + cl],
                        out.reads[ro:ro + nr] - base, out.kmer_mer[ko:ko + nk], out.kmer_pos[ko:ko + nk],
                        out.kmer_lth[ko:ko + nk], out.kmer_dist[ko:ko + nk], out.kmer_order[ko:ko + nk]):
                hsh.update(arr.tobytes())
            hsh.update(b"|")
        res[packed.names[r]] = hsh.hexdigest()
    return res


def digest_of_digests(by_name):
    """One checksum over the per-region digests in target-name order."""
    hsh = hashlib.sha1()
    for name in sorted(by_name):
        hsh.update(name.encode())
        hsh.update(by_name[name].encode())
    return hsh.hexdigest()


class DevicePipeline:
    """`inflight` handles of one device driven by ONE host thread: submit keeps up to `inflight` batches queued on the
    device (bk_batch_submit), results come back in submission order (bk_batch_wait).  long_regions=True sets the
    handles' "long_regions" option: regions with reads or contigs up to 65,535 bases are assembled in the same pass.
    rejected_contigs=True sets the option of that name: results also hold the contigs the acceptance test drops."""

    def __init__(self, device, inflight=3, spec_width=0, long_regions=False, rejected_contigs=False):
        from . import _lib
        self.device = device
        self.handles = [_lib.Handle(device) for _ in range(max(1, inflight))]
        for h in self.handles:
            h.set_option("blocking_sync", 1)           # a waiting host thread sleeps; it never competes with other GPUs' threads
            if spec_width:
                h.set_option("spec_width", spec_width)
            if long_regions:
                h.set_option("long_regions", 1)
            if rejected_contigs:
                h.set_option("rejected_contigs", 1)
        self._queue = []                               # (handle index, packed, tag) in submission order
        self.report = False                            # pop: read every batch's per-region report
        self._next = 0

    def full(self):
        return len(self._queue) >= len(self.handles)

    def submit(self, packed, tag=None):
        from . import batch
        if self.full():
            raise RuntimeError("DevicePipeline.submit: every handle is busy; pop() first")
        j = self._next
        self._next = (self._next + 1) % len(self.handles)
        batch.submit(self.handles[j], packed)
        self._queue.append((j, packed, tag))

    def pop(self, decode=True):
        """-> (result of the oldest batch in flight, its packed input, its tag).  The result's `.report` is the batch's
        batch.region_report, read before its handle takes another batch, if `self.report` is set or a region of the
        batch failed; else None.  With decode=False its `.rejected` is the batch's batch.rejected_tables (None unless the
        batch was submitted with the "rejected_contigs" option); a decoded result holds them already."""
        from . import batch
        j, packed, tag = self._queue.pop(0)
        res = batch.wait(self.handles[j], packed, decode=decode)
        res.report = batch.region_report_if(self.handles[j], res, self.report)
        if not decode:
            res.rejected = batch.rejected_tables(self.handles[j])
        return res, packed, tag

    def pending(self):
        return len(self._queue)

    def close(self):
        for h in self.handles:
            h.close()
        self.handles = []


def plan_chunks(costs, n_devices, max_per_chunk, key=None):
    """Chunks of similar static cost: consecutive runs of the indices ordered most expensive first (ties by index), at
    least one chunk per device and at most max_per_chunk indices per chunk.  Each chunk is sorted by `key` (None: by
    index)."""
    n = len(costs)
    if not n:
        return []
    order = sorted(range(n), key=lambda i: (-costs[i], i))
    per = -(-n // max(n_devices, -(-n // max_per_chunk)))
    return [sorted(order[a:a + per], key=key) for a in range(0, n, per)]


def drive_chunks(chunks, devices, inflight, pack, consume, pipe=None, decode=True, long_regions=False, report=False,
                 apply_thread=False, rejected_contigs=False):
    """Run `chunks` (lists of indices) on `devices`, each device taking the next chunk when it has room for it.
    pack(indices, slot) -> (packed, tag) parses a chunk into parse buffer `slot`; consume(result, packed, tag) takes the
    finished batches (pipe.pop(decode)), per device in submission order.  `pipe`: an open pipeline of devices[0], driven
    on the calling thread and left open; without it every device gets a thread and an `inflight`-handle DevicePipeline of
    its own, closed at the end.  long_regions, rejected_contigs and report set the handles' options and
    DevicePipeline.report for the call.

    Without apply_thread a device's thread pops the oldest batch of a full pipeline before it parses the next chunk, and
    one parse slot per handle rotates.  With apply_thread a second thread pops and consumes while the first parses ahead,
    so one more slot rotates, and a handle is free again only once its chunk has been consumed (the result arrays live in
    the handle's arena).  The first error of any thread is re-raised on the calling thread after every thread stopped."""
    from . import batch
    todo = iter(chunks)
    lock = threading.Lock()

    def take():
        with lock:
            return next(todo, None)

    def run(pipe):
        def drain_one():
            consume(*pipe.pop(decode=decode))

        n_handles = len(pipe.handles)
        free = threading.Semaphore(n_handles)
        posted = queue.SimpleQueue()                     # one True per submitted batch, then False
        apply_errors = []

        def applier():
            try:
                while posted.get():
                    drain_one()
                    free.release()
            except Exception as e:                       # noqa: BLE001 -- re-raised on the submitting thread
                apply_errors.append(e)
                free.release()

        pipe.report = report
        with batch.options(pipe.handles, long_regions=long_regions, rejected_contigs=rejected_contigs):
            if apply_thread:
                helper = threading.Thread(target=applier)
                helper.start()
            try:
                n = 0
                while not apply_errors and (idx := take()) is not None:
                    if not apply_thread and pipe.full():
                        drain_one()
                    packed, tag = pack(idx, n % (n_handles + 1 if apply_thread else n_handles))
                    if apply_thread:
                        free.acquire()
                        if apply_errors:
                            break
                    pipe.submit(packed, tag)
                    n += 1
                    if apply_thread:
                        posted.put(True)
                while not apply_thread and pipe.pending():
                    drain_one()
            finally:
                if apply_thread:
                    posted.put(False)
                    helper.join()
        if apply_errors:
            raise apply_errors[0]

    if pipe is not None:
        run(pipe)
        return
    errors = []

    def worker(dev):
        pipe = None
        try:
            pipe = DevicePipeline(dev, inflight=inflight)
            run(pipe)
        except Exception as e:                           # noqa: BLE001 -- re-raised on the calling thread
            errors.append(e)
        finally:
            if pipe is not None:
                pipe.close()

    threads = [threading.Thread(target=worker, args=(d,)) for d in devices]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]


def run_sharded(regions, devices=(0,), max_regions=2048, inflight=3, costs=None, pack=None, on_result=None, long_regions=False):
    """The region loop of sv_processor.py:185-201 over several GPUs of one box, single process.

    regions     region-like objects (see batch.PackedBatch)
    devices     CUDA device ordinals; one host thread and `inflight` handles per device
    pack        callable(list of regions) -> PackedBatch (default batch.PackedBatch)
    on_result   callable(indices, BatchOutput, PackedBatch) called from the worker threads, once per chunk
    long_regions  assemble regions with reads or contigs up to 65,535 bases in the same pass

    Chunks of at most max_regions regions (plan_chunks on the static `region_cost`, regions in input order inside a
    chunk) are handed out dynamically, most expensive first (drive_chunks).  Returns {region name: (BatchOutput, index
    in it)} ordered by target name (the host-side gather)."""
    from . import batch
    pack = pack or batch.PackedBatch
    costs = list(costs) if costs is not None else [region_cost(r) for r in regions]
    lock = threading.Lock()
    results = {}

    def consume(out, pk, idx):
        if on_result is not None:
            on_result(idx, out, pk)
        with lock:
            for j in range(len(idx)):
                results[pk.names[j]] = (out, j)

    drive_chunks(plan_chunks(costs, len(devices), max_regions), devices, inflight,
                 lambda idx, slot: (pack([regions[i] for i in idx]), idx), consume, long_regions=long_regions)
    return dict(sorted(results.items()))
