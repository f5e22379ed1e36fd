"""Drop-in for `target.compare_kmers()` (sv_processor.py:609-645) and a batched
form for the region loop (sv_processor.py:185-201).

`compare_kmers(target)` takes the reference's own `target` object (or anything
shaped like it) after `set_ref_data`, `extract_bam_reads` and `clean_reads` have
run, and leaves it in the state the reference method leaves it in:

    target.kmers['clusters']   list of contigs (breakmer_b200.sv_assembly.contig)
    target.kmers['ref'|'case'|'case_sc'|'case_only'] = {}       (:634-636, :644)
    target.files['sample_kmers']  "<kmers path>/<name>_sample_kmers.out" written
                                  as "<mer>\\t<case count>" lines (:625-632)
    target.files['kmer_clusters'] set (:639)
    target.cleaned_read_recs = None                              (:643)

What it reads from the target: files['target_ref_fn'][0] (forward reference
FASTA; the reverse-complement file the reference also counts is by construction
its reverse complement, utils.py:367-371, and is derived on the device),
files['cleaned_fq'], files['sv_sc_unmapped_fa'], cleaned_read_recs, read_len,
paths['kmers'], name, params.get_kmer_size(), params.get_sr_thresh('min').
An optional files['normal_fq'] enables normal-sample subtraction (K4).

`compare_kmers_batch(targets)` does the same for many targets in ONE device
pass; the reference loop becomes: extract+clean all targets, one batched call,
then resolve_sv per target.

With `ingest="native"` the inputs are not marshalled from the Python objects at all:
the four files of every target (target_ref_fn[0], cleaned_fq -- the filtered FASTQ
get_fastq_reads wrote next to cleaned_read_recs, utils.py:206,237 -- sv_sc_unmapped_fa,
normal_fq) are parsed by the library's host threads straight into page-locked memory
(bk_ingest_files, SURVEY.md section 8.7 f.1).  The reads of the returned contigs are then
fresh fq_read objects built from the parsed records (same .id/.seq/.qual/.indel_only as the
caller's; of these the rest of the reference only reads .id/.seq/.qual, SURVEY.md 8.3).
`devices=[0, 1, ...]` shards the targets by region over several GPUs (no collective, host-side gather by name).
`write_contigs=True` additionally writes, for every contig of every target, the files
contig.setup writes before blat (sv_processor.py:749-782) under target.paths['contigs'], on the
library's host threads (bk_write_contigs, SURVEY.md section 8.7 f.3).
`on_capacity="assemble"` assembles targets with reads or contigs above 4,095 bases (up to 65,535) in the
same device pass as all others (the handles' "long_regions" option).
`report={}` is filled with what the assembler did for every target (batch.region_report: why it stopped, which pass
assembled it, how many seeds, find_reads and check_align calls, and how many contigs were grown and rejected).
`rejected={}` is filled with the contigs themselves that the assembler grew and then rejected, per target (the handles'
"rejected_contigs" option).
`kmer_report={}` is filled with where every target's soft-clip k-mers went in the k-mer stage (batch.kmer_report), and
`normal_kmers={}` with the k-mers the normal sample removed from each target (the handles' "normal_kmers" option).
"""
import os

from . import batch, get_handle, utils
from .sv_assembly import contig, contig_list, rejected_contigs


class _TargetInput:
    def __init__(self, trgt):
        self.name = trgt.name
        self.k = int(trgt.params.get_kmer_size())
        self.rc_thresh = int(trgt.params.get_sr_thresh('min'))
        refs = utils.read_sequences(trgt.files['target_ref_fn'][0])
        self.ref_fwd = refs[0] if refs else ""
        self.reads = []
        self.objs = []
        for seq, group in trgt.cleaned_read_recs.items():
            for fr in group:
                self.reads.append((fr.id, fr.seq, fr.qual, bool(fr.indel_only)))
                self.objs.append(fr)
        self.sc_records = [("sc", s) for s in utils.read_sequences(trgt.files['sv_sc_unmapped_fa'])]
        nfq = trgt.files.get('normal_fq') if hasattr(trgt.files, "get") else None
        self.normal_reads = [("n", s) for s in utils.read_sequences(nfq)] if nfq else []
        self.read_len = int(trgt.read_len)


class _LazyReads:
    """objs[i] for the native ingest: fq_read of record i, built on first use.  The raw record text (ids, bases,
    qualities, flags) is copied out of the ingest buffer up front -- a few memcpys -- because that buffer is reused by
    the next batch; strings are only decoded for the records somebody asks for."""

    def __init__(self, pk):
        self._cache = {}
        t, s, n = pk._text, pk._s, pk.n_reads
        view = pk._view
        self._id_off = view(t.id_off, n + 1, "int64").copy()
        self._q_off = view(t.qual_off, n + 1, "int64").copy()
        self._s_off = view(s.read_off, n + 1, "int64").copy()
        self._ids = view(t.id_bytes, int(self._id_off[-1]) if n else 0, "uint8").tobytes()
        self._quals = view(t.qual_bytes, int(self._q_off[-1]) if n else 0, "uint8").tobytes()
        self._seqs = view(s.read_bases, int(self._s_off[-1]) if n else 0, "uint8").tobytes()
        self._flags = pk.read_flags.copy()

    def __getitem__(self, i):
        fr = self._cache.get(i)
        if fr is None:
            fr = self._cache[i] = utils.fq_read(self._ids[self._id_off[i]:self._id_off[i + 1]].decode(),
                                                self._seqs[self._s_off[i]:self._s_off[i + 1]].decode(),
                                                self._quals[self._q_off[i]:self._q_off[i + 1]].decode(),
                                                bool(self._flags[i]))
        return fr


_ingests = {}


def _get_ingest(slot=0):
    import threading
    from . import ingest as _ingest
    key = (threading.get_ident(), slot)            # an ingest object's buffer is reused call to call: one per thread
    if key not in _ingests:                        # (and per batch that thread keeps in flight)
        _ingests[key] = _ingest.Ingest()
    return _ingests[key]


class _K:
    def __init__(self, k):
        self.k = k


class CapacityError(RuntimeError):
    """Some targets exceeded a device limit: a read or contig longer than 4095 bases (compare_kmers_batch's default
    on_capacity="raise"), or longer than 65,535 bases (on_capacity="assemble", where the same pass assembles everything
    up to that length).  Every other target of the batch was completed; `.targets` lists the ones that were not (their state is untouched, so the
    reference's own compare_kmers() can still be run on them), and `.reasons` says why for each of them ({name: reason},
    the reason names of batch.REASONS: "read_too_long", "contig_too_long", "kmer_list_full", "too_many_contigs")."""

    def __init__(self, names, reasons=None):
        RuntimeError.__init__(self, "compare_kmers: device capacity exceeded for target(s) %s; all other targets completed"
                              % ", ".join(names))
        self.targets = list(names)
        self.reasons = dict(reasons or {})


def _apply_chunk(targets, pk, res, inputs_k, objs, ingest, write_contigs, failed, ing=None):
    """Results of one device call -> the state target.compare_kmers leaves behind, for the targets of that call.  Returns
    the call's BatchOutput, which holds the rejected contigs when res.rejected (the call's batch.rejected_tables) does."""
    import numpy as np
    n = len(targets)
    status = np.ctypeslib.as_array(res.region_status, shape=(max(n, 1),))[:n].tolist()
    join = os.path.join
    sk_paths = [join(t.paths['kmers'], t.name) + "_sample_kmers.out" for t in targets]
    if ingest == "native":
        ing = ing or _get_ingest()
        all_ok = not any(status)
        if write_contigs:
            # contig.setup's files for every contig of every completed target in one pass (sv_processor.py:749-782,
            # bk_write_contigs); the reference-side contig.__init__ then skips its own setup() call (INTEGRATION.md)
            ing.write_contigs(res, pk, [t.paths['contigs'] if st == 0 else None for t, st in zip(targets, status)],
                              [p[:-4] + "_merged.out" if st == 0 else None for p, st in zip(sk_paths, status)])
        # the "<mer>\t<count>" files of the completed targets in one multi-threaded sweep (bk_write_sample_kmers)
        ing.write_sample_kmers(res, pk.k, sk_paths if all_ok else [p if st == 0 else None for p, st in zip(sk_paths, status)])
    out = batch.BatchOutput(res, pk, getattr(res, "rejected", None), getattr(res, "normal", None))
    ctg_reg_off = out.ctg_reg_off.tolist()
    so_off = out.so_off.tolist()
    for i, trgt in enumerate(targets):
        if status[i] != 0:
            failed.append(trgt.name)
            continue
        files = trgt.files
        files['sample_kmers'] = sk_paths[i]
        if ingest != "native":
            with open(sk_paths[i], 'w') as f:
                for mer, cnt in out.sample_only(i).items():
                    f.write("\t".join([mer, str(cnt)]) + "\n")
        kmers = trgt.kmers
        kmers['ref'] = {}; kmers['case'] = {}; kmers['case_sc'] = {}
        logger = getattr(trgt, "logger", None)
        if logger is not None and logger.isEnabledFor(20):
            logger.info('Writing %d sample-only kmers to file %s' % (so_off[i + 1] - so_off[i], sk_paths[i]))
        files['kmer_clusters'] = sk_paths[i][:-4] + "_merged.out"
        kmers['clusters'] = contig_list(out, ctg_reg_off[i], ctg_reg_off[i + 1], objs, inputs_k[i])
        trgt.cleaned_read_recs = None
        kmers['case_only'] = {}
    return out


def _record_rejected(targets, out, objs, inputs_k, rejected):
    """rejected[name] = the rejected contigs of every target of one device call (out: its BatchOutput)"""
    for i, trgt in enumerate(targets):
        rejected[trgt.name] = rejected_contigs(out, i, objs, inputs_k[i])


def _record_kmer_stage(targets, out, rows, kmer_report, normal_kmers):
    """kmer_report[name] and normal_kmers[name] of every target of one device call (out: its BatchOutput, rows: its
    batch.kmer_report), for the dicts that are wanted"""
    for i, trgt in enumerate(targets):
        if kmer_report is not None:
            kmer_report[trgt.name] = rows[i]
        if normal_kmers is not None:
            normal_kmers[trgt.name] = out.normal_kmers(i)


def _record_report(targets, rows, failed, reasons, report):
    """The batch.region_report rows of one device call (None: not read) -> reasons[name] of its failed targets, and
    report[name] of all its targets when a report is wanted."""
    if rows is None:
        return
    at = {t.name: i for i, t in enumerate(targets)}
    for name in failed:
        reasons[name] = rows[at[name]]["reason"]
    if report is not None:
        for t, row in zip(targets, rows):
            report[t.name] = row


def _pack_targets(targets, ingest, slot=0):
    """-> (packed batch, per-target k, record index -> fq_read)"""
    import numpy as np
    if ingest == "native":
        get = lambda t, key: (t.files.get(key) if hasattr(t.files, "get") else None)   # noqa: E731
        k = int(targets[0].params.get_kmer_size())
        params = {id(t.params): t.params for t in targets}                  # (targets of a run share one params object)
        if any(int(p.get_kmer_size()) != k for p in params.values()):
            raise ValueError("one k per batch")
        nfq = [get(t, 'normal_fq') for t in targets]
        pk = _get_ingest(slot).files([t.files['target_ref_fn'][0] for t in targets], [t.files['cleaned_fq'] for t in targets],
                                 [t.files['sv_sc_unmapped_fa'] for t in targets], normal=nfq if any(nfq) else None,
                                 k=k, rc_thresh=int(targets[0].params.get_sr_thresh('min')),
                                 names=[t.name for t in targets])
        pk.read_len[:len(targets)] = [t.read_len for t in targets]   # what get_fastq_reads returned (utils.py:236,246)
        return pk, [k] * len(targets), _LazyReads(pk)
    if ingest == "python":
        inputs = [_TargetInput(t) for t in targets]
        pk = batch.PackedBatch(inputs, rc_thresh=inputs[0].rc_thresh)
        pk.read_len = np.array([inp.read_len for inp in inputs] + [0], dtype=np.int32)
        return pk, [inp.k for inp in inputs], [o for inp in inputs for o in inp.objs]
    raise ValueError("ingest must be 'python' or 'native'")


def compare_kmers_batch(targets, device=0, ingest="python", write_contigs=False, devices=None, max_targets=125, inflight=4,
                        apply_thread=False, on_capacity="raise", report=None, rejected=None, kmer_report=None,
                        normal_kmers=None):
    """target.compare_kmers() for many targets (the region loop of sv_processor.py:185-201 as one call).

    The targets are cut into chunks of at most max_targets, most expensive first (static cost, breakmer_b200.shard), and
    the chunks are pipelined: `inflight` of them are kept on the device at once (bk_batch_submit / bk_batch_wait) so the
    serial tail of one chunk's assembly overlaps the bulk of the next.  With `devices=[0, 1, ...]` the chunks are handed
    out dynamically to one host thread per GPU (region sharding, no collective); results are applied to the target objects
    as chunks complete.

    `apply_thread=True` gives every device a second host thread that waits for the results and applies them to the
    target objects while the first one parses and submits the next chunks.  (Measured neutral on a 500-target panel,
    profiles/r2_experiments.md: a chunk's results arrive one assembly latency -- its longest region's chain, ~20 ms --
    after it was submitted, whatever its size, and applying them is GIL-bound Python; the option pays when parsing is
    the larger share, i.e. big inputs per target.)

    Targets that exceed a limit of the batched assembler (a read or contig above 4,095 bases) do not disturb the others.
    With on_capacity="raise" (default) everything else completes, then CapacityError lists them (their state is
    untouched).  With on_capacity="assemble" every call runs with the handles' "long_regions" option: such targets are
    assembled in the same device pass as the others (reads and contigs up to 65,535 bases), on the device that ran their
    chunk, and their results applied like every other target's (files included); CapacityError then lists only the
    targets beyond that limit.  CapacityError.reasons says why each of them was not completed.

    `report`, a dict, receives report[target.name] = batch.region_report's dict of the target, for every target, in every
    form (one call, chunked, apply_thread, devices=[...]).

    `rejected`, a dict, receives rejected[target.name] = the contigs the assembler grew for the target and then dropped
    in its acceptance test (sv_assembly.py:53-59: total read support below the min sr_thresh, or not longer than
    read_len), in growth order, as sv_assembly.contig objects with `.rejected_for` "support" or "length", for every
    target (an empty list for one not completed), in every form.  The handles' "rejected_contigs" option is set for the
    call only; the accepted contigs, the target state and the files are the same as without it.

    `kmer_report`, a dict, receives kmer_report[target.name] = batch.kmer_report's dict of the target: how many distinct
    soft-clip k-mers it had, and how many of them the reads lacked, the reference held, the normal sample held, and were
    left as sample-only k-mers.  `normal_kmers`, a dict, receives normal_kmers[target.name] = {mer: case count} of the
    k-mers the normal sample removed (files['normal_fq']; empty without one), the entries the sample-only file would
    have held without the normal sample.  Both are filled for every target, in every form; the handles' "normal_kmers"
    option is set for the call only, and the target state and the files are the same as without it."""
    if on_capacity not in ("raise", "assemble"):
        raise ValueError("on_capacity must be 'raise' or 'assemble'")
    if not targets:
        return
    if write_contigs and ingest != "native":
        raise ValueError("write_contigs needs ingest='native' (the writer reads the parsed record text)")
    if ingest not in ("python", "native"):
        raise ValueError("ingest must be 'python' or 'native'")
    failed, reasons = [], {}
    devices = list(devices) if devices else [device]
    long_regions = on_capacity == "assemble"
    if len(targets) <= max_targets and len(devices) == 1:
        pk, ks, objs = _pack_targets(targets, ingest)
        h = get_handle(devices[0])
        with batch.options([h], long_regions=long_regions, rejected_contigs=rejected is not None,
                           normal_kmers=normal_kmers is not None):
            res = batch.run(h, pk, decode=False)
            rows = batch.region_report_if(h, res, report is not None)
            if rejected is not None:
                res.rejected = batch.rejected_tables(h)
            if normal_kmers is not None:
                res.normal = batch.normal_kmer_tables(h)
            kr_rows = batch.kmer_report(h) if kmer_report is not None else None
        out = _apply_chunk(targets, pk, res, ks, objs, ingest, write_contigs, failed)
        if rejected is not None:
            _record_rejected(targets, out, objs, ks, rejected)
        _record_kmer_stage(targets, out, kr_rows, kmer_report, normal_kmers)
        _record_report(targets, rows, failed, reasons, report)
    else:
        _sharded(targets, devices, ingest, write_contigs, max_targets, inflight, failed, apply_thread, long_regions, reasons,
                 report, rejected, kmer_report, normal_kmers)
    if failed:
        raise CapacityError(sorted(failed), reasons)


_pipes = {}


def _get_pipe(dev, inflight):
    """The calling thread's DevicePipeline (its handles keep their arenas from call to call)."""
    import threading
    from . import shard
    key = (threading.get_ident(), dev, inflight)
    if key not in _pipes:
        _pipes[key] = shard.DevicePipeline(dev, inflight=inflight)
    return _pipes[key]


def _sharded(targets, devices, ingest, write_contigs, max_targets, inflight, failed, apply_thread=False, long_regions=False,
             reasons=None, report=None, rejected=None, kmer_report=None, normal_kmers=None):
    """Chunked, pipelined (and with several devices region-sharded) pass: sv_processor.py:185-201 over `devices`."""
    import threading
    from . import shard
    lock = threading.Lock()

    def pack(idx, slot):
        chunk = [targets[i] for i in idx]
        pk, ks, objs = _pack_targets(chunk, ingest, slot=slot)
        # the applying thread's writer: made here so that it is cached under the submitting thread's key
        apply_ing = _get_ingest("apply") if (apply_thread and ingest == "native") else None
        return pk, (chunk, ks, objs, apply_ing)

    def consume(res, pk, tag):
        chunk, ks, objs, apply_ing = tag
        mine = []
        out = _apply_chunk(chunk, pk, res, ks, objs, ingest, write_contigs, mine, apply_ing)
        with lock:
            failed.extend(mine)
            _record_report(chunk, getattr(res, "report", None), mine, reasons, report)
            if rejected is not None:
                _record_rejected(chunk, out, objs, ks, rejected)
            _record_kmer_stage(chunk, out, getattr(res, "kmer_report", None), kmer_report, normal_kmers)

    chunks = shard.plan_chunks([_target_cost(t) for t in targets], len(devices), max_targets,
                               key=lambda i: (targets[i].name, i))               # sv_processor.py:175-176
    # one device: the calling thread drives it, and its handles keep their arenas from call to call
    pipe = _get_pipe(devices[0], inflight) if len(devices) == 1 else None
    try:
        shard.drive_chunks(chunks, devices, inflight, pack, consume, pipe, decode=False, long_regions=long_regions,
                           report=report is not None, apply_thread=apply_thread, rejected_contigs=rejected is not None,
                           kmer_report=kmer_report is not None, normal_kmers=normal_kmers is not None)
    except Exception:
        if pipe is not None:                             # a pipeline with batches in flight is not reusable
            _pipes.pop((threading.get_ident(), devices[0], inflight), None)
            pipe.close()
        raise


def _target_cost(trgt):
    """Static cost of a target before the device pass: shard.region_cost's read terms on the number of distinct read
    sequences the target object already holds (O(1); the byte term needs file sizes and is left out)."""
    from . import shard
    recs = getattr(trgt, "cleaned_read_recs", None)
    n = len(recs) if recs else 0
    return shard.COST_CELLS_PER_READ2 * n * n + shard.COST_CELLS_PER_READ * n + 1.0


def compare_kmers(target, device=0, ingest="python"):
    compare_kmers_batch([target], device=device, ingest=ingest)
