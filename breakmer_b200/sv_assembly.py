"""Drop-in for the reference's sv_assembly.init_assembly, running on the GPU.

    init_assembly(mers, fq_recs, kmer_len, rc_thresh, read_len) -> [contig]

keeps the reference signature (sv_assembly.py:30).  The returned objects carry
what the downstream code reads from a reference contig (SURVEY.md section 3.5,
sv_processor.py:731-746, sv_caller.py:159,242,271-277,634):

    .reads            set of the representative fq_read of each unique read
    .kmers            list of (mer, pos, less_than_half, dist_half, order) tuples
    .kmer_locs / get_kmer_locs()
    .aseq.seq / get_contig_seq()
    .aseq.counts / get_contig_counts()  with .indel_only, .others,
                      get_counts(p1, p2, sv_type), get_total_reads()
    get_total_read_support(), get_contig_len(), .kmer_len

The reference mutates its inputs while it runs (`fq_recs` loses keys, reads get
`.used = True`); the caller drops both right after the call
(sv_processor.py:643) and nothing downstream looks at them, so those mutations
are not replayed (SURVEY.md section 8.3).
"""
from . import batch, get_handle


class assembly_counts:
    """Result view of the reference class of the same name (sv_assembly.py:160-221)."""

    def __init__(self, indel_only, others):
        self.indel_only = list(indel_only)
        self.others = list(others)

    def get_counts(self, p1, p2, sv_type):                       # sv_assembly.py:167-176
        if sv_type == 'indel' or sv_type == 'rearr':
            if p1 == p2:
                return self.indel_only[p1] + self.others[p1]
            return [x + y for x, y in zip(self.indel_only[p1:p2], self.others[p1:p2])]
        if p1 == p2:
            return self.others[p1]
        return self.others[p1:p2]

    def get_total_reads(self):                                   # sv_assembly.py:178-179
        return max(self.indel_only) + max(self.others)


class assembly_seq:
    def __init__(self, seq, counts):
        self.seq = seq
        self.counts = counts


class _lazy(object):
    """Non-data descriptor: computes the attribute on first read and stores it on the instance (so it can also be
    assigned like a plain attribute, which the reference's downstream code is free to do)."""

    def __init__(self, fn):
        self.fn = fn
        self.name = fn.__name__

    def __get__(self, obj, owner=None):
        if obj is None:
            return self
        v = obj.__dict__[self.name] = self.fn(obj)
        return v


class contig:
    """What the rest of BreaKmer reads from an sv_assembly.contig (SURVEY.md section 3.5).  The Python lists, tuples and
    fq_read objects are built from the batch's result arrays on FIRST ACCESS of each attribute: resolve_sv touches few of
    them per contig, and building all of them eagerly costs 12x the device time of the batch."""

    def __init__(self, out, cidx, objs, kmer_len, rec=None):
        self._out = out
        self._c = int(cidx)
        self._objs = objs
        self.kmer_len = kmer_len
        self.setup = True
        if rec is not None:                                       # eager construction from a decoded record
            self.__dict__["reads"] = set(objs)
            self.__dict__["aseq"] = assembly_seq(rec["seq"], assembly_counts(rec["indel_only"], rec["others"]))
            self.__dict__["kmer_locs"] = list(rec["kmer_locs"])
            self.__dict__["kmers"] = [tuple(t) for t in rec["kmers"]]

    @_lazy
    def reads(self):
        o = self._out
        ro, nr = o.reads_off[self._c]
        objs = self._objs
        return set(objs[int(r)] for r in o.reads[ro:ro + nr])

    @_lazy
    def aseq(self):
        o = self._out
        so, sl = o.seq_off[self._c]
        co, cl = o.cnt_off[self._c]
        return assembly_seq(o.seq[so:so + sl].tobytes().decode(),
                            assembly_counts(o.indel_only[co:co + cl].tolist(), o.others[co:co + cl].tolist()))

    @_lazy
    def kmer_locs(self):
        o = self._out
        so, sl = o.seq_off[self._c]
        return o.kmer_locs[so:so + sl].tolist()

    @_lazy
    def kmers(self):
        o = self._out
        ko, nk = o.kmers_off[self._c]
        from . import _lib
        from .batch import ORDER_NAMES
        mers = _lib.codes_to_mers(o.kmer_mer[ko:ko + nk], o.k)
        return list(zip(mers, o.kmer_pos[ko:ko + nk].tolist(), o.kmer_lth[ko:ko + nk].tolist(),
                        o.kmer_dist[ko:ko + nk].tolist(), [ORDER_NAMES[x] for x in o.kmer_order[ko:ko + nk].tolist()]))

    def get_total_read_support(self):
        o = self._out
        if "aseq" not in self.__dict__ and o is not None:         # straight from the arrays
            co, cl = o.cnt_off[self._c]
            return int(o.indel_only[co:co + cl].max()) + int(o.others[co:co + cl].max())
        return self.aseq.counts.get_total_reads()

    def get_contig_len(self):
        if "aseq" not in self.__dict__ and self._out is not None:
            return int(self._out.seq_off[self._c][1])
        return len(self.aseq.seq)

    def get_kmer_locs(self):
        return self.kmer_locs

    def get_contig_seq(self):
        return self.aseq.seq

    def get_contig_counts(self):
        return self.aseq.counts


def _filled(name):
    def method(self, *a, **kw):
        self._fill()
        return getattr(list, name)(self, *a, **kw)
    method.__name__ = name
    return method


class contig_list(list):
    """kmers['clusters'] of one target: a list of `contig` objects that are created when the list is first looked at
    (len() and truth value come straight from the result tables).  A panel batch returns thousands of contigs; building
    every Python object eagerly costs more than the device pass."""

    def __init__(self, out, c0, c1, objs, kmer_len):
        list.__init__(self)
        self._pending = (out, int(c0), int(c1), objs, kmer_len)

    def _fill(self):
        if self._pending is not None:
            out, c0, c1, objs, k = self._pending
            self._pending = None
            list.extend(self, [contig(out, c, objs, k) for c in range(c0, c1)])

    def __len__(self):
        if self._pending is not None:
            return self._pending[2] - self._pending[1]
        return list.__len__(self)

    def __bool__(self):
        return len(self) > 0

    def __reduce__(self):
        self._fill()
        return (list, (list(self),))

    __iter__ = _filled("__iter__")
    __getitem__ = _filled("__getitem__")
    __setitem__ = _filled("__setitem__")
    __delitem__ = _filled("__delitem__")
    __contains__ = _filled("__contains__")
    __reversed__ = _filled("__reversed__")
    __eq__ = _filled("__eq__")
    __ne__ = _filled("__ne__")
    __add__ = _filled("__add__")
    __iadd__ = _filled("__iadd__")
    __mul__ = _filled("__mul__")
    __repr__ = _filled("__repr__")
    __hash__ = None
    append = _filled("append")
    extend = _filled("extend")
    insert = _filled("insert")
    pop = _filled("pop")
    remove = _filled("remove")
    index = _filled("index")
    count = _filled("count")
    sort = _filled("sort")
    reverse = _filled("reverse")
    copy = _filled("copy")
    clear = _filled("clear")


class _AssemblyInput:
    """Region-like view of one init_assembly call for batch.PackedBatch."""

    def __init__(self, name, fq_recs, kmer_len, rc_thresh):
        self.name = name
        self.k = int(kmer_len)
        self.rc_thresh = int(rc_thresh)
        self.ref_fwd = ""
        self.sc_records = []
        self.normal_reads = []
        self.reads = []
        self.objs = []
        for seq, group in fq_recs.items():                       # insertion order == fq_recs order (Q9 policy)
            for fr in group:
                self.reads.append((fr.id, fr.seq, fr.qual, bool(fr.indel_only)))
                self.objs.append(fr)


def _clean_mers(mers, kmer_len):
    """The reference takes any {str: int}: a mer that is not kmer_len upper-case ACGT characters can never be found in a
    read by str.find on upper-case reads... except that it CAN if reads hold the same odd characters.  Those exotic mers
    are not representable in the 2-bit table, so they are rejected loudly rather than silently dropped."""
    for m in mers:
        if len(m) != kmer_len:
            raise ValueError("init_assembly: mer %r does not have kmer_len=%d characters" % (m, kmer_len))
        if m.strip("ACGT"):
            raise ValueError("init_assembly: mer %r holds characters other than upper-case A, C, G, T" % (m,))
    return mers


def _assemble_calls(calls, device, long_regions, want_report=False):
    """One device pass over `calls` -> (contig list or None per call, indices of the calls reported BK_ERR_CAPACITY,
    batch.region_report of the pass or None).  long_regions: the pass also assembles calls with reads or contigs up to
    65,535 bases (the handle's option of that name, set for this call only).  The report is read when want_report or
    when a call was not completed."""
    import numpy as np
    inputs = [_AssemblyInput("r%d" % i, c[1], c[2], c[3]) for i, c in enumerate(calls)]
    pk = batch.PackedBatch(inputs, rc_thresh=int(calls[0][3]))
    pk.set_mers([_clean_mers(c[0], int(c[2])) for c in calls])
    pk.read_len = np.array([int(c[4]) for c in calls] + [0], dtype=np.int32)
    h = get_handle(device)
    with batch.long_regions([h], long_regions):
        out = batch.run(h, pk)
        rows = batch.region_report_if(h, out, want_report)
    objs = [o for inp in inputs for o in inp.objs]
    result = []
    bad = []
    for i, c in enumerate(calls):
        if out.region_status[i] != 0:
            bad.append(i)
            result.append(None)
            continue
        result.append([contig(out, cidx, objs, int(c[2])) for cidx in range(int(out.ctg_reg_off[i]), int(out.ctg_reg_off[i + 1]))])
    return result, bad, rows


def init_assembly_batch(calls, device=0, on_capacity="raise", report=None):
    """calls: [(mers, fq_recs, kmer_len, rc_thresh, read_len), ...] with one common
    kmer_len and rc_thresh -> list (per call) of contig lists.  One GPU pass.

    A call whose region exceeds a limit of the batched assembler (a read or contig longer than 4095 bases) does not
    disturb the others.  on_capacity says what happens to it:
      "raise" (default)  a RuntimeError naming those calls is raised after every other call was completed, the results
                         stored in the exception's `.results`;
      "none"             their entry in the returned list is None;
      "assemble"         the same pass assembles them too (the handle's "long_regions" option: reads and contigs up
                         to 65,535 bases); a RuntimeError as with "raise" names the calls that exceed that limit.
    The RuntimeError's `.reasons` says why each of those calls was not completed ({call index: reason name}, see
    batch.REASONS).  `report`, a list, is extended with batch.region_report's dict of every call, in call order: why it
    stopped, which pass assembled it, and what the assembler did."""
    if not calls:
        return []
    result, bad, rows = _assemble_calls(calls, device, on_capacity == "assemble", report is not None)
    if report is not None:
        report.extend(rows)
    limit = 65535 if on_capacity == "assemble" else 4095
    if bad and on_capacity in ("raise", "assemble"):
        err = RuntimeError("init_assembly: device capacity exceeded in call(s) %s (a read or contig longer than %d bases); "
                           "the other calls completed (see .results)" % (bad, limit))
        err.results = result
        err.reasons = {i: rows[i]["reason"] for i in bad}
        raise err
    return result


def init_assembly(mers, fq_recs, kmer_len, rc_thresh, read_len):
    if len(mers) == 0:                                           # sv_assembly.py:33-34
        return []
    return init_assembly_batch([(mers, fq_recs, kmer_len, rc_thresh, read_len)])[0]
