"""Marshalling between Python objects and the batched C-ABI entry point
bk_compare_kmers_batch (include/breakmer_b200.h).

`pack_regions` turns a list of region-like objects (anything with the attributes
of breakmer_b200.synth.Region: k, ref_fwd, reads, sc_records, normal_reads) into
the concatenated host arrays the ABI takes; `run` calls the library; `BatchOutput`
gives per-region views of the result in the reference's own shapes
({mer: count} dicts, contig records).
"""
import ctypes

import numpy as np

from . import _lib

ORDER_NAMES = ("for", "rev", "mid")
MAX_LEN = 4095             # longest read / contig of bk_compare_kmers_batch's assembler
LONG_MAX_LEN = 65535       # ... and of bk_compare_kmers_long's (run(..., long=True))


def _concat(seqs):
    return _lib.concat(seqs)


class PackedBatch:
    """Host arrays of one batch (kept alive for the duration of the calls)."""

    def __init__(self, regions, rc_thresh=None, with_normal=None, with_ref=True):
        self.n = len(regions)
        ks = {r.k for r in regions}
        if len(ks) > 1:
            raise ValueError("one k per batch")
        self.k = ks.pop() if ks else 15
        self.rc_thresh = int(rc_thresh if rc_thresh is not None else (regions[0].rc_thresh if regions else 2))
        self.names = [getattr(r, "name", str(i)) for i, r in enumerate(regions)]
        self.with_ref = with_ref          # False: the handle's reference k-mer cache is used (Handle.ref_cache_build)
        self.ref_bases, self.ref_off = _concat([r.ref_fwd for r in regions] if with_ref else [])
        reads, sc, normal = [], [], []
        self.read_reg_off = np.zeros(self.n + 1, np.int64)
        self.sc_reg_off = np.zeros(self.n + 1, np.int64)
        self.normal_reg_off = np.zeros(self.n + 1, np.int64)
        flags = []
        self.read_ids = []
        for i, r in enumerate(regions):
            for rec in r.reads:
                self.read_ids.append(rec[0])
                reads.append(rec[1])
                flags.append(1 if rec[3] else 0)
            sc.extend(rec[1] for rec in r.sc_records)
            normal.extend(rec[1] for rec in getattr(r, "normal_reads", ()))
            self.read_reg_off[i + 1] = len(reads)
            self.sc_reg_off[i + 1] = len(sc)
            self.normal_reg_off[i + 1] = len(normal)
        self.read_bases, self.read_off = _concat(reads)
        self.read_flags = np.array(flags, dtype=np.uint8) if flags else np.zeros(1, np.uint8)
        self.sc_bases, self.sc_off = _concat(sc)
        use_normal = (len(normal) > 0) if with_normal is None else with_normal
        self.has_normal = use_normal
        self.normal_bases, self.normal_off = _concat(normal)
        self.input_bytes = int(self.ref_bases.size + self.read_bases.size + self.sc_bases.size + self.normal_bases.size)
        self.in_mers = self.in_counts = self.in_mers_off = None
        self.read_len = None

    def pin(self):
        """Move the host arrays to page-locked memory (through torch, which is only plumbing here) so that the
        library's host->device copies are true asynchronous DMA transfers."""
        import torch
        for name in ("ref_bases", "ref_off", "read_bases", "read_off", "read_reg_off", "read_flags", "sc_bases", "sc_off",
                     "sc_reg_off", "normal_bases", "normal_off", "normal_reg_off", "in_mers", "in_counts", "in_mers_off",
                     "read_len"):
            a = getattr(self, name)
            if a is not None and a.size:
                setattr(self, name, torch.from_numpy(np.array(a, copy=True)).pin_memory().numpy())
        return self

    def set_mers(self, per_region_mers):
        """init_assembly shape: give each region's sample-only {mer: count} instead of
        running the k-mer stage."""
        mers, counts = [], []
        off = np.zeros(self.n + 1, np.int64)
        for i, d in enumerate(per_region_mers):
            items = sorted((_lib.mer_to_code(m), int(c)) for m, c in d.items())
            mers.extend(m for m, _ in items)
            counts.extend(c for _, c in items)
            off[i + 1] = len(mers)
        self.in_mers = np.array(mers + [0], dtype=np.uint64)
        self.in_counts = np.array(counts + [0], dtype=np.uint32)
        self.in_mers_off = off

    def struct(self):
        p = _lib._ptr
        s = _lib.BatchInput()
        s.n_regions = self.n
        s.k = self.k
        s.rc_thresh = self.rc_thresh
        s.have_mers = 1 if self.in_mers is not None else 0
        if self.with_ref:
            s.ref_bases, s.ref_off = p(self.ref_bases), p(self.ref_off)
        s.read_bases, s.read_off = p(self.read_bases), p(self.read_off)
        s.read_reg_off, s.read_flags = p(self.read_reg_off), p(self.read_flags)
        s.sc_bases, s.sc_off, s.sc_reg_off = p(self.sc_bases), p(self.sc_off), p(self.sc_reg_off)
        if self.has_normal:
            s.normal_bases, s.normal_off, s.normal_reg_off = p(self.normal_bases), p(self.normal_off), p(self.normal_reg_off)
        if self.in_mers is not None:
            s.in_mers, s.in_counts, s.in_mers_off = p(self.in_mers), p(self.in_counts), p(self.in_mers_off)
        if self.read_len is not None:
            s.read_len = p(self.read_len)
        return s


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)


class BatchOutput:
    """Copies of the library-owned result arrays of one call."""

    def __init__(self, res, packed):
        R = res.n_regions
        C = int(res.n_contigs)
        self.k = packed.k
        self._kmer_str = None
        self.n_regions = R
        self.n_contigs = C
        self._packed = packed                 # read ids are decoded only if somebody asks (contig_records)
        self.so_off = _arr(res.so_off, R + 1, np.int64)
        S = int(self.so_off[-1]) if R >= 0 and len(self.so_off) else 0
        self.so_mers = _arr(res.so_mers, S, np.uint64)
        self.so_counts = _arr(res.so_counts, S, np.uint32)
        self.uniq_reg_off = _arr(res.uniq_reg_off, R + 1, np.int64)
        NU = int(self.uniq_reg_off[-1]) if len(self.uniq_reg_off) else 0
        self.uniq_rec = _arr(res.uniq_rec, NU, np.int32)
        self.uniq_mult = _arr(res.uniq_mult, NU, np.uint32)
        self.ctg_reg_off = _arr(res.ctg_reg_off, R + 1, np.int64)
        self.seq_off = _arr(res.ctg_seq_off, 2 * C, np.int64).reshape(C, 2)
        self.cnt_off = _arr(res.ctg_cnt_off, 2 * C, np.int64).reshape(C, 2)
        self.reads_off = _arr(res.ctg_reads_off, 2 * C, np.int64).reshape(C, 2)
        self.kmers_off = _arr(res.ctg_kmers_off, 2 * C, np.int64).reshape(C, 2)
        n_seq = int((self.seq_off[:, 0] + self.seq_off[:, 1]).max()) if C else 0
        n_cnt = int((self.cnt_off[:, 0] + self.cnt_off[:, 1]).max()) if C else 0
        n_rd = int((self.reads_off[:, 0] + self.reads_off[:, 1]).max()) if C else 0
        n_km = int((self.kmers_off[:, 0] + self.kmers_off[:, 1]).max()) if C else 0
        self.seq = _arr(ctypes.cast(res.ctg_seq, ctypes.POINTER(ctypes.c_uint8)), n_seq, np.uint8)
        self.kmer_locs = _arr(res.ctg_kmer_locs, n_seq, np.int32)
        self.indel_only = _arr(res.ctg_indel_only, n_cnt, np.int32)
        self.others = _arr(res.ctg_others, n_cnt, np.int32)
        self.reads = _arr(res.ctg_reads, n_rd, np.int32)
        self.kmer_mer = _arr(res.ctg_kmer_mer, n_km, np.uint64)
        self.kmer_pos = _arr(res.ctg_kmer_pos, n_km, np.int32)
        self.kmer_lth = _arr(res.ctg_kmer_lth, n_km, np.int32)
        self.kmer_dist = _arr(res.ctg_kmer_dist, n_km, np.int32)
        self.kmer_order = _arr(res.ctg_kmer_order, n_km, np.int32)
        self.region_status = _arr(res.region_status, R, np.int32)
        self.region_dp_cells = _arr(res.region_dp_cells, R, np.int64)
        self.n_check_align = int(res.n_check_align)
        self.n_dp_cells = int(res.n_dp_cells)
        self.n_kmer_occurrences = int(res.n_kmer_occurrences)
        self.gpu_ms = float(res.gpu_ms)

    @property
    def read_ids(self):
        return self._packed.read_ids

    def sample_only(self, r):
        a, b = int(self.so_off[r]), int(self.so_off[r + 1])
        return dict(zip(_lib.codes_to_mers(self.so_mers[a:b], self.k), self.so_counts[a:b].tolist()))

    def _kmer_strings(self):
        if self._kmer_str is None:                      # all contig k-mers of the batch decoded at once
            self._kmer_str = _lib.codes_to_mers(self.kmer_mer, self.k)
        return self._kmer_str

    def contig_records(self, r, with_reads=True):
        """Contigs of region r in acceptance order, in the canonical comparable form
        (same shape as oracle.assembler_py.contig_record).  with_reads=False leaves "reads" out (callers that map
        ctg_reads to their own read objects do not need the sorted id list)."""
        out = []
        for c in range(int(self.ctg_reg_off[r]), int(self.ctg_reg_off[r + 1])):
            so, sl = self.seq_off[c]
            co, cl = self.cnt_off[c]
            ro, nr = self.reads_off[c]
            ko, nk = self.kmers_off[c]
            ks = self._kmer_strings()
            kmers = [list(t) for t in zip(ks[ko:ko + nk], self.kmer_pos[ko:ko + nk].tolist(), self.kmer_lth[ko:ko + nk].tolist(),
                                          self.kmer_dist[ko:ko + nk].tolist(),
                                          [ORDER_NAMES[o] for o in self.kmer_order[ko:ko + nk].tolist()])]
            out.append({
                "seq": self.seq[so:so + sl].tobytes().decode(),
                "indel_only": self.indel_only[co:co + cl].tolist(),
                "others": self.others[co:co + cl].tolist(),
                "reads": sorted(self.read_ids[int(i)] for i in self.reads[ro:ro + nr]) if with_reads else None,
                "kmers": kmers,
                "kmer_locs": self.kmer_locs[so:so + sl].tolist(),
            })
        return out


def run(handle, packed, resident=False, decode=True, long=False):
    """bk_compare_kmers_batch (or the resident variant after `upload`).  long=True: bk_compare_kmers_long, for regions
    with reads or contigs above MAX_LEN (up to LONG_MAX_LEN) bases, which the batched call reports as BK_ERR_CAPACITY."""
    res = _lib.BatchResult()
    if long:
        if resident:
            raise ValueError("the long entry takes its inputs in the call (no resident form)")
        s = packed.struct()
        handle._check(handle.lib.bk_compare_kmers_long(handle.h, ctypes.byref(s), ctypes.byref(res)))
    elif resident:
        handle._check(handle.lib.bk_compare_kmers_resident(handle.h, ctypes.byref(res)))
    else:
        s = packed.struct()
        handle._check(handle.lib.bk_compare_kmers_batch(handle.h, ctypes.byref(s), ctypes.byref(res)))
    if not decode:
        return res
    return BatchOutput(res, packed)


def submit(handle, packed=None):
    """bk_batch_submit: enqueue the device pass of `packed` (None: the batch uploaded with `upload`) and return.
    `packed` must stay alive until `wait` has returned."""
    if packed is None:
        handle._check(handle.lib.bk_batch_submit(handle.h, None))
    else:
        s = packed.struct()
        handle._check(handle.lib.bk_batch_submit(handle.h, ctypes.byref(s)))


def wait(handle, packed=None, decode=True):
    """bk_batch_wait: block until the submitted batch is done; BatchResult, or BatchOutput if decode."""
    res = _lib.BatchResult()
    handle._check(handle.lib.bk_batch_wait(handle.h, ctypes.byref(res)))
    if not decode:
        return res
    return BatchOutput(res, packed)


def upload(handle, packed):
    s = packed.struct()
    handle._check(handle.lib.bk_batch_upload(handle.h, ctypes.byref(s)))
