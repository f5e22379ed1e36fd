"""ctypes binding of the C ABI in include/breakmer_b200.h.

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a)
as breakmer_b200/lib/libbreakmer_b200.so.  There is no fallback of any kind: if
the library is missing, or no CUDA device is present, the call raises.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_double, c_int, c_int32, c_int64, c_uint8, c_uint32,
                    c_uint64, c_void_p)

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# BK_LIB: explicit path of another BUILD of the same library (instrumented builds of tools/, the test-only emulator build of
# tests/sim).  Never chosen automatically: unset, only the in-tree CUDA library is loaded, and load() raises without it.
LIB_PATH = os.environ.get("BK_LIB") or os.path.join(_HERE, "lib", "libbreakmer_b200.so")

BK_OK = 0
BK_ERR_CUDA = -1
BK_ERR_ARG = -2
BK_ERR_NOMEM = -3
BK_ERR_CAPACITY = -4
BK_ERR_EMPTY_SEQ = -5
BK_ERR_FORMAT = -6
BK_ERR_IO = -7


class BreakmerError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "breakmer_b200 error %d: %s" % (code, msg))
        self.code = code


class BatchInput(Structure):
    _fields_ = [
        ("n_regions", c_int32), ("k", c_int32), ("rc_thresh", c_int32), ("have_mers", c_int32),
        ("ref_bases", c_void_p), ("ref_off", c_void_p),
        ("read_bases", c_void_p), ("read_off", c_void_p), ("read_reg_off", c_void_p), ("read_flags", c_void_p),
        ("sc_bases", c_void_p), ("sc_off", c_void_p), ("sc_reg_off", c_void_p),
        ("normal_bases", c_void_p), ("normal_off", c_void_p), ("normal_reg_off", c_void_p),
        ("in_mers", c_void_p), ("in_counts", c_void_p), ("in_mers_off", c_void_p),
        ("read_len", c_void_p),
    ]


class BatchResult(Structure):
    _fields_ = [
        ("n_regions", c_int32), ("n_contigs", c_int64),
        ("so_off", POINTER(c_int64)), ("so_mers", POINTER(c_uint64)), ("so_counts", POINTER(c_uint32)),
        ("uniq_reg_off", POINTER(c_int64)), ("uniq_rec", POINTER(c_int32)), ("uniq_mult", POINTER(c_uint32)),
        ("ctg_reg_off", POINTER(c_int64)),
        ("ctg_seq_off", POINTER(c_int64)), ("ctg_seq", POINTER(c_uint8)), ("ctg_kmer_locs", POINTER(c_int32)),
        ("ctg_cnt_off", POINTER(c_int64)), ("ctg_indel_only", POINTER(c_int32)), ("ctg_others", POINTER(c_int32)),
        ("ctg_reads_off", POINTER(c_int64)), ("ctg_reads", POINTER(c_int32)),
        ("ctg_kmers_off", POINTER(c_int64)), ("ctg_kmer_mer", POINTER(c_uint64)), ("ctg_kmer_pos", POINTER(c_int32)),
        ("ctg_kmer_lth", POINTER(c_int32)), ("ctg_kmer_dist", POINTER(c_int32)), ("ctg_kmer_order", POINTER(c_int32)),
        ("region_status", POINTER(c_int32)),
        ("n_check_align", c_int64), ("n_dp_cells", c_int64), ("n_kmer_occurrences", c_int64),
        ("gpu_ms", c_double),
        ("n_sorted_keys", c_int64),
        ("region_dp_cells", POINTER(c_int64)),
        ("host_wait_ms", c_double), ("host_post_ms", c_double),
    ]


class Text(Structure):
    _fields_ = [("p", c_void_p), ("n", c_int64)]


class IngestText(Structure):
    _fields_ = [("id_bytes", POINTER(c_uint8)), ("id_off", POINTER(c_int64)),
                ("qual_bytes", POINTER(c_uint8)), ("qual_off", POINTER(c_int64)),
                ("n_reads", c_int64), ("read_flags", POINTER(c_uint8))]


_lib = None


def load():
    """Load the CUDA library; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "breakmer_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    H = c_void_p
    lib.bk_version.restype = c_int
    lib.bk_device_count.restype = c_int
    lib.bk_create.argtypes = [c_int, POINTER(H)]
    lib.bk_destroy.argtypes = [H]
    lib.bk_last_error.argtypes = [H]
    lib.bk_last_error.restype = c_char_p
    lib.bk_nw_batch.argtypes = [H, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int,
                                c_void_p, c_void_p, c_void_p, c_void_p]
    lib.bk_dedup_reads.argtypes = [H, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_double, c_void_p,
                                   c_void_p, POINTER(c_int64), POINTER(c_int32)]
    lib.bk_count_kmers.argtypes = [H, c_void_p, c_void_p, c_int64, c_void_p, c_int,
                                   POINTER(POINTER(c_uint64)), POINTER(POINTER(c_uint32)), POINTER(c_int64)]
    lib.bk_sample_only.argtypes = [H, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                                   c_void_p, c_int64,
                                   POINTER(POINTER(c_uint64)), POINTER(POINTER(c_uint32)), POINTER(c_int64)]
    lib.bk_compare_kmers_batch.argtypes = [H, POINTER(BatchInput), POINTER(BatchResult)]
    lib.bk_compare_kmers_long.argtypes = [H, POINTER(BatchInput), POINTER(BatchResult)]
    lib.bk_batch_submit.argtypes = [H, POINTER(BatchInput)]
    lib.bk_batch_wait.argtypes = [H, POINTER(BatchResult)]
    lib.bk_batch_upload.argtypes = [H, POINTER(BatchInput)]
    lib.bk_compare_kmers_resident.argtypes = [H, POINTER(BatchResult)]
    lib.bk_kernel_times.argtypes = [H, POINTER(c_char_p), POINTER(POINTER(c_double)), POINTER(POINTER(c_int64)),
                                    POINTER(c_int32)]
    lib.bk_kernel_times_reset.argtypes = [H, c_int]
    lib.bk_set_option.argtypes = [H, c_char_p, c_int64]
    lib.bk_ref_cache_build.argtypes = [H, c_void_p, c_void_p, c_int32, c_int32]
    lib.bk_ref_cache_clear.argtypes = [H]
    lib.bk_region_report.argtypes = [H, POINTER(POINTER(c_int32)), POINTER(c_int32)]
    lib.bk_ingest_create.argtypes = [c_int, c_int, POINTER(H)]
    lib.bk_ingest_destroy.argtypes = [H]
    lib.bk_ingest_last_error.argtypes = [H]
    lib.bk_ingest_last_error.restype = c_char_p
    lib.bk_ingest_buffers.argtypes = [H, c_int32, POINTER(Text), POINTER(Text), POINTER(Text), POINTER(Text),
                                      POINTER(BatchInput), POINTER(IngestText)]
    lib.bk_ingest_files.argtypes = [H, c_int32, POINTER(c_char_p), POINTER(c_char_p), POINTER(c_char_p),
                                    POINTER(c_char_p), POINTER(BatchInput), POINTER(IngestText)]
    lib.bk_write_contigs.argtypes = [H, POINTER(BatchResult), POINTER(BatchInput), POINTER(IngestText),
                                     POINTER(c_char_p), POINTER(c_char_p), POINTER(c_int64)]
    lib.bk_write_sample_kmers.argtypes = [H, POINTER(BatchResult), c_int32, POINTER(c_char_p), POINTER(c_int64)]
    for name in ("bk_ingest_create", "bk_ingest_destroy", "bk_ingest_buffers", "bk_ingest_files", "bk_write_contigs",
                 "bk_write_sample_kmers"):
        getattr(lib, name).restype = c_int
    for name in ("bk_create", "bk_destroy", "bk_nw_batch", "bk_dedup_reads", "bk_count_kmers", "bk_sample_only",
                 "bk_compare_kmers_batch", "bk_compare_kmers_long", "bk_batch_submit", "bk_batch_wait", "bk_batch_upload",
                 "bk_compare_kmers_resident", "bk_kernel_times", "bk_kernel_times_reset", "bk_set_option", "bk_ref_cache_build",
                 "bk_ref_cache_clear", "bk_region_report"):
        getattr(lib, name).restype = c_int
    _lib = lib
    return lib


EXPORTED_SYMBOLS = (
    "bk_version", "bk_device_count", "bk_create", "bk_destroy", "bk_last_error", "bk_nw_batch", "bk_dedup_reads",
    "bk_count_kmers", "bk_sample_only", "bk_compare_kmers_batch", "bk_compare_kmers_long", "bk_batch_submit", "bk_batch_wait", "bk_batch_upload", "bk_compare_kmers_resident", "bk_kernel_times",
    "bk_kernel_times_reset", "bk_set_option", "bk_ref_cache_build", "bk_ref_cache_clear", "bk_region_report",
    "bk_ingest_create", "bk_ingest_destroy", "bk_ingest_last_error", "bk_ingest_buffers", "bk_ingest_files",
    "bk_write_contigs", "bk_write_sample_kmers")


def _ptr(a):
    return None if a is None else a.ctypes.data_as(c_void_p)


def concat(seqs):
    """list of str/bytes -> (uint8 array, int64 offsets[n+1])."""
    if not isinstance(seqs, (list, tuple)):
        seqs = list(seqs)
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if not seqs:
        return np.zeros(0, dtype=np.uint8), off
    try:
        joined = "".join(seqs).encode()                  # all str (the usual case): one join, one encode
        np.cumsum(np.fromiter(map(len, seqs), dtype=np.int64, count=len(seqs)), out=off[1:])
        if len(joined) != off[-1]:                       # a non-ASCII character: byte lengths differ, do it per record
            raise TypeError
    except TypeError:
        bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
        np.cumsum([len(b) for b in bs], out=off[1:])
        joined = b"".join(bs)
    data = np.frombuffer(joined, dtype=np.uint8) if joined else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(data), off


class Handle:
    """One CUDA device + one stream (bk_create / bk_destroy)."""

    def __init__(self, device=0):
        self.lib = load()
        self.h = c_void_p()
        rc = self.lib.bk_create(int(device), byref(self.h))
        if rc != BK_OK:
            raise BreakmerError(rc, "bk_create(device=%d) failed: no usable CUDA device (there is no CPU fallback)"
                                % device)
        self.device = device
        self.result_regions = None         # n_regions of the handle's last result (batch.run / batch.wait set it)

    def close(self):
        if self.h:
            self.lib.bk_destroy(self.h)
            self.h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != BK_OK:
            raise BreakmerError(rc, self.lib.bk_last_error(self.h).decode())

    # ---- olc.nw -----------------------------------------------------------------
    def nw_batch(self, seqs, pair_a, pair_b, want_aln=False):
        data, off = concat(seqs)
        pa = np.ascontiguousarray(pair_a, dtype=np.int32)
        pb = np.ascontiguousarray(pair_b, dtype=np.int32)
        n = len(pa)
        out = np.zeros((n, 10), dtype=np.int32)
        if want_aln:
            lens = (off[1:] - off[:-1])
            cap = lens[pa] + lens[pb]
            aoff = np.zeros(n + 1, dtype=np.int64)
            np.cumsum(cap, out=aoff[1:])
            a1 = np.zeros(int(aoff[-1]) + 1, dtype=np.uint8)
            a2 = np.zeros(int(aoff[-1]) + 1, dtype=np.uint8)
            alen = np.zeros(n, dtype=np.int32)
            self._check(self.lib.bk_nw_batch(self.h, _ptr(data), _ptr(off), len(seqs), _ptr(pa), _ptr(pb), n,
                                             _ptr(out), 1, _ptr(a1), _ptr(a2), _ptr(aoff), _ptr(alen)))
            alns = [(a1[aoff[i]:aoff[i] + alen[i]].tobytes().decode(), a2[aoff[i]:aoff[i] + alen[i]].tobytes().decode())
                    for i in range(n)]
            return out, alns
        self._check(self.lib.bk_nw_batch(self.h, _ptr(data), _ptr(off), len(seqs), _ptr(pa), _ptr(pb), n, _ptr(out),
                                         0, None, None, None, None))
        return out, None

    # ---- read_batch.check_mer_read over whole batches (sv_assembly_mm2.py:290-355) ----
    def dedup_reads(self, seqs, mer_pos, batch_off, subseq_frac):
        """-> (check uint8[n], flags uint8[n], number of alignments computed)"""
        data, off = concat(seqs)
        n = len(seqs)
        mp = np.ascontiguousarray(mer_pos, dtype=np.int32)
        bo = np.ascontiguousarray(batch_off, dtype=np.int64)
        if len(mp) != n:
            raise ValueError("dedup_reads: one mer_pos per read")
        check = np.zeros(n, dtype=np.uint8)
        flags = np.zeros(n, dtype=np.uint8)
        n_pairs, n_launches = c_int64(), c_int32()
        self._check(self.lib.bk_dedup_reads(self.h, _ptr(data), _ptr(off), n, _ptr(mp), _ptr(bo), len(bo) - 1,
                                            float(subseq_frac), _ptr(check), _ptr(flags), byref(n_pairs),
                                            byref(n_launches)))
        self.last_dedup_launches = n_launches.value
        return check, flags, n_pairs.value

    # ---- jellyfish count + dump + load_kmers ----------------------------------------
    def count_kmers(self, seqs, k, mult=None):
        data, off = concat(seqs)
        m = None if mult is None else np.ascontiguousarray(mult, dtype=np.uint32)
        pm, pc, n = POINTER(c_uint64)(), POINTER(c_uint32)(), c_int64()
        self._check(self.lib.bk_count_kmers(self.h, _ptr(data), _ptr(off), len(seqs), _ptr(m), int(k),
                                            byref(pm), byref(pc), byref(n)))
        if n.value == 0:
            return np.zeros(0, np.uint64), np.zeros(0, np.uint32)
        return (np.ctypeslib.as_array(pm, shape=(n.value,)).copy(), np.ctypeslib.as_array(pc, shape=(n.value,)).copy())

    def sample_only(self, k, case, sc_mers, ref_mers, normal_mers=None):
        cm = np.ascontiguousarray(case[0], dtype=np.uint64)
        cc = np.ascontiguousarray(case[1], dtype=np.uint32)
        sm = np.ascontiguousarray(sc_mers, dtype=np.uint64)
        rm = np.ascontiguousarray(ref_mers, dtype=np.uint64)
        nm = None if normal_mers is None else np.ascontiguousarray(normal_mers, dtype=np.uint64)
        pm, pc, n = POINTER(c_uint64)(), POINTER(c_uint32)(), c_int64()
        self._check(self.lib.bk_sample_only(self.h, int(k), _ptr(cm), _ptr(cc), len(cm), _ptr(sm), len(sm), _ptr(rm),
                                            len(rm), _ptr(nm), 0 if nm is None else len(nm),
                                            byref(pm), byref(pc), byref(n)))
        if n.value == 0:
            return np.zeros(0, np.uint64), np.zeros(0, np.uint32)
        return (np.ctypeslib.as_array(pm, shape=(n.value,)).copy(), np.ctypeslib.as_array(pc, shape=(n.value,)).copy())

    def ref_cache_build(self, ref_seqs, k):
        data, off = concat(ref_seqs)
        self._check(self.lib.bk_ref_cache_build(self.h, _ptr(data), _ptr(off), len(ref_seqs), int(k)))

    def ref_cache_clear(self):
        self._check(self.lib.bk_ref_cache_clear(self.h))

    def set_option(self, name, value):
        self._check(self.lib.bk_set_option(self.h, name.encode(), int(value)))

    def region_report(self):
        """bk_region_report: the per-region report of the handle's last result (batch.run / batch.wait), as an
        (n_regions, BK_RR_FIELDS) int32 copy.  Read it before the handle's next call."""
        table, nf = POINTER(c_int32)(), c_int32()
        self._check(self.lib.bk_region_report(self.h, byref(table), byref(nf)))
        n = self.result_regions
        if n is None:                      # a result the library holds but this object did not see (no row count)
            raise BreakmerError(BK_ERR_ARG, "region_report: no result of batch.run / batch.wait on this handle")
        if n == 0:
            return np.zeros((0, nf.value), np.int32)
        return np.ctypeslib.as_array(table, shape=(int(n), nf.value)).copy()

    # ---- timers -------------------------------------------------------------------------
    def kernel_times_reset(self, enable=True):
        self._check(self.lib.bk_kernel_times_reset(self.h, 1 if enable else 0))

    def kernel_times(self):
        names, ms, ln, n = c_char_p(), POINTER(c_double)(), POINTER(c_int64)(), c_int32()
        self._check(self.lib.bk_kernel_times(self.h, byref(names), byref(ms), byref(ln), byref(n)))
        ns = names.value.decode().split(";")
        return {ns[i]: (ms[i], ln[i]) for i in range(n.value)}


_CODE = {"A": 0, "C": 1, "G": 2, "T": 3}
_BASES = "ACGT"


def mer_to_code(mer):
    v = 0
    for c in mer:
        v = (v << 2) | _CODE[c]
    return v


def code_to_mer(code, k):
    code = int(code)
    return "".join(_BASES[(code >> (2 * (k - 1 - i))) & 3] for i in range(k))


_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def codes_to_mers(codes, k):
    """Vectorised code_to_mer: uint64 array -> list of str (first base most significant)."""
    codes = np.ascontiguousarray(codes, dtype=np.uint64)
    if codes.size == 0:
        return []
    shifts = (2 * (k - 1 - np.arange(k))).astype(np.uint64)
    letters = _ACGT[((codes[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.intp)]
    return np.ascontiguousarray(letters).view("S%d" % k).ravel().astype("U%d" % k).tolist()
