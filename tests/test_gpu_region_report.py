"""The per-region report (bk_region_report, batch.region_report, the report= of the Python drop-ins): its counters
against the oracle's per region, the reason a region stopped in each mode, the same table through every entry point,
and CapacityError.reasons.

The oracle's stats dict counts seeds, find_reads and check_align; CountingAssembler adds the contigs Assembler.run grows
and, of those, the ones it does not return, split by the reason of its Q21 test.

Not produced here: BK_RR_KMER_LIST_FULL (a contig with more than 8,192 k-mer tuples), BK_RR_TOO_MANY_CONTIGS (2^20
contigs in one region) and BK_RR_OUTPUT_ARENA (contigs larger than 8 x the call's read bases, which the output arena's
retry then absorbs, so it can only appear as a first reason within an attempt that is redone): none is reached by an
input of test size."""
import pytest

from breakmer_b200 import synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only
from test_gpu_long_inline import MIX_READ_LEN, mixed_region
from test_gpu_long_regions import GROWING_REGION, LONG_READ_REGIONS, _targets, over_limit_region

pytestmark = pytest.mark.gpu

COUNTERS = ("seeds", "find_reads", "check_align", "grown", "rejected_support", "rejected_length")


class CountingAssembler(assembler_py.Assembler):
    """Assembler with the contigs it grows counted: every contig run() grows and does not return was rejected by the
    Q21 test (sv_assembly.py:53-59), which tests support first"""

    def _grow(self, ct):
        assembler_py.Assembler._grow(self, ct)
        self._grown.append(ct)

    def run(self):
        self._grown = []
        out = assembler_py.Assembler.run(self)
        kept = {id(ct) for ct in out}
        for ct in self._grown:
            self._bump("grown")
            if id(ct) not in kept:
                self._bump("rejected_support" if ct.total_reads() < self.rc_thresh else "rejected_length")
        return out


def oracle_report(region, read_len=None):
    """-> (contig records, {counter: value}) of the oracle for one region"""
    _r, _c, _s, only = oracle_sample_only(region)
    reads = assembler_py.group_reads(region.reads)
    stats = dict.fromkeys(COUNTERS, 0)
    asm = CountingAssembler(only, reads, region.k, region.rc_thresh, region.read_len if read_len is None else read_len,
                            stats=stats)
    ctgs = [assembler_py.contig_record(ct, reads) for ct in asm.run()]
    return ctgs, {k: stats[k] for k in COUNTERS}


def check_counters(row, region, n_contigs, read_len=None):
    ctgs, exp = oracle_report(region, read_len)
    assert {k: row[k] for k in COUNTERS} == exp, region.name
    assert n_contigs == len(ctgs), region.name
    assert row["grown"] == n_contigs + row["rejected_support"] + row["rejected_length"], region.name


def golden_regions():
    from conftest import golden
    out = []
    for c in golden("assembly_golden.json")["cases"][:24]:
        kw = dict(c["kwargs"]); kw["event"] = tuple(kw["event"])
        out.append(synth.make_region(c["name"], **kw))
    return out


@pytest.fixture(scope="module")
def handle():
    from breakmer_b200 import _lib
    h = _lib.Handle(0)
    yield h
    h.close()


def run_report(handle, regions, long_regions=False, long=False, read_len=None):
    import numpy as np
    from breakmer_b200 import batch
    pk = batch.PackedBatch(regions)
    if read_len is not None:
        pk.read_len = np.array(read_len + [0], dtype=np.int32)
    with batch.long_regions([handle], long_regions):
        out = batch.run(handle, pk, long=long)
        return out, batch.region_report(handle)


@pytest.mark.parametrize("spec_width", [1, 2, 4, 8])
def test_counters_match_the_oracle(handle, spec_width):
    by_k = {}
    for r in golden_regions():
        by_k.setdefault(r.k, []).append(r)
    groups = list(by_k.values()) + [list(synth.config_regions("C2", n=15, start=0))]
    handle.set_option("spec_width", spec_width)
    try:
        for regions in groups:
            out, rows = run_report(handle, regions)
            assert len(rows) == len(regions)
            assert sum(row["check_align"] for row in rows) == out.n_check_align
            for i, (r, row) in enumerate(zip(regions, rows)):
                assert (row["reason"], row["pass"], row["first_reason"]) == ("ok", "batched", "ok"), r.name
                check_counters(row, r, int(out.ctg_reg_off[i + 1] - out.ctg_reg_off[i]))
    finally:
        handle.set_option("spec_width", 0)


def test_reasons_of_a_long_read(handle):
    r = synth.make_region(LONG_READ_REGIONS[0][0], **LONG_READ_REGIONS[0][1])
    c2 = synth.config_region("C2", 1)
    out, rows = run_report(handle, [c2, r])
    assert list(out.region_status) == [0, -4]
    assert rows[1] == dict(reason="read_too_long", first_reason="ok", **{"pass": "none"}, **dict.fromkeys(COUNTERS, 0))
    assert (rows[0]["reason"], rows[0]["pass"]) == ("ok", "batched")
    out, rows = run_report(handle, [c2, r], long_regions=True)
    assert list(out.region_status) == [0, 0]
    assert (rows[1]["reason"], rows[1]["pass"], rows[1]["first_reason"]) == ("ok", "long", "read_too_long")
    assert (rows[0]["reason"], rows[0]["pass"], rows[0]["first_reason"]) == ("ok", "batched", "ok")
    for i, reg in enumerate([c2, r]):
        check_counters(rows[i], reg, int(out.ctg_reg_off[i + 1] - out.ctg_reg_off[i]))


def test_reasons_of_a_growing_contig(handle):
    r = synth.make_region(*GROWING_REGION[:1], **GROWING_REGION[1])
    out, rows = run_report(handle, [r])
    assert list(out.region_status) == [-4]
    assert (rows[0]["reason"], rows[0]["pass"], rows[0]["first_reason"]) == ("contig_too_long", "batched", "ok")
    out, rows = run_report(handle, [r], long_regions=True)
    assert list(out.region_status) == [0]
    assert (rows[0]["reason"], rows[0]["pass"], rows[0]["first_reason"]) == ("ok", "long", "contig_too_long")
    check_counters(rows[0], r, int(out.ctg_reg_off[1]))


def test_the_abandoned_attempt_is_not_counted(handle):
    """the mixed region: assemble_kernel accepts contigs before the growing one stops it; the long pass starts over"""
    r = mixed_region()
    out, rows = run_report(handle, [r], long_regions=True, read_len=[MIX_READ_LEN])
    assert (rows[0]["reason"], rows[0]["pass"], rows[0]["first_reason"]) == ("ok", "long", "contig_too_long")
    check_counters(rows[0], r, int(out.ctg_reg_off[1]), read_len=MIX_READ_LEN)


@pytest.mark.parametrize("mode", ["off", "route", "long"])
def test_a_read_beyond_every_limit(handle, mode):
    from breakmer_b200 import batch
    c2 = synth.config_region("C2", 2)
    over = over_limit_region(batch.LONG_MAX_LEN + 1)
    out, rows = run_report(handle, [over, c2], long_regions=mode == "route", long=mode == "long")
    assert list(out.region_status) == [-4, 0]
    assert (rows[0]["reason"], rows[0]["pass"], rows[0]["first_reason"]) == ("read_too_long", "none", "ok")
    assert rows[1]["reason"] == "ok" and rows[1]["pass"] == ("long" if mode == "long" else "batched")
    check_counters(rows[1], c2, int(out.ctg_reg_off[2] - out.ctg_reg_off[1]))


def test_the_long_entry(handle):
    regions = list(synth.config_regions("C2", n=4, start=0)) + [synth.make_region(LONG_READ_REGIONS[0][0], **LONG_READ_REGIONS[0][1]),
                                                               synth.make_region(*GROWING_REGION[:1], **GROWING_REGION[1])]
    out, rows = run_report(handle, regions, long=True)
    assert sum(row["check_align"] for row in rows) == out.n_check_align
    for i, (r, row) in enumerate(zip(regions, rows)):
        assert (row["reason"], row["pass"], row["first_reason"]) == ("ok", "long", "ok"), r.name
        check_counters(row, r, int(out.ctg_reg_off[i + 1] - out.ctg_reg_off[i]))


def test_every_entry_point_gives_the_same_table(handle):
    from breakmer_b200 import batch
    regions = list(synth.config_regions("C2", n=6, start=0)) + [synth.make_region(*GROWING_REGION[:1], **GROWING_REGION[1])]
    pk = batch.PackedBatch(regions)
    with batch.long_regions([handle]):
        batch.run(handle, pk)
        one = handle.region_report()
        batch.submit(handle, pk)
        batch.wait(handle, pk)
        two = handle.region_report()
        batch.upload(handle, pk)
        batch.run(handle, pk, resident=True)
        three = handle.region_report()
    assert one.shape == (len(regions), len(batch.REPORT_FIELDS))
    assert (one == two).all() and (one == three).all()
    assert one[-1].tolist()[:3] == [0, 2, 2]                     # ok, long pass, first reason contig_too_long


def test_the_getter_refuses_while_a_batch_is_in_flight():
    from breakmer_b200 import _lib, batch
    h = _lib.Handle(0)
    try:
        with pytest.raises(_lib.BreakmerError) as ei:          # no result yet
            h.region_report()
        assert ei.value.code == _lib.BK_ERR_ARG
        pk = batch.PackedBatch([synth.config_region("C2", 3)])
        batch.submit(h, pk)
        with pytest.raises(_lib.BreakmerError) as ei:
            h.region_report()
        assert ei.value.code == _lib.BK_ERR_ARG
        batch.wait(h, pk)
        assert h.region_report()[0, 0] == 0
        h.count_kmers(["ACGTACGTACGTACGTACGT"], 15)             # another call reuses the result's memory
        with pytest.raises(_lib.BreakmerError) as ei:
            h.region_report()
        assert ei.value.code == _lib.BK_ERR_ARG
    finally:
        h.close()


@pytest.mark.parametrize("form", [dict(), dict(max_targets=2), dict(max_targets=2, apply_thread=True), dict(devices=[0, 0])])
def test_compare_kmers_batch_report(tmp_path, form):
    from breakmer_b200 import sv_processor
    pairs = _targets(tmp_path / "a")
    report = {}
    sv_processor.compare_kmers_batch([t for _r, t in pairs], on_capacity="assemble", report=report, **form)
    assert sorted(report) == sorted(t.name for _r, t in pairs)
    for r, t in pairs:
        row = report[t.name]
        assert row["reason"] == "ok"
        assert row["pass"] == ("long" if t.name == "zz_long" else "batched")
        check_counters(row, r, len(t.kmers['clusters']))
    pairs = _targets(tmp_path / "b")
    report = {}
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in pairs], report=report, **form)
    assert ei.value.targets == ["zz_long"]
    assert ei.value.reasons == {"zz_long": "read_too_long"}
    assert report["zz_long"]["pass"] == "none" and len(report) == len(pairs)


def test_capacity_error_reasons_without_a_report(tmp_path):
    from breakmer_b200 import sv_processor
    pairs = _targets(tmp_path)
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in pairs], max_targets=2)
    assert ei.value.reasons == {"zz_long": "read_too_long"}


def test_init_assembly_batch_report():
    from breakmer_b200 import sv_assembly, utils
    calls, regions = [], []
    for name, kw in [("c2", None), LONG_READ_REGIONS[0], GROWING_REGION]:
        r = synth.config_region("C2", 1) if kw is None else synth.make_region(name, **kw)
        _r, _c, _s, only = oracle_sample_only(r)
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        calls.append((only, recs, r.k, r.rc_thresh, r.read_len))
        regions.append(r)
    report = []
    with pytest.raises(RuntimeError) as ei:
        sv_assembly.init_assembly_batch(calls, report=report)
    assert ei.value.reasons == {1: "read_too_long", 2: "contig_too_long"}
    assert [row["reason"] for row in report] == ["ok", "read_too_long", "contig_too_long"]
    report = []
    got = sv_assembly.init_assembly_batch(calls, on_capacity="assemble", report=report)
    assert [row["pass"] for row in report] == ["batched", "long", "long"]
    for g, r, row in zip(got, regions, report):
        check_counters(row, r, len(g))
