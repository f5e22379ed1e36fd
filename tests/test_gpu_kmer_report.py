"""The k-mer stage's per-region report (bk_kmer_report) and the "normal_kmers" option (bk_normal_kmers) against the
oracle breakdown of tests/test_oracle_kmer_report.py, through every entry point: bk_compare_kmers_batch, submit / wait,
the resident form, bk_compare_kmers_long, the "long_regions" pass, the reference k-mer cache, and the Python drop-ins."""
import dataclasses

import numpy as np
import pytest

from breakmer_b200 import _lib, batch, shard, synth
from conftest import golden
from test_gpu_long_regions import LONG_READ_REGIONS, _Target, over_limit_region
from test_oracle_kmer_report import region_breakdown

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle():
    h = _lib.Handle(0)
    yield h
    h.close()


def golden_kmer_regions():
    out = []
    for case in golden("kmers_golden.json")["cases"]:
        kw = dict(case["kwargs"]); kw["event"] = tuple(kw["event"])
        out.append(synth.make_region(case["name"], **kw))
    return out


def with_foreign_clips(region, i=0):
    """the region with two more soft-clip records whose k-mers no read holds (BK_KR_NOT_IN_READS)"""
    extra = [("x%d" % i, ("ACGGTCATTGCAAGTC" * 4)[i % 7:]), ("y%d" % i, "GATTACAGATTACCCATTAGGA")]
    return dataclasses.replace(region, name=region.name + "_x", sc_records=list(region.sc_records) + extra)


def check_report(h, regions, pk, out=None, skipped=()):
    """bk_kmer_report of the handle's last result == the oracle breakdown of every region (an all-zero row for the
    regions left out at upload); with `out`, sample_only agrees with the result's sample-only table"""
    rows = batch.kmer_report(h)
    assert len(rows) == len(regions)
    for i, (r, row) in enumerate(zip(regions, rows)):
        if i in skipped:
            assert row == dict.fromkeys(batch.KMER_REPORT_FIELDS, 0), r.name
            continue
        exp, _removed = region_breakdown(r, with_normal=pk.has_normal)
        assert row == exp, (r.name, row, exp)
        if out is not None:
            assert row["sample_only"] == len(out.sample_only(i)), r.name
    return rows


def check_normal(regions, out, pk):
    """the result's normal k-mers == the oracle's, ascending, with case counts"""
    off, mers, counts = out.normal
    assert len(off) == len(regions) + 1
    for i, r in enumerate(regions):
        a, b = int(off[i]), int(off[i + 1])
        assert np.all(mers[a + 1:b] > mers[a:b - 1]), r.name
        _row, removed = region_breakdown(r, with_normal=pk.has_normal)
        assert out.normal_kmers(i) == removed, r.name
    return int(off[-1])


def run_with(h, pk, **opts):
    with batch.options([h], **opts):
        return batch.run(h, pk)


def test_report_on_the_golden_regions_every_k(handle):
    regions = golden_kmer_regions()
    ks = sorted({r.k for r in regions})
    assert len(ks) > 1
    for k in ks:
        regs = [r for r in regions if r.k == k]
        regs = regs + [with_foreign_clips(regs[0])]
        pk = batch.PackedBatch(regs)
        out = batch.run(handle, pk)
        rows = check_report(handle, regs, pk, out)
        assert rows[-1]["not_in_reads"] > 0


@pytest.mark.parametrize("cfg,n,start", [("C2", 12, 0), ("C3", 12, 0), ("C4", 4, 0), ("C5", 60, 100)])
def test_report_on_the_configs(handle, cfg, n, start):
    regions = list(synth.config_regions(cfg, n=n, start=start))
    pk = batch.PackedBatch(regions)
    out = batch.run(handle, pk)
    rows = check_report(handle, regions, pk, out)
    if cfg == "C3":
        assert pk.has_normal and any(row["in_normal"] > 0 for row in rows)
    if cfg == "C4":                               # at least one region's table is a slice of the global table
        assert max(sum(len(s) for _n, s in r.sc_records) for r in regions) >= 16384


def test_report_with_the_reference_cache():
    regions = list(synth.config_regions("C3", n=6))
    h = _lib.Handle(0)
    try:
        h.ref_cache_build([r.ref_fwd for r in regions], regions[0].k)
        pk = batch.PackedBatch(regions, with_ref=False)
        out = run_with(h, pk, normal_kmers=True)
        check_report(h, regions, pk, out)
        assert check_normal(regions, out, pk) > 0
    finally:
        h.close()


def test_edge_regions(handle):
    base = synth.config_region("C2", 2)
    no_reads = dataclasses.replace(base, name="no_reads", reads=[])
    no_clips = dataclasses.replace(base, name="no_clips", sc_records=[])
    regions = [no_reads, no_clips, over_limit_region(5000), base]
    pk = batch.PackedBatch(regions)
    out = batch.run(handle, pk)
    assert out.region_status[2] != 0
    rows = check_report(handle, regions, pk, out, skipped=(2,))
    assert rows[0]["soft_clip"] == rows[0]["not_in_reads"] > 0
    assert rows[1] == dict.fromkeys(batch.KMER_REPORT_FIELDS, 0)
    # a batch without a single read base: the k-mer stage still counts the candidates
    pk = batch.PackedBatch([no_reads])
    batch.run(handle, pk)
    check_report(handle, [no_reads], pk)


def test_refusals(handle):
    h = _lib.Handle(0)
    try:
        with pytest.raises(_lib.BreakmerError):
            h.kmer_report()                                          # before any result
        regions = list(synth.config_regions("C3", n=3))
        pk = batch.PackedBatch(regions)
        batch.run(h, pk)
        assert batch.normal_kmer_tables(h) is None                   # the option was off
        with pytest.raises(_lib.BreakmerError):
            h.normal_kmers()
        h.set_option("normal_kmers", 1)
        batch.submit(h, pk)
        for get in (h.kmer_report, h.normal_kmers):                  # a batch in flight
            with pytest.raises(_lib.BreakmerError):
                get()
        batch.wait(h, pk)
        h.kmer_report(); h.normal_kmers()
        h.ref_cache_build([r.ref_fwd for r in regions], regions[0].k)   # reuses the result's memory
        for get in (h.kmer_report, h.normal_kmers):
            with pytest.raises(_lib.BreakmerError):
                get()
        with pytest.raises(_lib.BreakmerError):
            h.set_option("normal_kmers", 2)
        # have_mers: no k-mer stage ran
        r = regions[0]
        pm = batch.PackedBatch([r])
        pm.set_mers([region_breakdown(r)[1] or {"A" * r.k: 3}])
        batch.run(h, pm)
        for get in (h.kmer_report, h.normal_kmers):
            with pytest.raises(_lib.BreakmerError) as e:
                get()
            assert e.value.code == _lib.BK_ERR_ARG
    finally:
        h.close()


def _same_outputs(a, b, pk):
    assert shard.region_digests(a, pk) == shard.region_digests(b, pk)
    for name in ("so_off", "so_mers", "so_counts", "uniq_reg_off", "uniq_rec", "uniq_mult", "ctg_reg_off", "region_status"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    for r in range(a.n_regions):                # (the contig payload arrays are in device completion order: compare records)
        assert a.contig_records(r) == b.contig_records(r), r


def test_normal_kmers_against_the_oracle_and_without_the_normal(handle):
    regions = list(synth.config_regions("C3", n=16))
    pk = batch.PackedBatch(regions)
    off = batch.run(handle, pk)
    rep_off = batch.region_report(handle)
    kr_off = batch.kmer_report(handle)
    on = run_with(handle, pk, normal_kmers=True)
    assert check_normal(regions, on, pk) > 0
    _same_outputs(off, on, pk)                                       # every other output is the same with the option on
    assert batch.region_report(handle) == rep_off and batch.kmer_report(handle) == kr_off
    rows = batch.kmer_report(handle)
    bare = batch.PackedBatch(regions, with_normal=False)
    without = batch.run(handle, bare)
    for i, r in enumerate(regions):
        so, nm = on.sample_only(i), on.normal_kmers(i)
        assert not set(so) & set(nm)
        assert {**so, **nm} == without.sample_only(i), r.name
        assert len(nm) == rows[i]["in_normal"]


def test_normal_kmers_option_is_read_at_upload():
    regions = list(synth.config_regions("C3", n=4))
    pk = batch.PackedBatch(regions)
    h = _lib.Handle(0)
    try:
        h.set_option("normal_kmers", 1)
        batch.submit(h, pk)
        h.set_option("normal_kmers", 0)
        out = batch.wait(h, pk)
        assert out.normal is not None and check_normal(regions, out, pk) > 0
        batch.submit(h, pk)
        h.set_option("normal_kmers", 1)
        assert batch.wait(h, pk).normal is None
        # the resident form keeps the mode of its upload
        batch.upload(h, pk)                                          # (uploaded with the option on)
        h.set_option("normal_kmers", 0)
        out = batch.run(h, pk, resident=True)
        check_report(h, regions, pk, out)
        assert check_normal(regions, out, pk) > 0
    finally:
        h.close()


def test_normal_kmers_in_the_long_forms(handle):
    regions = list(synth.config_regions("C3", n=3)) + [synth.make_region("lr0", **dict(LONG_READ_REGIONS)["lr0"])]
    pk = batch.PackedBatch(regions)
    with batch.options([handle], normal_kmers=True):
        out = batch.run(handle, pk, long=True)
        check_report(handle, regions, pk, out)
        assert check_normal(regions, out, pk) > 0
        with batch.options([handle], long_regions=True):
            out = batch.run(handle, pk)
        assert list(out.region_status) == [0] * len(regions)
        check_report(handle, regions, pk, out)
        assert check_normal(regions, out, pk) > 0


def _c3_targets(tmp_path, n=5):
    from breakmer_b200 import utils
    out = []
    for r in synth.config_regions("C3", n=n):
        d = tmp_path / r.name
        for sub in ("kmers", "contigs"):
            (d / sub).mkdir(parents=True)
        (d / "ref.fa").write_text(">%s\n%s\n" % (r.name, r.ref_fwd))
        (d / "reads.fastq").write_text("".join("%s\n%s\n+\n%s\n" % (rid, seq, q) for rid, seq, q, _io in r.reads))
        (d / "sc.fa").write_text("".join(">%s\n%s\n" % (nm, s) for nm, s in r.sc_records))
        (d / "normal.fastq").write_text("".join("@n%d\n%s\n+\n%s\n" % (j, s, "I" * len(s)) for j, (_n, s) in enumerate(r.normal_reads)))
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        t = _Target(r, recs, str(d / "ref.fa"), str(d / "reads.fastq"), str(d / "sc.fa"), str(d))
        t.files['normal_fq'] = str(d / "normal.fastq")
        out.append((r, t))
    return out


@pytest.mark.parametrize("ingest", ["python", "native"])
@pytest.mark.parametrize("form", ["one_call", "chunked", "apply_thread", "devices"])
def test_dropin_fills_both_dicts(tmp_path, ingest, form):
    from breakmer_b200 import get_handle, sv_processor
    pairs = _c3_targets(tmp_path / "on")
    plain = _c3_targets(tmp_path / "off")
    kw = {"one_call": {}, "chunked": dict(max_targets=2), "apply_thread": dict(max_targets=2, apply_thread=True),
          "devices": dict(devices=[0], max_targets=2)}[form]
    kr, nm = {}, {}
    sv_processor.compare_kmers_batch([t for _r, t in pairs], ingest=ingest, kmer_report=kr, normal_kmers=nm, **kw)
    sv_processor.compare_kmers_batch([t for _r, t in plain], ingest=ingest, **kw)
    assert sorted(kr) == sorted(nm) == sorted(r.name for r, _t in pairs)
    for (r, t), (_r2, t2) in zip(pairs, plain):
        row, removed = region_breakdown(r)
        assert kr[r.name] == row
        assert nm[r.name] == removed
        with open(t.files['sample_kmers']) as a, open(t2.files['sample_kmers']) as b:
            assert a.read() == b.read()                                # target state and files are unchanged
        assert len(t.kmers['clusters']) == len(t2.kmers['clusters'])
    assert any(nm.values())
    # the handles went back to option 0
    handles = [get_handle(0)] + [h for pipe in sv_processor._pipes.values() for h in pipe.handles]
    pk = batch.PackedBatch([pairs[0][0]])
    for h in handles:
        batch.run(h, pk)
        assert batch.normal_kmer_tables(h) is None
