"""The "rejected_contigs" option: the contigs the assembler grows and then drops in its acceptance test (Q21,
sv_assembly.py:53-59), with the reason, through every entry point (bk_rejected_contigs, BatchOutput.rejected_records,
the rejected= of the Python drop-ins), against the oracle; and the accepted contigs unchanged by it.

RejectingAssembler is the oracle with every contig Assembler.run grows and does not return recorded in growth order,
with the reason of its Q21 test (support is tested first)."""
import dataclasses
import filecmp
import os

import numpy as np
import pytest

from breakmer_b200 import synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only
from test_gpu_long_inline import MIX_READ_LEN, mixed_region
from test_gpu_long_regions import LONG_READ_REGIONS, _targets, over_limit_region

pytestmark = pytest.mark.gpu

# the calls that reject every contig: for support (no contig has that many reads), for length (read_len above every contig)
ALL_SUPPORT = 10 ** 6
ALL_LENGTH = 10000


class RejectingAssembler(assembler_py.Assembler):
    """Assembler that keeps the contigs run() grows and drops, with the reason of the Q21 test"""

    def _grow(self, ct):
        assembler_py.Assembler._grow(self, ct)
        self._grown.append(ct)

    def run(self):
        self._grown = []
        out = assembler_py.Assembler.run(self)
        kept = {id(ct) for ct in out}
        self.rejected = [("support" if ct.total_reads() < self.rc_thresh else "length", ct)
                         for ct in self._grown if id(ct) not in kept]
        return out


_ORACLE = {}


def oracle_rejected(region, read_len=None):
    """-> (accepted contig records, [(reason, contig record), ...] of the rejected ones) of the oracle for one region;
    cached by region name, rc_thresh and read_len"""
    read_len = region.read_len if read_len is None else read_len
    key = (region.name, region.k, region.rc_thresh, read_len)
    if key not in _ORACLE:
        _r, _c, _s, only = oracle_sample_only(region)
        reads = assembler_py.group_reads(region.reads)
        asm = RejectingAssembler(only, reads, region.k, region.rc_thresh, read_len)
        acc = [assembler_py.contig_record(ct, reads) for ct in asm.run()]
        _ORACLE[key] = (acc, [(why, assembler_py.contig_record(ct, reads)) for why, ct in asm.rejected])
    return _ORACLE[key]


def golden_regions():
    from conftest import golden
    out = []
    for c in golden("assembly_golden.json")["cases"][:24]:
        kw = dict(c["kwargs"]); kw["event"] = tuple(kw["event"])
        out.append(synth.make_region(c["name"], **kw))
    return out


def forced(regions, why):
    """the regions with every contig rejected for `why`: (regions, per-region read_len or None)"""
    if why == "support":
        return [dataclasses.replace(r, name=r.name + "_s", rc_thresh=ALL_SUPPORT) for r in regions], None
    return [dataclasses.replace(r, name=r.name + "_l") for r in regions], [ALL_LENGTH] * len(regions)


@pytest.fixture(scope="module")
def handle():
    from breakmer_b200 import _lib
    h = _lib.Handle(0)
    yield h
    h.close()


def packed(regions, read_len=None):
    from breakmer_b200 import batch
    pk = batch.PackedBatch(regions)
    if read_len is not None:
        pk.read_len = np.array(list(read_len) + [0], dtype=np.int32)
    return pk


def run(handle, pk, on=True, long_regions=False, long=False):
    """-> (BatchOutput, region_report rows) of one bk_compare_kmers_batch / _long call with the option `on`"""
    from breakmer_b200 import batch
    with batch.options([handle], long_regions=long_regions, rejected_contigs=on):
        out = batch.run(handle, pk, long=long)
        return out, batch.region_report(handle)


def check_regions(out, rows, regions, read_len=None):
    """every completed region's accepted and rejected contigs against the oracle, and the report's counts"""
    n_rej = 0
    for i, r in enumerate(regions):
        if out.region_status[i] != 0:
            assert out.rejected_records(i) == [], r.name
            continue
        acc, rej = oracle_rejected(r, None if read_len is None else read_len[i])
        assert out.contig_records(i) == acc, r.name
        assert out.rejected_records(i) == rej, r.name
        whys = [w for w, _rec in rej]
        assert (rows[i]["rejected_support"], rows[i]["rejected_length"]) == (whys.count("support"), whys.count("length")), r.name
        n_rej += len(rej)
    assert out.rej_reg_off[-1] == len(out.rej_reason) == n_rej
    return n_rej


def same_accepted(handle, pk, out_on, long_regions=False, long=False):
    """the accepted contigs (and everything else region_digests covers) equal those of the same call without the option"""
    from breakmer_b200 import shard
    out_off, _rows = run(handle, pk, on=False, long_regions=long_regions, long=long)
    assert out_off.rej_reg_off is None
    assert shard.region_digests(out_on, pk) == shard.region_digests(out_off, pk)
    assert out_on.n_contigs == out_off.n_contigs


@pytest.mark.parametrize("spec_width", [1, 2, 4, 8])
def test_rejected_contigs_match_the_oracle(handle, spec_width):
    by_k = {}
    for r in golden_regions():
        by_k.setdefault(r.k, []).append(r)
    groups = list(by_k.values()) + [list(synth.config_regions("C2", n=15, start=0))]
    handle.set_option("spec_width", spec_width)
    try:
        n_rej = 0
        for regions in groups:
            pk = packed(regions)
            out, rows = run(handle, pk)
            n_rej += check_regions(out, rows, regions)
            same_accepted(handle, pk, out)
        assert n_rej > 0
    finally:
        handle.set_option("spec_width", 0)


@pytest.mark.parametrize("why", ["support", "length"])
def test_every_contig_rejected_for_one_reason(handle, why):
    regions, read_len = forced(golden_regions()[:6] + list(synth.config_regions("C2", n=4, start=0)), why)
    regions = [r for r in regions if r.k == 15]
    pk = packed(regions, read_len)
    out, rows = run(handle, pk)
    assert out.n_contigs == 0
    assert check_regions(out, rows, regions, read_len) > 0
    # support is tested first: a contig below rc_thresh is rejected for support whatever read_len is
    reasons = set(out.rej_reason.tolist())
    assert reasons == {1} if why == "support" else 2 in reasons
    assert all(row["rejected_support"] + row["rejected_length"] == row["grown"] for row in rows)


def test_the_long_pass_keeps_only_its_own_attempt(handle):
    """the mixed region with every contig rejected for support: assemble_kernel grows and rejects the C2 contigs
    before the growing one stops it; those never appear, the long pass's do (once each, as the oracle has them)"""
    r = dataclasses.replace(mixed_region(), rc_thresh=ALL_SUPPORT)
    pk = packed([r], [MIX_READ_LEN])
    out, rows = run(handle, pk, long_regions=True)
    assert (rows[0]["pass"], rows[0]["first_reason"]) == ("long", "contig_too_long")
    assert check_regions(out, rows, [r], [MIX_READ_LEN]) > 0
    same_accepted(handle, pk, out, long_regions=True)


def test_the_long_entry(handle):
    regions = list(synth.config_regions("C2", n=4, start=0)) + [synth.make_region(LONG_READ_REGIONS[0][0], **LONG_READ_REGIONS[0][1])]
    pk = packed(regions)
    out, rows = run(handle, pk, long=True)
    assert all(row["pass"] == "long" for row in rows)
    assert check_regions(out, rows, regions) > 0
    same_accepted(handle, pk, out, long=True)


@pytest.mark.parametrize("mode", ["off", "route", "long"])
def test_a_region_left_out_at_upload_shifts_the_read_indices(handle, mode):
    """the left-out region comes first, so every other region's read indices are shifted back by its record"""
    from breakmer_b200 import batch
    regions, _ = forced([over_limit_region(batch.LONG_MAX_LEN + 1)] + list(synth.config_regions("C2", n=2, start=2)), "support")
    pk = packed(regions)
    out, rows = run(handle, pk, long_regions=mode == "route", long=mode == "long")
    assert out.region_status[0] != 0 and list(out.region_status[1:]) == [0, 0]
    assert out.rej_reg_off[1] == 0
    assert check_regions(out, rows, regions) > 0
    for i in (1, 2):
        a, b = int(out.rej_reg_off[i]), int(out.rej_reg_off[i + 1])
        for c in range(out.n_contigs + a, out.n_contigs + b):
            ro, nr = out.reads_off[c]
            assert ((out.reads[ro:ro + nr] >= pk.read_reg_off[i]) & (out.reads[ro:ro + nr] < pk.read_reg_off[i + 1])).all()


def test_submit_wait_and_resident(handle):
    """submit / wait honours the option; a resident batch keeps the mode it was uploaded with"""
    from breakmer_b200 import batch
    regions = list(synth.config_regions("C2", n=6, start=0))
    pk = packed(regions)
    one, rows = run(handle, pk)
    handle.set_option("rejected_contigs", 1)
    try:
        batch.submit(handle, pk)
        two = batch.wait(handle, pk)
        batch.upload(handle, pk)
    finally:
        handle.set_option("rejected_contigs", 0)
    three = batch.run(handle, pk, resident=True)
    check_regions(one, rows, regions)
    for o in (two, three):
        assert [o.rejected_records(i) for i in range(len(regions))] == [one.rejected_records(i) for i in range(len(regions))]
        assert [o.contig_records(i) for i in range(len(regions))] == [one.contig_records(i) for i in range(len(regions))]
    batch.upload(handle, pk)                                        # uploaded with the option off: none, even if set now
    handle.set_option("rejected_contigs", 1)
    try:
        four = batch.run(handle, pk, resident=True)
    finally:
        handle.set_option("rejected_contigs", 0)
    assert four.rej_reg_off is None and batch.rejected_tables(handle) is None


def test_the_getter_refuses():
    from breakmer_b200 import _lib, batch
    h = _lib.Handle(0)

    def refused():
        with pytest.raises(_lib.BreakmerError) as ei:
            h.rejected_contigs()
        return ei.value.code == _lib.BK_ERR_ARG

    try:
        assert refused()                                            # no result yet
        pk = packed([synth.config_region("C2", 3)])
        batch.run(h, pk)
        assert refused()                                            # a result made with the option off
        with batch.options([h], rejected_contigs=True):
            batch.submit(h, pk)
            assert refused()                                        # in flight
            batch.wait(h, pk)
        off, why = h.rejected_contigs()
        assert len(off) == 2 and off[-1] == len(why)
        h.count_kmers(["ACGTACGTACGTACGTACGT"], 15)                 # another call reuses the result's memory
        assert refused()
    finally:
        h.close()


def _contig_record(ct):
    return {"seq": ct.get_contig_seq(), "indel_only": ct.aseq.counts.indel_only, "others": ct.aseq.counts.others,
            "reads": sorted(rd.id for rd in ct.reads), "kmers": [list(t) for t in ct.kmers], "kmer_locs": ct.get_kmer_locs()}


def _tree(path):
    return sorted(os.path.relpath(os.path.join(dp, f), path) for dp, _dn, fns in os.walk(path) for f in fns)


@pytest.mark.parametrize("form", [dict(), dict(ingest="native", write_contigs=True), dict(max_targets=2),
                                  dict(ingest="native", write_contigs=True, max_targets=2, apply_thread=True),
                                  dict(devices=[0, 0])])
def test_compare_kmers_batch_rejected(tmp_path, form):
    from breakmer_b200 import get_handle, sv_processor
    on, off = _targets(tmp_path / "on"), _targets(tmp_path / "off")
    rejected = {}
    sv_processor.compare_kmers_batch([t for _r, t in on], on_capacity="assemble", rejected=rejected, **form)
    sv_processor.compare_kmers_batch([t for _r, t in off], on_capacity="assemble", **form)
    assert sorted(rejected) == sorted(t.name for _r, t in on)
    n_rej = 0
    for (r, t), (_r2, t2) in zip(on, off):
        acc, rej = oracle_rejected(r)
        assert [(c.rejected_for, _contig_record(c)) for c in rejected[t.name]] == rej, t.name
        assert [_contig_record(c) for c in t.kmers['clusters']] == [_contig_record(c) for c in t2.kmers['clusters']] == acc
        assert all(c.rejected_for is None for c in t.kmers['clusters'])
        n_rej += len(rej)
        # the hand-off files of the two runs are the same
        for sub in ("kmers", "contigs"):
            a, b = os.path.join(t.paths[sub]), os.path.join(t2.paths[sub])
            assert _tree(a) == _tree(b), t.name
            assert all(filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False) for f in _tree(a)), t.name
    assert n_rej > 0
    # CapacityError still names the target beyond the batched limit; the others' rejected contigs are still returned
    pairs = _targets(tmp_path / "raise")
    rejected = {}
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in pairs], rejected=rejected, **form)
    assert ei.value.targets == ["zz_long"] and ei.value.reasons == {"zz_long": "read_too_long"}
    assert rejected["zz_long"] == []
    assert [(c.rejected_for, _contig_record(c)) for c in rejected[pairs[0][1].name]] == oracle_rejected(pairs[0][0])[1]
    # the handles are back at the default: a later call without rejected= holds no rejected contigs
    from breakmer_b200 import batch
    h = get_handle(0)
    batch.run(h, packed([synth.config_region("C2", 1)]))
    assert batch.rejected_tables(h) is None


def test_init_assembly_batch_rejected():
    from breakmer_b200 import batch, get_handle, sv_assembly, utils
    calls, regions = [], []
    for name, kw in [("c2a", None), LONG_READ_REGIONS[0], ("c2b", None)]:
        r = synth.config_region("C2", 1 if name == "c2a" else 5) if kw is None else synth.make_region(name, **kw)
        _r, _c, _s, only = oracle_sample_only(r)
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        calls.append((only, recs, r.k, r.rc_thresh, r.read_len))
        regions.append(r)
    rejected = []
    with pytest.raises(RuntimeError) as ei:
        sv_assembly.init_assembly_batch(calls, rejected=rejected)
    assert ei.value.reasons == {1: "read_too_long"} and rejected[1] == []
    rejected = []
    got = sv_assembly.init_assembly_batch(calls, on_capacity="assemble", rejected=rejected)
    assert len(rejected) == len(calls)
    n_rej = 0
    for g, rej, r in zip(got, rejected, regions):
        acc, exp = oracle_rejected(r)
        assert [(c.rejected_for, _contig_record(c)) for c in rej] == exp, r.name
        assert [_contig_record(c) for c in g] == acc, r.name
        n_rej += len(rej)
    assert n_rej > 0
    h = get_handle(0)
    batch.run(h, packed([synth.config_region("C2", 1)]))
    assert batch.rejected_tables(h) is None
