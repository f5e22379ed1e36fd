"""The "long_regions" option of the batched entries: regions with reads or contigs above 4,095 bases (up to 65,535) are
assembled in the same device pass as all others (assemble_kernel, then route_long_kernel and assemble_long_kernel on
the device queue), in every form: bk_compare_kmers_batch, bk_batch_submit / bk_batch_wait, bk_batch_upload +
bk_compare_kmers_resident, and the Python drop-ins' on_capacity="assemble"."""
import dataclasses
import functools

import pytest

from breakmer_b200 import synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only
from test_gpu_long_regions import GROWING_REGION, LONG_READ_REGIONS, _check_targets, _targets, oracle_region, over_limit_region

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle():
    from breakmer_b200 import _lib
    h = _lib.Handle(0)
    yield h
    h.close()


@functools.lru_cache(maxsize=None)
def _oracle(name, k):
    if name == "mix":
        r = _region(name, k)
        _r, _c, _s, only = oracle_sample_only(r)
        return only, assembler_py.init_assembly(only, r.reads, r.k, r.rc_thresh, MIX_READ_LEN)
    return oracle_region(_region(name, k))


@functools.lru_cache(maxsize=None)
def _region(name, k):
    if name == "over":
        return dataclasses.replace(over_limit_region(65536), k=k)
    if name.startswith("C2_"):
        r = synth.config_region("C2", int(name[3:]))
        return r if k == r.k else dataclasses.replace(r, k=k)
    if name == GROWING_REGION[0]:
        return synth.make_region(name, **GROWING_REGION[1])
    if name == "mix":
        return mixed_region()
    return synth.make_region(name, **dict(LONG_READ_REGIONS)[name])


def mixed_names(k):
    """test 1's call at k: 20 C2 regions (3 at k = 21), the long-read regions of that k, the growing region (k = 15) and
    a region with a read of 65,536 bases, last"""
    names = ["C2_%05d" % i for i in range(20 if k == 15 else 3)]
    names += [n for n, kw in LONG_READ_REGIONS if kw["k"] == k]
    if k == GROWING_REGION[1]["k"]:
        names.append(GROWING_REGION[0])
    return names + ["over"]


def mixed_regions(k):
    return [_region(n, k) for n in mixed_names(k)]


# the read length the mixed region is assembled with (the C2 reads'; a contig is kept only if it is longer)
MIX_READ_LEN = 100


def mixed_region():
    """the reads and reference of a C2 region at 200x and those of GROWING_REGION (60x) as one region: the C2 seeds
    come first, so with a read length of MIX_READ_LEN assemble_kernel emits their contigs before the growing contig stops
    it"""
    c2 = synth.config_region("C2", 1)
    g = synth.make_region(*GROWING_REGION[:1], **GROWING_REGION[1])
    reads = c2.reads + [("@G" + rid[1:], seq, q, io) for rid, seq, q, io in g.reads]
    return synth.Region(name="mix", k=15, ref_fwd=c2.ref_fwd + g.ref_fwd, reads=reads, sc_records=c2.sc_records + g.sc_records)


def check_mixed(out, regions, k):
    from breakmer_b200 import _lib
    for i, r in enumerate(regions):
        if r.name == "zz_over":
            assert out.region_status[i] == _lib.BK_ERR_CAPACITY
            assert out.contig_records(i) == []
            continue
        only, ctg = _oracle(r.name, k)
        assert out.region_status[i] == 0, r.name
        assert out.sample_only(i) == only, r.name
        assert out.contig_records(i) == ctg, r.name


@pytest.mark.parametrize("spec_width", [1, 2, 4, 8])
@pytest.mark.parametrize("k", [15, 21])
def test_mixed_call(handle, k, spec_width):
    from breakmer_b200 import batch
    regions = mixed_regions(k)
    handle.set_option("spec_width", spec_width)
    handle.set_option("long_regions", 1)
    try:
        out = batch.run(handle, batch.PackedBatch(regions))
    finally:
        handle.set_option("long_regions", 0)
        handle.set_option("spec_width", 0)
    check_mixed(out, regions, k)


def test_nothing_changes_for_normal_calls(handle):
    from conftest import golden
    from breakmer_b200 import batch
    import numpy as np
    by_k = {}
    for c in golden("assembly_golden.json")["cases"][:24]:
        kw = dict(c["kwargs"]); kw["event"] = tuple(kw["event"])
        by_k.setdefault(kw["k"], []).append(synth.make_region(c["name"], **kw))
    groups = list(by_k.values()) + [list(synth.config_regions("C2", n=15, start=0)), list(synth.config_regions("C5", n=15, start=0))]
    for regions in groups:
        pk = batch.PackedBatch(regions)
        a = batch.run(handle, pk)
        handle.set_option("long_regions", 1)
        try:
            b = batch.run(handle, pk)
        finally:
            handle.set_option("long_regions", 0)
        for f in ("n_regions", "n_contigs", "n_check_align", "n_dp_cells", "n_kmer_occurrences"):
            assert getattr(a, f) == getattr(b, f), f
        for f in ("so_off", "so_mers", "so_counts", "uniq_reg_off", "uniq_rec", "uniq_mult", "ctg_reg_off", "region_status",
                  "region_dp_cells"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
        for i in range(len(regions)):
            assert a.contig_records(i) == b.contig_records(i), regions[i].name


def test_abandoned_contigs_are_dropped(handle):
    from breakmer_b200 import _lib, batch
    import numpy as np
    pk = batch.PackedBatch([_region("mix", 15)])
    pk.read_len = np.array([MIX_READ_LEN, 0], dtype=np.int32)
    off = batch.run(handle, pk)
    assert list(off.region_status) == [_lib.BK_ERR_CAPACITY]
    assert off.ctg_reg_off[1] > 0                      # contigs of the abandoned attempt are in the default result
    handle.set_option("long_regions", 1)
    try:
        on = batch.run(handle, pk)
    finally:
        handle.set_option("long_regions", 0)
    only, ctg = _oracle("mix", 15)
    assert list(on.region_status) == [0]
    assert on.sample_only(0) == only
    assert on.contig_records(0) == ctg
    assert on.n_contigs == len(ctg)


def test_submit_wait_on_a_device_pipeline():
    from breakmer_b200 import batch, shard
    regions = mixed_regions(15)
    # chunks that mix long and normal regions
    chunks = [regions[i::4] for i in range(4)]
    pipe = shard.DevicePipeline(0, inflight=3, long_regions=True)
    try:
        results = []
        for c in chunks:
            if pipe.full():
                results.append(pipe.pop())
            pipe.submit(batch.PackedBatch(c), c)
        while pipe.pending():
            results.append(pipe.pop())
    finally:
        pipe.close()
    assert len(results) == len(chunks)
    for out, _pk, c in results:
        check_mixed(out, c, 15)


def test_the_mode_is_fixed_at_upload(handle):
    from breakmer_b200 import batch
    regions = mixed_regions(15)
    pk = batch.PackedBatch(regions)
    handle.set_option("long_regions", 1)
    batch.upload(handle, pk)
    handle.set_option("long_regions", 0)               # after the upload: the uploaded batch keeps its mode
    check_mixed(batch.run(handle, pk, resident=True), regions, 15)
    handle.set_option("long_regions", 1)
    batch.submit(handle, pk)
    handle.set_option("long_regions", 0)               # a batch in flight keeps its mode
    check_mixed(batch.wait(handle, pk), regions, 15)


# ---- Python drop-ins ---------------------------------------------------------------------------------------------
@pytest.fixture
def counted(monkeypatch):
    """counts the targets _pack_targets packs and records every batch.run(..., long=...) call"""
    from breakmer_b200 import batch, sv_processor
    packed, runs = [], []
    pack, run = sv_processor._pack_targets, batch.run

    def pack_counted(targets, *a, **kw):
        packed.extend(t.name for t in targets)
        return pack(targets, *a, **kw)

    def run_counted(*a, **kw):
        runs.append(kw.get("long", False))
        return run(*a, **kw)

    monkeypatch.setattr(sv_processor, "_pack_targets", pack_counted)
    monkeypatch.setattr(batch, "run", run_counted)
    return packed, runs


@pytest.mark.parametrize("form", [dict(ingest="python"), dict(ingest="native", write_contigs=True), dict(ingest="python", max_targets=2),
                                  dict(ingest="native", max_targets=2, apply_thread=True), dict(ingest="python", devices=[0, 0])])
def test_compare_kmers_batch_one_pass(tmp_path, counted, form):
    from breakmer_b200 import sv_processor
    packed, runs = counted
    pairs = _targets(tmp_path / "a")
    sv_processor.compare_kmers_batch([t for _r, t in pairs], on_capacity="assemble", **form)
    _check_targets(pairs, write_contigs=form.get("write_contigs", False))
    assert sorted(packed) == sorted(t.name for _r, t in pairs)          # each target packed exactly once
    assert True not in runs                                             # never the long entry
    # the handles and cached pipelines of this thread are left in the default mode
    again = _targets(tmp_path / "b")
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in again], **{k: v for k, v in form.items() if k != "write_contigs"})
    assert ei.value.targets == ["zz_long"]


def test_init_assembly_batch_one_pass(counted):
    from breakmer_b200 import sv_assembly, utils
    _packed, runs = counted
    calls, exp = [], []
    for name in ["C2_00001", LONG_READ_REGIONS[0][0], GROWING_REGION[0]]:
        r = _region(name, 15)
        only, ctg = _oracle(name, 15)
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        calls.append((only, recs, r.k, r.rc_thresh, r.read_len))
        exp.append(ctg)
    got = sv_assembly.init_assembly_batch(calls, on_capacity="assemble")
    assert runs == [False]                                               # one device call
    for g, e in zip(got, exp):
        assert [c.get_contig_seq() for c in g] == [c["seq"] for c in e]
        assert [c.get_kmer_locs() for c in g] == [c["kmer_locs"] for c in e]
        assert [sorted(rd.id for rd in c.reads) for c in g] == [c["reads"] for c in e]
    with pytest.raises(RuntimeError):                                   # the handle is back in the default mode
        sv_assembly.init_assembly_batch(calls)
