"""The long assembler (bk_compare_kmers_long: assemble_long_kernel, reads and contigs up to 65,535 bases) against the
oracle, which has no length limit, and against bk_compare_kmers_batch where both apply; and the Python drop-ins'
on_capacity="assemble"."""
import os

import pytest

from breakmer_b200 import synth
from oracle import assembler_py
from oracle.make_golden import oracle_sample_only

pytestmark = pytest.mark.gpu

# reads of 4,500-6,000 bases at low coverage (their contigs grow longer still)
LONG_READ_REGIONS = [
    ("lr0", dict(seed=11, L=10000, cov=6, k=15, e=0.003, event=("del", 300, None), rl=4500)),
    ("lr1", dict(seed=12, L=12000, cov=6, k=21, e=0.003, event=("ins", 60), rl=5200)),
    ("lr2", dict(seed=13, L=13000, cov=5, k=15, e=0.003, event=("tdup", 400), rl=6000)),
]
# 3,000-base reads across one junction whose contig grows to 4,123 bases
GROWING_REGION = ("grow", dict(seed=22, L=7000, cov=60, k=15, e=0.002, event=("del", 300, None), rl=3000))


@pytest.fixture(scope="module")
def handle():
    from breakmer_b200 import _lib
    h = _lib.Handle(0)
    yield h
    h.close()


def oracle_region(region):
    _r, _c, _s, only = oracle_sample_only(region)
    return only, assembler_py.init_assembly(only, region.reads, region.k, region.rc_thresh, region.read_len)


def over_limit_region(n):
    """one read of n bases (its region cannot be assembled by either entry when n > 65,535)"""
    return synth.Region(name="zz_over", k=15, ref_fwd="ACGT" * 50, reads=[("@a:1:1:1:1/1_0", ("ACGTT" * (n // 5 + 1))[:n], "I" * n, False)],
                        sc_records=[("a", "ACGT" * 10)])


def check_long(handle, regions):
    from breakmer_b200 import batch
    out = batch.run(handle, batch.PackedBatch(regions), long=True)
    for i, r in enumerate(regions):
        only, ctg = oracle_region(r)
        assert out.region_status[i] == 0, r.name
        assert out.sample_only(i) == only, r.name
        assert out.contig_records(i) == ctg, r.name
    return out


@pytest.mark.parametrize("k", [15, 21])
def test_reads_above_4095_bases(handle, k):
    regions = [synth.make_region(n, **kw) for n, kw in LONG_READ_REGIONS if kw["k"] == k]
    assert regions and all(max(len(x[1]) for x in r.reads) > 4095 for r in regions)
    out = check_long(handle, regions)
    assert out.n_contigs >= len(regions)


def test_a_contig_grows_past_4095_bases_from_shorter_reads(handle):
    from breakmer_b200 import _lib, batch
    name, kw = GROWING_REGION
    r = synth.make_region(name, **kw)
    assert max(len(x[1]) for x in r.reads) <= 4095
    pk = batch.PackedBatch([r])
    assert list(batch.run(handle, pk).region_status) == [_lib.BK_ERR_CAPACITY]      # the growth check of the fast kernel
    out = check_long(handle, [r])
    assert max(len(c["seq"]) for c in out.contig_records(0)) > 4095


def test_same_results_as_the_batched_entry_where_both_apply(handle):
    """golden regions and C2 / C5 regions: every pair is within the warp DP's reach, so this pins the shared state
    machine, the wide packed keys and the warp-DP route of the long kernel"""
    from conftest import golden
    from breakmer_b200 import batch
    cases = golden("assembly_golden.json")["cases"]
    by_k = {}
    for c in cases[:24]:
        kw = dict(c["kwargs"]); kw["event"] = tuple(kw["event"])
        by_k.setdefault(kw["k"], []).append(synth.make_region(c["name"], **kw))
    groups = list(by_k.values()) + [list(synth.config_regions("C2", n=15, start=0)), list(synth.config_regions("C5", n=15, start=0))]
    for regions in groups:
        pk = batch.PackedBatch(regions)
        a = batch.run(handle, pk)
        b = batch.run(handle, pk, long=True)
        assert list(a.region_status) == list(b.region_status)
        assert a.n_check_align == b.n_check_align and a.n_dp_cells == b.n_dp_cells
        for i in range(len(regions)):
            assert a.sample_only(i) == b.sample_only(i)
            assert a.contig_records(i) == b.contig_records(i), regions[i].name


def test_a_read_beyond_the_long_limit_is_reported_and_the_rest_completes(handle):
    from breakmer_b200 import _lib, batch
    over = over_limit_region(batch.LONG_MAX_LEN + 1)
    r0 = synth.make_region(LONG_READ_REGIONS[0][0], **LONG_READ_REGIONS[0][1])
    normal = list(synth.config_regions("C2", n=3, start=3))
    regions = [normal[0], over, r0] + normal[1:]
    out = batch.run(handle, batch.PackedBatch(regions), long=True)
    for i, r in enumerate(regions):
        if r is over:
            assert out.region_status[i] == _lib.BK_ERR_CAPACITY
            assert out.contig_records(i) == []
        else:
            only, ctg = oracle_region(r)
            assert out.region_status[i] == 0, r.name
            assert out.sample_only(i) == only, r.name
            assert out.contig_records(i) == ctg, r.name


# ---- Python drop-ins ---------------------------------------------------------------------------------------------
def _targets(tmp_path):
    """three C2 targets and one with 4,500-base reads (last), as the slice of sv_processor.target that compare_kmers
    touches, with their files"""
    from breakmer_b200 import utils
    regions = list(synth.config_regions("C2", n=3, start=0)) + [synth.make_region("zz_long", **LONG_READ_REGIONS[0][1])]
    out = []
    for r in regions:
        d = tmp_path / r.name
        for sub in ("kmers", "contigs"):
            (d / sub).mkdir(parents=True)
        ref_fn = d / "ref.fa"
        ref_fn.write_text(">%s\n%s\n" % (r.name, r.ref_fwd))
        fq = d / "reads.fastq"
        fq.write_text("".join("%s\n%s\n+\n%s\n" % (rid, seq, q) for rid, seq, q, _io in r.reads))
        sc = d / "sc.fa"
        sc.write_text("".join(">%s\n%s\n" % (n, s) for n, s in r.sc_records))
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        out.append((r, _Target(r, recs, str(ref_fn), str(fq), str(sc), str(d))))
    return out


class _Params:
    def __init__(self, k, rc):
        self.k, self.rc = k, rc

    def get_kmer_size(self):
        return self.k

    def get_sr_thresh(self, _which):
        return self.rc


class _Target:
    def __init__(self, r, recs, ref_fn, fq, sc, d):
        self.name = r.name
        self.params = _Params(r.k, r.rc_thresh)
        self.files = {'target_ref_fn': [ref_fn], 'cleaned_fq': fq, 'sv_sc_unmapped_fa': sc}
        self.paths = {'kmers': os.path.join(d, "kmers"), 'contigs': os.path.join(d, "contigs")}
        self.cleaned_read_recs = recs
        self.read_len = r.read_len
        self.kmers = {}


def _check_targets(pairs, write_contigs=False):
    for r, t in pairs:
        only, ctg = oracle_region(r)
        got = [c.get_contig_seq() for c in t.kmers['clusters']]
        assert got == [c["seq"] for c in ctg], r.name
        assert [c.get_kmer_locs() for c in t.kmers['clusters']] == [c["kmer_locs"] for c in ctg], r.name
        assert [sorted(x.id for x in c.reads) for c in t.kmers['clusters']] == [c["reads"] for c in ctg], r.name
        with open(t.files['sample_kmers']) as f:
            lines = [ln.rstrip("\n").split("\t") for ln in f if ln.strip()]
        assert {m: int(c) for m, c in lines} == only, r.name
        assert t.cleaned_read_recs is None
        if write_contigs and ctg:
            assert os.listdir(t.paths['contigs']), r.name


@pytest.mark.parametrize("form", [dict(ingest="python"), dict(ingest="native"), dict(ingest="native", write_contigs=True),
                                  dict(ingest="python", max_targets=2, apply_thread=True),
                                  dict(ingest="native", max_targets=2, apply_thread=True), dict(ingest="python", devices=[0, 0])])
def test_compare_kmers_batch_assembles_the_long_target(tmp_path, form):
    from breakmer_b200 import sv_processor
    pairs = _targets(tmp_path)
    sv_processor.compare_kmers_batch([t for _r, t in pairs], on_capacity="assemble", **form)
    _check_targets(pairs, write_contigs=form.get("write_contigs", False))


def test_compare_kmers_batch_still_raises_by_default(tmp_path):
    from breakmer_b200 import sv_processor
    pairs = _targets(tmp_path)
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in pairs])
    assert ei.value.targets == ["zz_long"]


def test_compare_kmers_batch_raises_beyond_the_long_limit(tmp_path):
    from breakmer_b200 import batch, sv_processor
    pairs = _targets(tmp_path)
    t = pairs[-1][1]
    n = batch.LONG_MAX_LEN + 1
    seq = ("ACGTT" * (n // 5 + 1))[:n]
    from breakmer_b200 import utils
    t.cleaned_read_recs = {seq: [utils.fq_read("@a:1:1:1:1/1_0", seq, "I" * n, False)]}
    with pytest.raises(sv_processor.CapacityError) as ei:
        sv_processor.compare_kmers_batch([t for _r, t in pairs], on_capacity="assemble")
    assert ei.value.targets == ["zz_long"]
    _check_targets(pairs[:-1])


def test_init_assembly_batch_assembles_the_long_call():
    from breakmer_b200 import sv_assembly, utils
    calls, exp = [], []
    for name, kw in [("c2", None), LONG_READ_REGIONS[0], GROWING_REGION]:
        r = synth.config_region("C2", 1) if kw is None else synth.make_region(name, **kw)
        only, ctg = oracle_region(r)
        recs = {}
        for rid, seq, q, io in r.reads:
            recs.setdefault(seq, []).append(utils.fq_read(rid, seq, q, io))
        calls.append((only, recs, r.k, r.rc_thresh, r.read_len))
        exp.append(ctg)
    with pytest.raises(RuntimeError):
        sv_assembly.init_assembly_batch(calls)
    got = sv_assembly.init_assembly_batch(calls, on_capacity="assemble")
    for g, e in zip(got, exp):
        assert [c.get_contig_seq() for c in g] == [c["seq"] for c in e]
        assert [c.get_kmer_locs() for c in g] == [c["kmer_locs"] for c in e]
        assert [sorted(rd.id for rd in c.reads) for c in g] == [c["reads"] for c in e]
