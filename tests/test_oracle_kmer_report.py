"""Where the k-mer stage's soft-clip k-mers go, restated on the oracle (rows K1-K4 of oracle/kmers_py.py), and checked
against oracle/kmers_py.sample_only.  `kmer_breakdown` is the reference for bk_kmer_report and the "normal_kmers"
option (tests/test_gpu_kmer_report.py, tests/test_simt_kmer_report.py)."""
from breakmer_b200 import synth
from conftest import golden
from oracle import kmers_py

FIELDS = ("soft_clip", "not_in_reads", "in_reference", "in_normal", "sample_only")


def kmer_breakdown(ref_fwd, read_seqs, sc_seqs, k, normal_seqs=None):
    """-> (row, removed): row = {field: count of distinct k-mers} in the order of the reference's set operations
    ((case & case_sc) - ref, then the normal sample's k-mers), removed = {mer: case count} of the k-mers the normal sample
    removed"""
    ref = kmers_py.count_kmers([ref_fwd], k)
    kmers_py.count_kmers([kmers_py.revcomp(ref_fwd)], k, into=ref)
    case = kmers_py.count_kmers(read_seqs, k)
    sc = set(kmers_py.count_kmers(sc_seqs, k))
    in_reads = sc & set(case)
    kept = in_reads - set(ref)
    normal = set(kmers_py.count_kmers(normal_seqs, k)) if normal_seqs is not None else set()
    removed = kept & normal
    row = {"soft_clip": len(sc), "not_in_reads": len(sc - in_reads), "in_reference": len(in_reads & set(ref)),
           "in_normal": len(removed), "sample_only": len(kept - normal)}
    return row, {m: case[m] for m in removed}


def region_breakdown(region, with_normal=True):
    normal = [x[1] for x in region.normal_reads] if (with_normal and region.normal_reads) else None
    return kmer_breakdown(region.ref_fwd, [x[1] for x in region.reads], [x[1] for x in region.sc_records], region.k, normal)


def _golden_regions():
    for case in golden("kmers_golden.json")["cases"]:
        kw = dict(case["kwargs"]); kw["event"] = tuple(kw["event"])
        yield synth.make_region(case["name"], **kw)


def _check(region):
    row, removed = region_breakdown(region)
    assert list(row) == list(FIELDS)
    assert row["soft_clip"] == row["not_in_reads"] + row["in_reference"] + row["in_normal"] + row["sample_only"]
    seqs = ([x[1] for x in region.reads], [x[1] for x in region.sc_records])
    normal = [x[1] for x in region.normal_reads] if region.normal_reads else None
    _r, _c, _s, only = kmers_py.sample_only(region.ref_fwd, *seqs, region.k, normal)
    _r, _c, _s, only_without = kmers_py.sample_only(region.ref_fwd, *seqs, region.k)
    assert row["sample_only"] == len(only)
    assert not (set(removed) & set(only))
    assert {**only, **removed} == only_without                       # the normal set is what the normal sample took away
    return row, removed


def test_breakdown_of_the_golden_regions():
    rows = [_check(r)[0] for r in _golden_regions()]
    assert rows and all(r["in_normal"] == 0 for r in rows)
    assert any(r["in_reference"] for r in rows) and any(r["sample_only"] for r in rows)     # (their soft clips are read bases)


def test_breakdown_with_a_normal_sample():
    rows = [_check(synth.config_region("C3", i)) for i in range(4)]
    assert any(row["in_normal"] > 0 and removed for row, removed in rows)     # germline events: the normal removes k-mers


def test_breakdown_of_edge_regions():
    # soft clips and no reads: every candidate is missing from the reads; no soft clips: nothing at all
    row, removed = kmer_breakdown("ACGTACGTAC" * 5, [], ["ACGTTTTTGGGCCCAAA", "NNNNACGTTTTTGGGCC"], 5)
    assert row["soft_clip"] > 0 and row["soft_clip"] == row["not_in_reads"] and removed == {}
    row, removed = kmer_breakdown("ACGTACGTAC" * 5, ["ACGTTTTTGGGCCCAAA"], [], 5, ["ACGTTTTTGGGCCCAAA"])
    assert row == dict.fromkeys(FIELDS, 0) and removed == {}
