"""The k-mer stage, read grouping and the k-mer/read index of bk_compare_kmers_batch at the input sizes where the kernels
change path, against the oracle (oracle/kmers_py.py; group_reads and init_assembly of oracle/assembler_py.py; the k-mer
report breakdown of tests/test_oracle_kmer_report.py):

  * region_kmer_kernel's table classes: 1,024 to 16,384 slots in shared memory, 32,768 and more in a slice of the global
    table, and the three sorts of rk_sort_staged (in shared memory; in shared memory for a region whose table is global;
    inside the global slice);
  * every k from 2 to 31 (at k = 16 a k-mer fills exactly 32 bits), and bk_count_kmers / bk_sample_only across the
    1,024-position emit tile;
  * windows at record starts, N bases and the 2,048-position tile of the window enumeration, on shared and global tables;
  * the reference k-mer cache built in chunks of 2^min(63 - 2k, 16) regions;
  * the unique-read tables and the index keys at 2^n - 1, 2^n and 2^n + 1 records, and a grouping call of 300,000 reads;
  * one call of 65,535 regions, the most a call takes, and the refusal of 65,536.

Every test asserts that its input reaches the path it is named for, through table_slots and cache_chunks below, which
restate the library's rules (breakmer_b200/csrc/pipeline_impl.cuh).  A change to a rule then fails the test instead of
leaving it to test another path."""
import dataclasses
import multiprocessing as mp
import os
import random

import numpy as np
import pytest

from breakmer_b200 import _lib, batch, synth
from oracle import assembler_py, kmers_py
from test_oracle_kmer_report import region_breakdown

pytestmark = pytest.mark.gpu

# the emulated library (tests/sim_util.py) runs every kernel on the host: the 65,535-region call takes it too long
EMULATED = "simt" in os.path.basename(os.environ.get("BK_LIB", ""))

RK_MIN_SLOTS = 1024            # smallest k-mer table of a region
RK_SMEM_CAP_MAX = 16384        # largest table in shared memory (region_kmers.cuh)
MAX_REGIONS = 65535            # regions of one call


def table_slots(n_sc_bases):
    """-> (slots, shared) of a region's k-mer table, as pipeline_upload_into sizes it: the smallest power of two of at
    least RK_MIN_SLOTS slots above the region's soft-clip base count, in shared memory up to RK_SMEM_CAP_MAX slots, else a
    slice of the global table"""
    slots = RK_MIN_SLOTS
    while slots <= n_sc_bases:
        slots <<= 1
    return slots, slots <= RK_SMEM_CAP_MAX


def smem_cap(regions):
    """the launch's shared table size: the largest shared table of the call's regions, at least RK_MIN_SLOTS"""
    return max([RK_MIN_SLOTS] + [s for s, shared in (table_slots(sc_bases(r)) for r in regions) if shared])


def sorts_in_global_slice(n_staged, cap):
    """rk_sort_staged sorts n_staged pairs inside the region's global slice when their power-of-two padding is above the
    launch's shared table"""
    n_pad = 2
    while n_pad < n_staged:
        n_pad <<= 1
    return n_staged > 1 and n_pad > cap


def cache_chunks(n_regions, k):
    """-> region counts of the chunks bk_ref_cache_build sorts one after the other: 2^min(63 - 2k, 16) regions each, so
    that the region index and the k-mer share one 64-bit sort key"""
    size = min(max(n_regions, 1), 1 << min(63 - 2 * k, 16))
    return [min(size, n_regions - a) for a in range(0, n_regions, size)]


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def _seq(rng, n):
    return "".join(rng.choices("ACGT", k=n))


def sc_bases(region):
    return sum(len(s) for _n, s in region.sc_records)


def fit_clips(region, n_bases, seed=0, filler="random"):
    """the region with exactly n_bases soft-clip bases: its own records as far as they fit, then "foreign" records that
    no read holds (filler "random"; at small k their k-mers can be read k-mers, which the oracle sees as well) or records
    of N bases (filler "N"), which hold no window and change no result"""
    rng = random.Random(seed)
    recs, total = [], 0
    for name, s in region.sc_records:
        if total + len(s) > n_bases:
            break
        recs.append((name, s))
        total += len(s)
    i = 0
    while total < n_bases:
        n = min(300, n_bases - total)
        recs.append(("foreign%d" % i, "N" * n if filler == "N" else _seq(rng, n)))
        total += n
        i += 1
    return dataclasses.replace(region, name="%s_sc%d" % (region.name, n_bases), sc_records=recs)


def event_region(name, k, seed, L=400, cov=20, event=("ins", 40)):
    """a small region with one planted event, error free: a few dozen junction reads and their soft clips"""
    return synth.make_region(name, seed, L, cov, k, 0.0, event, n_rate=0.0)


def insertion_region(name, k, seed, novel=2400, flank=300, step=6, rl=100, normal_cover=0):
    """a long novel insertion between two flanks of reference, covered by a read every `step` bases; every read that
    touches the insertion is also a soft-clip record (about 42,000 soft-clip bases, more than 2,000 sample-only k-mers).
    normal_cover: the normal sample covers the first that many bases of the insertion, so it removes their k-mers."""
    rng = random.Random(seed)
    left, ins, right = _seq(rng, flank), _seq(rng, novel), _seq(rng, flank)
    g = left + ins + right
    reads, sc = [], []
    for j, a in enumerate(range(0, len(g) - rl + 1, step)):
        rid = "@INS%d:1:1:%d:%d/1_%d" % (seed, a, j, int(j % 5 == 0))
        reads.append((rid, g[a:a + rl], "I" * rl, j % 5 == 0))
        if a + rl > flank and a < flank + novel:
            sc.append((rid[1:], g[a:a + rl]))
    normal = [("n%d" % j, ins[a:a + rl]) for j, a in enumerate(range(0, normal_cover - rl + 1, step))]
    return synth.Region(name, k, left + right, reads, sc, normal)


def plain_region(name, k, ref, reads, sc, normal=()):
    return synth.Region(name, k, ref, [("@%s:1:1:%d:%d/1_0" % (name, j, j), s, "I" * len(s), False) for j, s in enumerate(reads)],
                        [("%s_sc%d" % (name, j), s) for j, s in enumerate(sc)], [("%s_n%d" % (name, j), s) for j, s in enumerate(normal)])


# ---------------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------------
def expected_kstage(region, with_normal):
    """-> (sample-only {mer: count}, k-mer report row, {mer: count} the normal sample removed)"""
    row, removed = region_breakdown(region, with_normal=with_normal)
    normal = [x[1] for x in region.normal_reads] if (with_normal and region.normal_reads) else None
    only = kmers_py.sample_only(region.ref_fwd, [x[1] for x in region.reads], [x[1] for x in region.sc_records], region.k,
                                normal)[3]
    return only, row, removed


def _oracle_contigs(args):
    only, r = args
    return assembler_py.init_assembly(only, r.reads, r.k, r.rc_thresh, r.read_len)


def expected_groups(region):
    """-> [(record index of the group's first read, group size)] of group_reads, in its order"""
    index = {rec[0]: j for j, rec in enumerate(region.reads)}
    assert len(index) == len(region.reads)                     # (the inputs give every record its own id)
    return [(index[u.rep_id], u.nreads) for u in assembler_py.group_reads(region.reads)]


@pytest.fixture(scope="module")
def pool():
    # forked before this module's handle exists; the workers never touch CUDA
    p = mp.get_context("fork").Pool(os.cpu_count() or 1)
    yield p
    p.close()
    p.join()


@pytest.fixture(scope="module")
def handle(pool):
    h = _lib.Handle(0)
    yield h
    h.close()


def run_call(h, regions, normal_kmers=False, **pk_kw):
    pk = batch.PackedBatch(regions, **pk_kw)
    with batch.options([h], normal_kmers=normal_kmers):
        out = batch.run(h, pk)
    assert out.n_regions == len(regions)
    return pk, out, batch.kmer_report(h)


def assert_ascending(mers, what):
    mers = np.asarray(mers, dtype=np.uint64)
    assert np.all(mers[1:] > mers[:-1]), what                  # (np.diff of uint64 wraps: a descent would pass it)


def check_kstage(regions, pk, out, rows, exp=None):
    """sample-only k-mers, the k-mer report and (with the "normal_kmers" option) the normal k-mers of every region ==
    the oracle, each region's arrays strictly ascending; -> the expected (only, row, removed) per region"""
    exp = exp or [expected_kstage(r, pk.has_normal) for r in regions]
    for i, (r, (only, row, removed)) in enumerate(zip(regions, exp)):
        a, b = int(out.so_off[i]), int(out.so_off[i + 1])
        assert_ascending(out.so_mers[a:b], r.name)
        assert out.sample_only(i) == only, r.name
        assert rows[i] == row, (r.name, rows[i], row)
        if out.normal is not None:
            off, mers = out.normal[0], out.normal[1]
            assert_ascending(mers[int(off[i]):int(off[i + 1])], r.name)
            assert out.normal_kmers(i) == removed, r.name
    return exp


def check_contigs(pool, regions, out, exp, which):
    got = [out.contig_records(i) for i in which]
    want = pool.map(_oracle_contigs, [(exp[i][0], regions[i]) for i in which])
    for i, g, w in zip(which, got, want):
        assert g == w, regions[i].name
    return sum(len(w) for w in want)


def check_groups(regions, out, exp_groups=None):
    """uniq_reg_off, uniq_rec (the caller's record numbering) and uniq_mult == group_reads of every region"""
    exp_groups = exp_groups or [expected_groups(r) for r in regions]
    first = 0
    for i, (r, groups) in enumerate(zip(regions, exp_groups)):
        a, b = int(out.uniq_reg_off[i]), int(out.uniq_reg_off[i + 1])
        assert b - a == len(groups), r.name
        assert out.uniq_rec[a:b].tolist() == [first + j for j, _n in groups], r.name
        assert out.uniq_mult[a:b].tolist() == [n for _j, n in groups], r.name
        first += len(r.reads)
    assert int(out.uniq_reg_off[-1]) == sum(len(g) for g in exp_groups)


# ---------------------------------------------------------------------------------------------------------------------
# 1. table size classes of region_kmer_kernel
# ---------------------------------------------------------------------------------------------------------------------
CLASS_SIZES = (1023, 1024, 2047, 2048, 8191, 8192, 16383, 16384)


def class_regions(k=21):
    regs = [fit_clips(event_region("cls%d" % i, k, 300 + i), n, seed=i) for i, n in enumerate(CLASS_SIZES)]
    big = insertion_region("novel", k, 7)
    big_normal = insertion_region("novel_normal", k, 8, normal_cover=1400)
    return regs, big, big_normal


def test_table_size_classes(pool, handle):
    regs, big, big_normal = class_regions()
    slots = [table_slots(sc_bases(r)) for r in regs + [big]]
    assert slots == [(1024, True), (2048, True), (2048, True), (4096, True), (8192, True), (16384, True), (16384, True),
                     (32768, False), (65536, False)]
    assert 38000 <= sc_bases(big) <= 44000 and not table_slots(sc_bases(big_normal))[1]
    exp = {r.name: expected_kstage(r, True) for r in regs + [big, big_normal]}
    n_only = {name: len(e[0]) for name, e in exp.items()}
    assert n_only["novel"] > 1024 and n_only["novel_normal"] > 1024 and len(exp["novel_normal"][2]) > 1024
    assert all(n_only[r.name] > 0 for r in regs)

    # all classes in one call: the launch's shared table has 16,384 slots, and the global regions sort in shared memory
    mix = regs + [big, big_normal]
    assert smem_cap(mix) == RK_SMEM_CAP_MAX
    assert not sorts_in_global_slice(n_only["novel"], smem_cap(mix))
    pk, out, rows = run_call(handle, mix, normal_kmers=True)
    check_kstage(mix, pk, out, rows, [exp[r.name] for r in mix])
    assert check_contigs(pool, mix, out, [exp[r.name] for r in mix], [0, 3, 5, 6, 7]) > 0
    all_in_one = {r.name: out.sample_only(i) for i, r in enumerate(mix)}

    # global regions only: the launch's shared table stays at 1,024 slots, so the deep regions' sample-only and normal
    # k-mers are sorted inside their global slices
    glob = [regs[-1], big, big_normal]
    assert smem_cap(glob) == RK_MIN_SLOTS
    assert sorts_in_global_slice(n_only["novel"], smem_cap(glob))
    assert sorts_in_global_slice(len(exp["novel_normal"][2]), smem_cap(glob))
    pk, out, rows = run_call(handle, glob, normal_kmers=True)
    check_kstage(glob, pk, out, rows, [exp[r.name] for r in glob])
    assert check_contigs(pool, glob, out, [exp[r.name] for r in glob], [0]) > 0
    assert {r.name: out.sample_only(i) for i, r in enumerate(glob)} == {r.name: all_in_one[r.name] for r in glob}

    # one small shared region alone
    one = [regs[0]]
    assert smem_cap(one) == RK_MIN_SLOTS and table_slots(sc_bases(regs[0])) == (1024, True)
    pk, out, rows = run_call(handle, one, normal_kmers=True)
    check_kstage(one, pk, out, rows, [exp[regs[0].name]])
    check_contigs(pool, one, out, [exp[regs[0].name]], [0])


# ---------------------------------------------------------------------------------------------------------------------
# 2. every k
# ---------------------------------------------------------------------------------------------------------------------
ALL_K = list(range(2, 32))


def test_every_k_shared_and_global_tables(handle):
    n_only = 0
    for k in ALL_K:
        small = event_region("k%d_shared" % k, k, 900 + k)
        deep = fit_clips(event_region("k%d_global" % k, k, 950 + k), 16400, seed=k)
        assert table_slots(sc_bases(small))[1] and table_slots(sc_bases(deep)) == (32768, False), k
        regions = [small, deep]
        pk, out, rows = run_call(handle, regions)
        exp = check_kstage(regions, pk, out, rows)
        n_only += sum(len(e[0]) for e in exp)
        assert all(e[1]["soft_clip"] > 0 for e in exp), k
    assert n_only > 0


def _tile_records(rng, k):
    """records whose lengths straddle the 1,024-position tile of kmer_emit_kernel (and twice that), with short records of
    k - 1, k and k + 1 bases, N bases and lower case"""
    core = _seq(rng, 5000)
    lens = [1023, 1, 1024, 1025, max(k - 1, 1), k, k + 1, 2047, 2048, 2049, 1000, 24, 3]
    out, at = [], 0
    for n in lens:
        out.append(core[at:at + n])
        at += n // 3 + 1                     # overlapping pieces of one sequence: their k-mers recur across records
    out.append(core[100:1200].lower())
    out.append(core[500:1540] + "N" + core[1541:2100])
    return core, out


def test_count_and_sample_only_across_the_emit_tile_every_k(handle):
    for k in ALL_K:
        rng = random.Random(5000 + k)
        core, seqs = _tile_records(rng, k)
        mult = [rng.randint(1, 5) for _ in seqs]
        mers, counts = handle.count_kmers(seqs, k)
        assert_ascending(mers, k)
        assert dict(zip(_lib.codes_to_mers(mers, k), counts.tolist())) == kmers_py.count_kmers(seqs, k), k
        mers, counts = handle.count_kmers(seqs, k, mult=mult)
        want = {}
        for s, m in zip(seqs, mult):
            for mer, c in kmers_py.count_kmers([s], k).items():
                want[mer] = want.get(mer, 0) + c * m
        assert dict(zip(_lib.codes_to_mers(mers, k), counts.tolist())) == want, k
        # sample-only: soft clips around the tile edges, a reference and a normal sample that each take part of them
        sc = [core[1000:1100], core[2000:2100], core[3040:3140], _seq(rng, 60)]
        ref = core[1020:1060] + _seq(rng, 50)
        normal = [core[2040:2080]]
        case = handle.count_kmers(seqs, k)
        sc_m = handle.count_kmers(sc, k)[0]
        ref_m = handle.count_kmers([ref, kmers_py.revcomp(ref)], k)[0]
        for nm in (None, normal):
            got = handle.sample_only(k, case, sc_m, ref_m, None if nm is None else handle.count_kmers(nm, k)[0])
            assert_ascending(got[0], k)
            want = kmers_py.sample_only(ref, seqs, sc, k, nm)[3]
            assert dict(zip(_lib.codes_to_mers(got[0], k), got[1].tolist())) == want, (k, nm is None)


# ---------------------------------------------------------------------------------------------------------------------
# 3. windows, records and tiles of the window enumeration, on shared and global tables
# ---------------------------------------------------------------------------------------------------------------------
def _as_regions(tag, k, sc, reads, ref, normal=None):
    return [plain_region("%s_%d" % (tag, r), k, ref[r], reads[r], sc[r], normal[r] if normal else ()) for r in range(len(sc))]


def _both_tables(h, regions):
    """the regions as they are (shared tables) and padded with N records past 16,384 soft-clip bases (global tables):
    both calls give the oracle's result"""
    exp = None
    for pad in (False, True):
        regs = [fit_clips(r, RK_SMEM_CAP_MAX + 16, filler="N") for r in regions] if pad else regions
        assert all(table_slots(sc_bases(r))[1] != pad for r in regs)
        pk, out, rows = run_call(h, regs, normal_kmers=True)
        exp = check_kstage(regs, pk, out, rows, exp)
    return exp


def test_windows_never_span_records_or_invalid_bases(handle):
    """adjacent pieces of one sequence as separate records: a window that (wrongly) spanned the cut would be a real k-mer
    of the other inputs, so it would show up in the result -- in every set, at every position of a thread's 4-window strip"""
    rng = random.Random(17)
    x = "".join(rng.choice("ACGT") for _ in range(400))
    y = "".join(rng.choice("ACGT") for _ in range(300))
    for k in (2, 3, 4, 5, 15, 22):
        plain, with_normal = [], []
        for cut in range(100, 109):
            sc = [[x[40:cut], x[cut:260]],                       # candidates cut in two; the reads hold the uncut sequence
                  [x[30:300]],                                   # uncut candidates; the reads are cut
                  [x[30:300]],                                   # uncut candidates and reads; the reference is cut / holds an N
                  [x[40:cut] + "N" + x[cut + 1:260]]]
            reads = [[x[0:400], x[20:380]],
                     [x[0:cut], x[cut:400], x[10:cut], x[cut:390]],
                     [x[0:400], x[0:400]],
                     [x[0:400], x[0:400]]]
            ref = [y, y, x[0:cut] + "N" + x[cut + 1:150] + y, y]
            normal = [[], [], [x[150:cut + 100], x[cut + 100:300]], []]
            plain += _as_regions("cut%d" % cut, k, sc, reads, ref)
            with_normal += _as_regions("cutn%d" % cut, k, sc, reads, ref, normal)
        exp = _both_tables(handle, plain)
        assert any(e[0] for e in exp) or k <= 5, k           # (at small k the reference holds every k-mer)
        exp = _both_tables(handle, with_normal)
        assert any(e[2] for e in exp) or k <= 5, k


def test_tile_boundaries(handle):
    """records and windows that straddle the 2,048-position tile of the window enumeration"""
    rng = random.Random(2)
    g = lambda n: "".join(rng.choice("ACGT") for _ in range(n))
    big = g(5000)
    sc = [[big[2030:2070], big[4090:4110], big[0:30]], [big[1000:3100]]]
    reads = [[big[0:2047], big[2047:2049], big[2049:4200], big[4080:4130]], [big[i:i + 101] for i in range(900, 3200, 7)]]
    ref = [g(2100), big[2000:2050] + g(2100)]
    for k in (4, 15, 31):
        regions = _as_regions("tile", k, sc, reads, ref)
        assert sum(len(s) for s in reads[0]) > 2 * 2048 and sc_bases(regions[1]) > 2048
        exp = _both_tables(handle, regions)
        assert exp[1][0] or k == 4, k                        # (a random 2,100-base reference holds nearly every 4-mer)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the reference k-mer cache in chunks
# ---------------------------------------------------------------------------------------------------------------------
def check_cache_call(h, pool, regions, contigs_of):
    """a batch on the handle's reference k-mer cache == the same batch with its reference sequences == the oracle"""
    k = regions[0].k
    assert len(cache_chunks(len(regions), k)) > 1
    h.ref_cache_build([r.ref_fwd for r in regions], k)
    try:
        pk_c, out_c, rows_c = run_call(h, regions, with_ref=False)
        pk, out, rows = run_call(h, regions)
    finally:
        h.ref_cache_clear()
    exp = check_kstage(regions, pk, out, rows)
    check_kstage(regions, pk_c, out_c, rows_c, exp)
    assert rows_c == rows
    assert sum(e[1]["in_reference"] for e in exp) > 0            # the reference removes k-mers in these regions
    for i in contigs_of:
        assert out_c.contig_records(i) == out.contig_records(i), regions[i].name
    return exp, out


@pytest.mark.parametrize("k,n_regions,chunks", [(31, 7, [2, 2, 2, 1]), (28, 300, [128, 128, 44])])
def test_reference_cache_in_chunks(pool, handle, k, n_regions, chunks):
    assert cache_chunks(n_regions, k) == chunks
    regions = [event_region("cache%d_%d" % (k, i), k, 7000 + i, L=200, cov=10,
                            event=[("ins", 30), ("del", 40, None), ("tdup", 80)][i % 3]) for i in range(n_regions)]
    exp, out = check_cache_call(handle, pool, regions, range(n_regions))
    assert check_contigs(pool, regions, out, exp, range(n_regions)) > 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. read grouping and the index key widths
# ---------------------------------------------------------------------------------------------------------------------
def records_region(name, k, seed, n_records, duplicates):
    """a region of exactly n_records read records: the junction reads of a small insertion (which hold the sample-only
    k-mers) spread through distinct reads of the reference, the last record a junction read, so that the region's last
    unique read has the largest local index the index keys hold; `duplicates`: every fourth record repeats an earlier one"""
    ev = event_region(name, k, seed)
    rng = random.Random(seed)
    w = ev.ref_fwd
    junction = list({rec[1]: rec for rec in reversed(ev.reads)}.values())[::-1]   # (one record of each sequence)
    n_bg = n_records - len(junction)
    spots = rng.sample([(a, n) for n in range(60, 101) for a in range(0, len(w) - n + 1)], n_bg)
    background = [("@BG%d:1:1:%d:%d/1_0" % (seed, a, n), w[a:a + n], "I" * n, False) for a, n in spots]
    step = max(1, n_bg // len(junction))
    recs = []
    for j, rec in enumerate(junction):
        recs += background[j * step:(j + 1) * step] if j < len(junction) - 1 else background[j * step:]
        recs.append(rec)
    if duplicates:
        for j in range(4, len(recs) - 1, 4):
            src = recs[rng.randrange(j)]
            recs[j] = ("%s_dup%d" % (src[0], j), src[1], src[2], src[3])
    assert len(recs) == n_records and recs[-1] is junction[-1]
    return dataclasses.replace(ev, name="%s_%d%s" % (name, n_records, "d" if duplicates else ""), reads=recs)


@pytest.mark.parametrize("n", [10, 12])
def test_grouping_and_index_at_powers_of_two(pool, handle, n):
    for duplicates in (False, True):
        for n_records in (2 ** n - 1, 2 ** n, 2 ** n + 1):
            r = records_region("rec", 21, 60 + n, n_records, duplicates)
            groups = expected_groups(r)
            if not duplicates:
                assert len(groups) == n_records                 # the last unique read has local index n_records - 1
            pk, out, rows = run_call(handle, [r])
            exp = check_kstage([r], pk, out, rows)
            check_groups([r], out, [groups])
            assert exp[0][0] and check_contigs(pool, [r], out, exp, [0]) > 0
    # soft-clip base counts at 2^n - 1, 2^n and 2^n + 1: the widths of the mer fields of the index keys
    for n_sc in (2 ** n - 1, 2 ** n, 2 ** n + 1):
        r = fit_clips(event_region("scw", 21, 80 + n), n_sc, seed=n_sc)
        assert sc_bases(r) == n_sc
        pk, out, rows = run_call(handle, [r])
        exp = check_kstage([r], pk, out, rows)
        check_groups([r], out)
        check_contigs(pool, [r], out, exp, [0])


def test_grouping_volume_without_soft_clips(handle):
    """300,000 distinct reads and more in one call: about n^2 / 2^33 ~ 10 pairs of them share the low 32 bits of their
    hash, the part group_leader_kernel sorts on, so equal-hash runs of different reads are resolved byte by byte (the
    test cannot tell which pairs collide; the size is what makes collisions likely).  Mixed in: duplicates scattered
    through the call, lower-case twins (a different read to the reference's dict), one sequence in two regions (never
    merged) and reads that are prefixes of other reads.  No soft clips: no k-mer stage output and no assembly."""
    rs = np.random.default_rng(11)
    n_regions, per_region = 48, 6400
    letters = np.frombuffer(b"ACGT", np.uint8)
    regions = []
    for i in range(n_regions):
        lens = rs.integers(36, 61, per_region)
        codes = letters[rs.integers(0, 4, int(lens.sum()))].tobytes().decode()
        cuts = np.concatenate([[0], np.cumsum(lens)])
        seqs = [codes[cuts[j]:cuts[j + 1]] for j in range(per_region)]
        for j in range(7, per_region, 97):
            seqs[j] = seqs[rs.integers(0, j)]                               # duplicates
        for j in range(11, per_region, 211):
            seqs[j] = seqs[j - 5].lower()                                   # lower-case twins
        for j in range(13, per_region, 173):
            seqs[j] = seqs[j - 3][:-7]                                      # prefixes
        regions.append(plain_region("vol%d" % i, 15, "", seqs, []))
    shared = regions[0].reads[100][1]
    regions[1].reads[200] = (regions[1].reads[200][0], shared, "I" * len(shared), False)   # one sequence in two regions
    groups = [expected_groups(r) for r in regions]
    n_uniq = sum(len(g) for g in groups)
    assert n_uniq >= 300000 and n_uniq < sum(len(r.reads) for r in regions)
    pk, out, rows = run_call(handle, regions)
    assert int(out.so_off[-1]) == 0 and int(out.ctg_reg_off[-1]) == 0
    check_groups(regions, out, groups)


# ---------------------------------------------------------------------------------------------------------------------
# 6. the region cap
# ---------------------------------------------------------------------------------------------------------------------
CAP_K = 24
CAP_STRIDE = 257


def tiny_region(i):
    """region i of the 65,535-region call: empty, reads only, soft clips only, or a small insertion with its junction
    reads and soft clips, in turn"""
    rng = random.Random(90000 + i)
    kind = i % 4
    ref = _seq(rng, 100)
    name = "cap%05d" % i
    if kind == 0:
        return plain_region(name, CAP_K, ref, [], [])
    if kind == 1:
        return plain_region(name, CAP_K, ref, [ref[a:a + 40] for a in range(0, 60, 12)], [])
    if kind == 2:
        return plain_region(name, CAP_K, ref, [], [ref[10:50], _seq(rng, 40)])
    g = ref[:50] + _seq(rng, 20) + ref[50:]
    reads = [g[a:a + 40] for a in range(14, 62, 4)]
    return plain_region(name, CAP_K, ref, reads, [s for s in reads if s != ref[:40]])


def _oracle_tiny(i):
    r = tiny_region(i)
    only, row, _removed = expected_kstage(r, False)
    ctg = _oracle_contigs((only, r)) if i % CAP_STRIDE == 0 else None
    return only, row, expected_groups(r), ctg


@pytest.mark.skipif(EMULATED, reason="65,535 regions take the emulated library too long")
def test_65535_regions_in_one_call(pool, handle):
    R = MAX_REGIONS
    pending = pool.map_async(_oracle_tiny, range(R), chunksize=512)
    regions = [tiny_region(i) for i in range(R)]
    assert len(regions) == R
    assert cache_chunks(R, CAP_K) == [32768, 32767]
    pk, out, rows = run_call(handle, regions)
    exp = pending.get()
    for i, (only, row, _g, _c) in enumerate(exp):
        assert out.sample_only(i) == only, i
        assert rows[i] == row, i
    assert sum(len(e[0]) for e in exp) > 0
    check_groups(regions, out, [e[2] for e in exp])
    stride = range(0, R, CAP_STRIDE)
    for i in stride:
        assert out.contig_records(i) == exp[i][3], i
    assert sum(len(exp[i][3]) for i in stride) > 0

    # the same call on a reference k-mer cache built in two chunks
    handle.ref_cache_build([r.ref_fwd for r in regions], CAP_K)
    try:
        _pk, out_c, rows_c = run_call(handle, regions, with_ref=False)
    finally:
        handle.ref_cache_clear()
    assert rows_c == rows
    for name in ("so_off", "so_mers", "so_counts", "uniq_reg_off", "uniq_rec", "uniq_mult", "ctg_reg_off"):
        assert np.array_equal(getattr(out_c, name), getattr(out, name)), name
    for i in stride:
        assert out_c.contig_records(i) == exp[i][3], i


def test_65536_regions_are_refused(handle):
    regions = [plain_region("r%d" % i, CAP_K, "ACGT" * 10, [], []) for i in range(MAX_REGIONS + 1)]
    with pytest.raises(_lib.BreakmerError) as e:
        batch.run(handle, batch.PackedBatch(regions))
    assert e.value.code == _lib.BK_ERR_ARG
    small = [tiny_region(i) for i in range(3, 3 + 4 * 4, 4)]
    pk, out, rows = run_call(handle, small)
    check_kstage(small, pk, out, rows)
    check_groups(small, out)
