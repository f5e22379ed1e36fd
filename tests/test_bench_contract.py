"""bench.py prints ONE JSON line with the keys the driver reads (both arms)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--workload", "C1", "--steps", "1", "--warmup", "0"], env={"BK_REF_BUDGET_S": "5"})
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "target_regions_assembled_per_sec" and d["unit"] == "regions/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0
    # both arms describe the workload with the same config object
    import bench
    assert d["config"] == bench.config_dict("C1", 1)


@pytest.mark.gpu
def test_gpu_arm_line():
    d = _run(["--regions", "60", "--steps", "8", "--warmup", "3", "--no-cpu-baseline"])
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["metric"] == "target_regions_assembled_per_sec" and d["n_gpus"] == 1 and d["steps"] == 8 and d["warmup"] == 3
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["from_files"]["value"] > 0 and d["from_files"]["n_contigs"] > 0
    assert d["with_ref_kmer_cache"]["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["sharding_check"]["equal_to_single_gpu_run"] is True and d["sharding_check"]["regions"] == 60
    assert d["e2e_dropin"]["value"] > 0 and d["run"]["host_threads_per_rank"] == 1
    assert all(v["frac"] is None or v["frac"] >= 0 for v in d["roofline_per_kernel"].values())


def _dumped_records(A, g, k):
    """region g of result_arrays(...) -> (sample-only {mer: count}, unique records, contig records with region-local
    read indices)"""
    import numpy as np
    from breakmer_b200 import _lib, batch
    off = {n: np.concatenate([[0], np.cumsum(A[n + "_len"])]).astype(np.int64)
           for n in ("so", "uniq", "ctg", "ctg_seq", "ctg_cnt", "ctg_reads", "ctg_kmers")}
    i = list(A["region"]).index(g)
    s = slice(off["so"][i], off["so"][i + 1])
    only = dict(zip(_lib.codes_to_mers(A["so_mers"][s].astype(np.uint64), k), A["so_counts"][s].astype(int).tolist()))
    s = slice(off["uniq"][i], off["uniq"][i + 1])
    uniq = list(zip(A["uniq_rec"][s].astype(int).tolist(), A["uniq_mult"][s].astype(int).tolist()))
    ctgs = []
    for c in range(off["ctg"][i], off["ctg"][i + 1]):
        sq, cn, rd, km = (slice(off[n][c], off[n][c + 1]) for n in ("ctg_seq", "ctg_cnt", "ctg_reads", "ctg_kmers"))
        ctgs.append({"seq": A["ctg_seq"][sq].astype(np.uint8).tobytes().decode(),
                     "indel_only": A["ctg_indel_only"][cn].astype(int).tolist(), "others": A["ctg_others"][cn].astype(int).tolist(),
                     "reads": A["ctg_reads"][rd].astype(int).tolist(),
                     "kmers": [list(t) for t in zip(_lib.codes_to_mers(A["ctg_kmer_mer"][km].astype(np.uint64), k),
                                                    A["ctg_kmer_pos"][km].astype(int).tolist(),
                                                    A["ctg_kmer_lth"][km].astype(int).tolist(),
                                                    A["ctg_kmer_dist"][km].astype(int).tolist(),
                                                    [batch.ORDER_NAMES[int(o)] for o in A["ctg_kmer_order"][km]])],
                     "kmer_locs": A["ctg_kmer_locs"][sq].astype(int).tolist()})
    return only, uniq, ctgs


@pytest.mark.gpu
def test_dumped_arrays_hold_the_batch_records():
    """result_arrays (what --dump-outputs writes) decodes to the records the library returned, and does not depend on
    how the regions were packed into calls; above its size limit it keeps the same seeded sample of whole regions"""
    import bench
    import numpy as np
    from breakmer_b200 import _lib, batch, synth
    regions = list(synth.config_regions("C2", 4, start=8)) + list(synth.config_regions("C5", 4, start=40))
    calls = [[0, 2, 4, 6], [1, 3, 5, 7]]
    h = _lib.Handle(0)
    try:
        packed = {c: batch.PackedBatch([regions[i] for i in calls[c]]) for c in range(2)}
        outs = {c: batch.run(h, packed[c]) for c in range(2)}
        A = bench.result_arrays(outs, calls, packed)
        assert A["region"].tolist() == list(range(8)) and all(a.dtype == np.float64 for a in A.values())
        for c in range(2):
            o, pk = outs[c], packed[c]
            for r, g in enumerate(calls[c]):
                base = int(pk.read_reg_off[r])
                a, b = o.uniq_reg_off[r], o.uniq_reg_off[r + 1]
                only, uniq, ctgs = _dumped_records(A, g, pk.k)
                assert only == o.sample_only(r)
                assert uniq == list(zip((o.uniq_rec[a:b] - base).tolist(), o.uniq_mult[a:b].tolist()))
                want = o.contig_records(r)
                assert len(ctgs) == len(want)
                for got, exp in zip(ctgs, want):
                    assert sorted(pk.read_ids[base + i] for i in got.pop("reads")) == exp.pop("reads")
                    assert got == exp
        one = {0: batch.PackedBatch(regions)}
        B = bench.result_arrays({0: batch.run(h, one[0])}, [list(range(8))], one)
    finally:
        h.close()
    assert A.keys() == B.keys() and all(np.array_equal(A[n], B[n]) for n in A)
    limit = sum(a.nbytes for a in A.values()) // 2
    S = bench.result_arrays(outs, calls, packed, limit)
    assert sum(a.nbytes for a in S.values()) <= limit and 0 < len(S["region"]) < 8
    for g in S["region"].astype(int):
        assert _dumped_records(S, g, 15) == _dumped_records(A, g, 15)
    S2 = bench.result_arrays(outs, calls, packed, limit)
    assert all(np.array_equal(S[n], S2[n]) for n in S)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_outputs_of_its_last_step(tmp_path):
    import bench
    import numpy as np
    from breakmer_b200 import _lib, batch, synth
    d = _run(["--regions", "24", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-ref-cache-leg", "--no-ingest-leg",
              "--no-dropin-leg", "--dump-outputs", str(tmp_path)])
    assert d["steps"] == 2
    got = {fn[:-4]: np.load(os.path.join(str(tmp_path), fn)) for fn in os.listdir(str(tmp_path))}
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_LIMIT
    packed = {0: batch.PackedBatch(list(synth.config_regions("C2", 24)))}
    h = _lib.Handle(0)
    try:
        want = bench.result_arrays({0: batch.run(h, packed[0])}, [list(range(24))], packed)
    finally:
        h.close()
    assert got.keys() == want.keys()
    for n in want:
        assert got[n].dtype == np.float64 and np.array_equal(got[n], want[n]), n
    assert got["ctg_len"].sum() > 0
