"""Host logic of sv_processor.compare_kmers_batch's chunked pass and of shard.run_sharded (no device: the pipeline, the
parser and the result application are replaced by recording fakes).  What is under test is the scheduling: every target
applied exactly once, never more chunks un-applied than there are handles, errors of either thread reach the caller
without a hang."""
import itertools
import threading
import time

import pytest

from breakmer_b200 import shard, sv_processor


class _T:
    def __init__(self, i, n_reads):
        self.name = "t%03d" % i
        self.cleaned_read_recs = {j: None for j in range(n_reads)}


class _FakePipe:
    def __init__(self, inflight, log):
        self.handles = list(range(inflight))
        self._queue = []
        self.log = log
        self.closed = False

    def full(self):
        return len(self._queue) >= len(self.handles)

    def pending(self):
        return len(self._queue)

    def submit(self, pk, tag=None):
        assert not self.full(), "submitted onto a busy handle"
        with self.log["lock"]:
            self.log["submitted"] += 1
            un_applied = self.log["submitted"] - self.log["applied"]
            self.log["max_unapplied"] = max(self.log["max_unapplied"], un_applied)
            assert un_applied <= len(self.handles), "a handle was reused before its chunk was applied"
        self._queue.append((pk, tag))

    def pop(self, decode=True):
        pk, tag = self._queue.pop(0)
        time.sleep(0.002)                                  # the device
        return ("res", pk), pk, tag

    def close(self):
        self.closed = True


def _new_log():
    return {"lock": threading.Lock(), "submitted": 0, "applied": 0, "max_unapplied": 0, "order": [], "threads": set(),
            "packed": 0, "slots": []}


def _install(monkeypatch, inflight, fail_apply_at=None, fail_pack_at=None):
    log = _new_log()
    pipe = _FakePipe(inflight, log)
    monkeypatch.setattr(sv_processor, "_get_pipe", lambda dev, n: pipe)
    monkeypatch.setattr(sv_processor, "_get_ingest", lambda slot=0: "ingest-%s" % slot)

    def pack(targets, ingest, slot=0):
        log["packed"] += 1
        log["slots"].append(slot)
        if fail_pack_at is not None and log["packed"] == fail_pack_at:
            raise ValueError("pack failed")
        time.sleep(0.001)
        return [t.name for t in targets], [15] * len(targets), None

    def apply(targets, pk, res, ks, objs, ingest, write_contigs, failed, ing=None):
        assert res == ("res", pk) and pk == [t.name for t in targets]
        if fail_apply_at is not None and log["applied"] + 1 == fail_apply_at:
            raise RuntimeError("apply failed")
        time.sleep(0.001)
        with log["lock"]:
            log["applied"] += 1
            log["order"].extend(t.name for t in targets)
            log["threads"].add(threading.get_ident())
        if any(t.name == "t007" for t in targets):
            failed.append("t007")

    monkeypatch.setattr(sv_processor, "_pack_targets", pack)
    monkeypatch.setattr(sv_processor, "_apply_chunk", apply)
    return log, pipe


@pytest.mark.parametrize("apply_thread", [False, True])
@pytest.mark.parametrize("n,max_targets,inflight", [(50, 7, 3), (50, 7, 1), (23, 5, 8), (9, 2, 2)])
def test_every_target_applied_once(monkeypatch, apply_thread, n, max_targets, inflight):
    log, pipe = _install(monkeypatch, inflight)
    targets = [_T(i, (i * 37) % 11) for i in range(n)]
    with pytest.raises(sv_processor.CapacityError) as e:      # the fake reports t007 as over the limit
        sv_processor.compare_kmers_batch(targets, ingest="native", max_targets=max_targets, inflight=inflight,
                                         apply_thread=apply_thread)
    assert e.value.targets == ["t007"]
    assert sorted(log["order"]) == sorted(t.name for t in targets)
    assert log["submitted"] == log["applied"] == -(-n // (-(-n // -(-n // max_targets))))
    assert 1 <= log["max_unapplied"] <= inflight
    assert (threading.get_ident() in log["threads"]) == (not apply_thread)
    # parse buffers rotate so that none is reused while its chunk is still in flight
    assert set(log["slots"]) <= set(range(inflight + (1 if apply_thread else 0)))
    assert not pipe.closed and pipe.pending() == 0


@pytest.mark.parametrize("apply_thread", [False, True])
def test_errors_of_either_side_reach_the_caller(monkeypatch, apply_thread):
    log, pipe = _install(monkeypatch, 3, fail_apply_at=2)
    monkeypatch.setattr(sv_processor, "_pipes", {})
    targets = [_T(i, 3) for i in range(40)]
    with pytest.raises(RuntimeError, match="apply failed"):
        sv_processor.compare_kmers_batch(targets, ingest="native", max_targets=5, apply_thread=apply_thread)
    assert pipe.closed                                        # a pipeline with batches in flight is not kept
    log, pipe = _install(monkeypatch, 3, fail_pack_at=4)
    with pytest.raises(ValueError, match="pack failed"):
        sv_processor.compare_kmers_batch(targets, ingest="native", max_targets=5, apply_thread=apply_thread)
    assert pipe.closed


class _Packed:
    def __init__(self, regions):
        self.names = [r.name for r in regions]


def _install_pipes(monkeypatch):
    """shard.DevicePipeline -> a _FakePipe with a log of its own per worker thread; -> (every pipe made, applied() to
    call from the thread that consumed a chunk)"""
    pipes = []
    mine = threading.local()

    def make(dev, inflight, **options):
        mine.pipe = _FakePipe(inflight, _new_log())
        pipes.append(mine.pipe)
        return mine.pipe

    def applied():
        with mine.pipe.log["lock"]:
            mine.pipe.log["applied"] += 1

    monkeypatch.setattr(shard, "DevicePipeline", make)
    return pipes, applied


@pytest.mark.parametrize("n,n_devices,max_regions,inflight", [(50, 1, 7, 3), (50, 3, 7, 2), (23, 2, 5, 1), (3, 4, 5, 2)])
def test_run_sharded_returns_every_region_once(monkeypatch, n, n_devices, max_regions, inflight):
    pipes, applied = _install_pipes(monkeypatch)
    regions = [_T(i, 0) for i in range(n)][::-1]                 # names against input order
    chunks = []

    def on_result(idx, out, pk):
        assert out == ("res", pk) and pk.names == [regions[i].name for i in idx]
        assert threading.get_ident() != here
        applied()
        chunks.append(idx)

    here = threading.get_ident()
    got = shard.run_sharded(regions, devices=list(range(n_devices)), max_regions=max_regions, inflight=inflight,
                            costs=[(i * 37) % 11 for i in range(n)], pack=_Packed, on_result=on_result)
    assert list(got) == sorted(r.name for r in regions)
    assert all(out[1].names[j] == name for name, (out, j) in got.items())
    assert sorted(i for idx in chunks for i in idx) == list(range(n))
    assert all(idx == sorted(idx) and len(idx) <= max_regions for idx in chunks)
    assert len(chunks) >= min(n, n_devices)
    assert len(pipes) == n_devices and all(p.closed and p.pending() == 0 for p in pipes)


@pytest.mark.parametrize("fail", ["pack", "consume"])
def test_run_sharded_errors_reach_the_caller(monkeypatch, fail):
    pipes, applied = _install_pipes(monkeypatch)
    regions = [_T(i, 3) for i in range(40)]
    calls = itertools.count(1)

    def pack(rs):
        if fail == "pack" and next(calls) == 4:
            raise ValueError("pack failed")
        return _Packed(rs)

    def on_result(idx, out, pk):
        if fail == "consume" and next(calls) == 2:
            raise RuntimeError("consume failed")
        applied()

    with pytest.raises(ValueError if fail == "pack" else RuntimeError, match=fail + " failed"):
        shard.run_sharded(regions, devices=[0, 1], max_regions=5, inflight=2, costs=[1.0] * 40, pack=pack,
                          on_result=on_result)
    assert len(pipes) == 2 and all(p.closed for p in pipes)
