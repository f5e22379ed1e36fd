// C ABI of breakmer_b200 (include/breakmer_b200.h).  Host orchestration only:
// every byte of arithmetic on the hot path runs in the kernels of this
// directory.  There is no CPU fallback -- without a CUDA device bk_create fails.
#include "../../include/breakmer_b200.h"

#include <algorithm>
#include <functional>
#include <memory>

#include "host_util.cuh"
#include "kmers.cuh"
#include "region_kmers.cuh"
#include "nw_batch.cuh"
#include "nw_long.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "pipeline.cuh"
#include "assemble_long.cuh"
#include "ingest.cuh"
#include "dedup.cuh"

using namespace bk;

struct bk_handle_s {
  int device = 0;
  cudaStream_t st = nullptr;
  int sm_count = 148;
  int spec_width = 0;      // assembler speculation width (bk_set_option); 0 = choose per batch
  int long_regions = 0;    // bk_set_option "long_regions": the batched entries also assemble regions up to 65,535 bases
  cudaEvent_t sync_ev = nullptr;   // blocking-sync event (BK_BLOCKING_SYNC=1)
  bool spin_sync = true;
  Arena<false> dev;        // per-call device scratch
  Arena<true> pin;         // per-call pinned host staging / results
  Arena<false> resident;   // bk_batch_upload
  Arena<false> cache;      // bk_ref_cache_build
  const uint64_t* ref_cache_mers = nullptr;   // sorted reference k-mers per region (forward + reverse complement)
  const int64_t* ref_cache_koff = nullptr;    // n_regions + 1
  int ref_cache_regions = 0, ref_cache_k = 0;
  KernelTimers timers;
  std::string err;
  std::unique_ptr<Pipeline> pipe;
  PendingBatch pending;            // the batch between bk_batch_submit and bk_batch_wait
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // device time of a batch
  // bk_kernel_times result storage
  double kt_ms[KF_COUNT_];
  int64_t kt_launches[KF_COUNT_];
};

namespace {

// Wait for everything queued on the handle's stream.  Default: cudaStreamSynchronize (spins; lowest latency -- the
// pipeline has ~8 short waits per batch).  BK_BLOCKING_SYNC=1 makes waiting host threads sleep on a blocking event
// instead, for hosts with fewer cores than in-flight batches (measured on a 16-core B200 box: +1.3 ms per sequential
// step, no throughput gain with 6 batches in flight).
cudaError_t stream_wait(bk_handle_t h) {
  if (h->spin_sync || !h->sync_ev) return cudaStreamSynchronize(h->st);
  cudaError_t e = cudaEventRecord(h->sync_ev, h->st);
  if (e != cudaSuccess) return e;
  return cudaEventSynchronize(h->sync_ev);
}

template <typename F>
int guarded(bk_handle_t h, F&& f) {
  if (!h) return BK_ERR_ARG;
  try {
    BK_CUDA(cudaSetDevice(h->device));
    f();
    return BK_OK;
  } catch (const ApiError& e) {
    h->err = e.msg;
    return e.code;
  } catch (const CudaError& e) {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at api line %d: %s", (int)e.e, cudaGetErrorString(e.e), e.line, e.what);
    h->err = buf;
    cudaGetLastError();
    return e.e == cudaErrorMemoryAllocation ? BK_ERR_NOMEM : BK_ERR_CUDA;       // (out of device / pinned memory: not sticky)
  } catch (const std::bad_alloc&) {
    h->err = "host allocation failed";
    return BK_ERR_NOMEM;
  }
}

template <typename T>
T* to_device(bk_handle_t h, Arena<false>& a, const T* src, size_t n) {
  T* d = a.get<T>(n ? n : 1);
  if (n) BK_CUDA(cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, h->st));
  return d;
}

int bits_for(uint64_t n_values) {   // bits needed to represent 0 .. n_values-1
  int b = 0;
  while (b < 63 && (1ull << b) < n_values) ++b;
  return b;
}

// sort + run-length select + compaction on keys already emitted on the device.  Nothing here waits for the device: the
// number of selected k-mers stays in device memory (d_n) and every output is allocated for its upper bound `sel_cap`.
struct SelectOut {
  uint64_t* mers;         // device, written at [base, base + *d_n) where base = *dst_base_dev (or 0)
  uint32_t* counts;
  uint32_t* d_n;          // device: number of k-mers selected by this call
  uint32_t* seg_counts;   // device, n_seg (or null)
};

inline unsigned blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

// sel_cap: upper bound of the number of selected runs (SELECT_ALL selects at most n; a sample-only run holds a case k-mer).
SelectOut sort_and_select(bk_handle_t h, uint64_t* keys, uint32_t* vals, int64_t n, int k, int seg_bits, int mode,
                          int64_t n_seg, int64_t sel_cap) {
  SelectOut o{nullptr, nullptr, nullptr, nullptr};
  cudaStream_t st = h->st;
  if (n_seg > 0) {
    o.seg_counts = h->dev.get<uint32_t>(n_seg);
    BK_CUDA(cudaMemsetAsync(o.seg_counts, 0, n_seg * sizeof(uint32_t), st));
  }
  if (sel_cap > n) sel_cap = n;
  if (!o.mers) {
    o.mers = h->dev.get<uint64_t>(sel_cap ? sel_cap : 1);
    o.counts = h->dev.get<uint32_t>(sel_cap ? sel_cap : 1);
  }
  o.d_n = h->dev.get<uint32_t>(1);
  if (n == 0 || sel_cap == 0) {
    BK_CUDA(cudaMemsetAsync(o.d_n, 0, sizeof(uint32_t), st));
    return o;
  }
  const int64_t tiles = rs_num_tiles(n);
  RadixSortScratch sc;
  sc.keys_alt = h->dev.get<uint64_t>(n);
  sc.vals_alt = h->dev.get<uint32_t>(n);
  sc.table = h->dev.get<uint32_t>(256 * tiles);
  sc.scan_tmp = h->dev.get<uint32_t>(scan_tmp_elems(256 * tiles));
  uint64_t* sk;
  uint32_t* sv;
  const int key_bits = 2 * k + seg_bits + 1;   // +1: the all-ones invalid key sorts last
  radix_sort_pairs(keys, vals, n, key_bits, sc, st, &sk, &sv, h->timers);
  RunParams rp{};
  rp.keys = sk; rp.vals = sv; rp.n = n; rp.k = k; rp.mode = mode;
  rp.flags = h->dev.get<uint32_t>(n);
  rp.run_count = h->dev.get<uint32_t>(n);
  uint32_t* pos = h->dev.get<uint32_t>(n);
  uint32_t* scan_tmp = h->dev.get<uint32_t>(scan_tmp_elems(n));
  const unsigned blocks = blocks_for(n, 256);
  {
    TimedLaunch t(h->timers, st, KF_RUN_SELECT);
    run_select_kernel<<<blocks, 256, 0, st>>>(rp);
  }
  {
    TimedLaunch t(h->timers, st, KF_SCAN, 3);
    exclusive_scan_u32(rp.flags, pos, n, scan_tmp, o.d_n, st);
  }
  rp.pos = pos;
  rp.out_mers = o.mers; rp.out_counts = o.counts; rp.seg_counts = o.seg_counts;
  TimedLaunch t(h->timers, st, KF_RUN_SCATTER);
  run_scatter_kernel<<<blocks, 256, 0, st>>>(rp);
  BK_CUDA(cudaGetLastError());
  return o;
}

// number of k-mers a finished select produced (host round trip; used by the small entry points only)
int64_t select_count(bk_handle_t h, const SelectOut& so) {
  uint32_t* hn = h->pin.get<uint32_t>(1);
  BK_CUDA(cudaMemcpyAsync(hn, so.d_n, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
  BK_CUDA(stream_wait(h));
  return (int64_t)*hn;
}

}  // namespace

// expose helpers to pipeline.cu-style code in this TU
#include "pipeline_impl.cuh"

extern "C" {

int bk_version(void) { return 1; }

int bk_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int bk_create(int device, bk_handle_t* out) {
  if (!out) return BK_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return BK_ERR_CUDA; }   // no fallback
  if (device < 0 || device >= n) return BK_ERR_ARG;
  bk_handle_t h = new (std::nothrow) bk_handle_s();
  if (!h) return BK_ERR_NOMEM;
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    delete h;
    return BK_ERR_CUDA;
  }
  cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (cudaEventCreateWithFlags(&h->sync_ev, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError();
    h->sync_ev = nullptr;
  }
  h->spin_sync = getenv("BK_BLOCKING_SYNC") == nullptr;
  if (cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) {
    cudaGetLastError();
    cudaStreamDestroy(h->st);
    delete h;
    return BK_ERR_CUDA;
  }
  *out = h;
  return BK_OK;
}

int bk_destroy(bk_handle_t h) {
  if (!h) return BK_ERR_ARG;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->st);
  if (h->sync_ev) cudaEventDestroy(h->sync_ev);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  h->pipe.reset();
  h->dev.release();
  h->pin.release();
  h->resident.release();
  h->cache.release();
  cudaStreamDestroy(h->st);
  delete h;
  return BK_OK;
}

const char* bk_last_error(bk_handle_t h) { return h ? h->err.c_str() : "null handle"; }

}  // extern "C"

namespace {

// Sequences and per-warp scratch kept on the device between the launches of one call (bk_dedup_reads aligns the same
// reads round after round): filled by the first nw_batch_run of the call, reused by the others.
struct NwResident {
  const uint8_t* seqs = nullptr;
  const int64_t* seq_off = nullptr;
  uint2* lastcol = nullptr;
  int2* edge = nullptr;
  uint8_t* tab = nullptr;
};

// Body of bk_nw_batch.  keep == nullptr: a self-contained call (arenas reset, everything uploaded).
void nw_batch_run(bk_handle_t h, const char* seqs, const int64_t* seq_off, int64_t n_seq, const int32_t* pair_a,
                  const int32_t* pair_b, int64_t n_pairs, int32_t* out, int want_aln, char* aln1, char* aln2,
                  const int64_t* aln_off, int32_t* aln_len, NwResident* keep) {
  {
    if (n_pairs < 0 || n_seq < 0 || (n_pairs > 0 && (!seqs || !seq_off || !pair_a || !pair_b || !out)))
      fail(BK_ERR_ARG, "bk_nw_batch: null argument");
    if (want_aln && (!aln1 || !aln2 || !aln_off || !aln_len)) fail(BK_ERR_ARG, "bk_nw_batch: alignment buffers missing");
    if (n_pairs == 0) return;
    const bool first = !keep || !keep->seqs;
    if (!keep) {
      h->dev.reset();
      h->pin.reset();
    }
    if (n_seq > 0 && seq_off) {                        // the whole table is uploaded: all of it must be a valid offset table
      if (seq_off[0] != 0) fail(BK_ERR_ARG, "bk_nw_batch: seq_off must start at 0");
      for (int64_t q = 0; q < n_seq; ++q)
        if (seq_off[q + 1] < seq_off[q]) fail(BK_ERR_ARG, "bk_nw_batch: seq_off not monotone at %lld", (long long)q);
    }
    int max_m = 0;
    std::vector<int64_t> ptr_off, long_idx, long_ptr_off;
    int64_t ptr_total = 0, aln_total = 0, aln_end_prev = 0, long_max = 0, long_ptr_total = 0;
    if (want_aln) ptr_off.resize(n_pairs);
    for (int64_t p = 0; p < n_pairs; ++p) {
      const int a = pair_a[p], b = pair_b[p];
      if (a < 0 || a >= n_seq || b < 0 || b >= n_seq) fail(BK_ERR_ARG, "bk_nw_batch: pair %lld out of range", (long long)p);
      const int64_t m = seq_off[a + 1] - seq_off[a], n = seq_off[b + 1] - seq_off[b];
      if (m <= 0 || n <= 0) fail(BK_ERR_EMPTY_SEQ, "nw: empty sequence in pair %lld (olc.nw raises NameError)", (long long)p);
      // olc.nw has no length limit (olc.py:40-52): pairs beyond the packed-cell kernels' 4095 bases take nw_long_kernel
      const bool is_long = m > NW_MAX_LEN || n > NW_MAX_LEN;
      if (m >= (int64_t(1) << 30) || n >= (int64_t(1) << 30))
        fail(BK_ERR_CAPACITY, "nw: sequence of 2^30 bases or more in pair %lld", (long long)p);
      if (is_long) {
        long_idx.push_back(p);
        long_max = std::max(long_max, std::max(m, n));
      } else {
        max_m = std::max<int>(max_m, (int)m);
      }
      if (want_aln) {
        // the two strings of pair p occupy [aln_off[p], aln_off[p] + m + n): non-negative, and not overlapping the next pair's
        if (aln_off[p] < 0 || (p > 0 && aln_off[p] < aln_end_prev))
          fail(BK_ERR_ARG, "bk_nw_batch: aln_off[%lld] is negative or overlaps the previous pair's strings", (long long)p);
        aln_end_prev = aln_off[p] + m + n;
        if (is_long) {
          long_ptr_off.push_back(long_ptr_total);
          long_ptr_total += (m + 1) * (n + 1);
          ptr_off[p] = 0;
        } else {
          ptr_off[p] = ptr_total;
          ptr_total += (m + 1) * (n + 1);
        }
        aln_total = std::max<int64_t>(aln_total, aln_off[p] + m + n);
      }
    }
    NwBatchParams P{};
    if (first) {
      P.seqs = (const uint8_t*)to_device(h, h->dev, seqs, (size_t)seq_off[n_seq]);
      P.seq_off = to_device(h, h->dev, seq_off, (size_t)n_seq + 1);
    } else {
      P.seqs = keep->seqs;
      P.seq_off = keep->seq_off;
    }
    P.pair_a = to_device(h, h->dev, pair_a, (size_t)n_pairs);
    P.pair_b = to_device(h, h->dev, pair_b, (size_t)n_pairs);
    P.n_pairs = n_pairs;
    P.out = h->dev.get<int32_t>(n_pairs * 10);
    int64_t want_blocks = (n_pairs + NWB_WARPS - 1) / NWB_WARPS;
    const int grid = (int)std::min<int64_t>(want_blocks, (int64_t)h->sm_count * 8);
    const bool use_tab = !want_aln && !getenv("BK_NW_PACKED");      // score pass + traceback (nw.cuh) where its table fits
    if (!keep) {
      if (use_tab) P.tab = h->dev.get<uint8_t>((size_t)grid * NWB_WARPS * NW_TAB_BYTES);
      if (max_m > 256) {
        P.edge_stride = NW_MAX_LEN + 1;
        P.edge = h->dev.get<int2>((size_t)grid * NWB_WARPS * 2 * P.edge_stride);
      }
      P.lastcol = h->dev.get<uint2>((size_t)grid * NWB_WARPS * (NW_MAX_LEN / 2 + 1));
    } else {
      if (first) {                                   // scratch for the largest grid and the longest sequence of the call
        const size_t warps = (size_t)h->sm_count * 8 * NWB_WARPS;
        int64_t longest = 0;
        for (int64_t q = 0; q < n_seq; ++q) longest = std::max(longest, seq_off[q + 1] - seq_off[q]);
        keep->seqs = P.seqs;
        keep->seq_off = P.seq_off;
        keep->edge = longest > 256 ? h->dev.get<int2>(warps * 2 * (NW_MAX_LEN + 1)) : nullptr;
        keep->lastcol = h->dev.get<uint2>(warps * (NW_MAX_LEN / 2 + 1));
        keep->tab = use_tab ? h->dev.get<uint8_t>(warps * NW_TAB_BYTES) : nullptr;
      }
      P.tab = keep->tab;
      if (max_m > 256) {
        P.edge_stride = NW_MAX_LEN + 1;
        P.edge = keep->edge;
      }
      P.lastcol = keep->lastcol;
    }
    P.want_aln = want_aln;
    if (want_aln) {
      P.ptr_scratch = h->dev.get<uint8_t>(ptr_total);
      P.ptr_off = to_device(h, h->dev, ptr_off.data(), (size_t)n_pairs);
      P.aln1 = h->dev.get<uint8_t>(aln_total);
      P.aln2 = h->dev.get<uint8_t>(aln_total);
      P.aln_off = to_device(h, h->dev, aln_off, (size_t)n_pairs);
      P.aln_len = h->dev.get<int32_t>(n_pairs);
    }
    {
      TimedLaunch t(h->timers, h->st, KF_NW_BATCH);
      nw_batch_kernel<<<grid, NWB_WARPS * 32, 0, h->st>>>(P);
    }
    BK_CUDA(cudaGetLastError());
    if (!long_idx.empty()) {                           // rare: one CTA per (pair, direction), 32-bit anti-diagonal sweep
      NwLongParams Q{};
      const size_t n_long = long_idx.size();
      Q.seqs = P.seqs;
      Q.seq_off = P.seq_off;
      Q.pair_a = P.pair_a;
      Q.pair_b = P.pair_b;
      Q.long_idx = to_device(h, h->dev, long_idx.data(), n_long);
      Q.out = P.out;
      Q.diag_stride = (long_max + 1 + 31) & ~int64_t(31);
      Q.diag = h->dev.get<int32_t>(2 * n_long * 9 * (size_t)Q.diag_stride);
      Q.want_aln = want_aln;
      if (want_aln) {
        Q.ptr_scratch = h->dev.get<uint8_t>((size_t)long_ptr_total);
        Q.ptr_off = to_device(h, h->dev, long_ptr_off.data(), n_long);
        Q.aln1 = P.aln1;
        Q.aln2 = P.aln2;
        Q.aln_off = P.aln_off;
        Q.aln_len = P.aln_len;
      }
      if (2 * n_long > (size_t)0x7fffffff) fail(BK_ERR_CAPACITY, "bk_nw_batch: more than 2^30 pairs above %d bases", NW_MAX_LEN);
      {
        TimedLaunch t(h->timers, h->st, KF_NW_BATCH);
        nw_long_kernel<<<(unsigned)(2 * n_long), NWL_THREADS, 0, h->st>>>(Q);
      }
      BK_CUDA(cudaGetLastError());
    }
    BK_CUDA(cudaMemcpyAsync(out, P.out, n_pairs * 10 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    if (want_aln) {
      BK_CUDA(cudaMemcpyAsync(aln1, P.aln1, aln_total, cudaMemcpyDeviceToHost, h->st));
      BK_CUDA(cudaMemcpyAsync(aln2, P.aln2, aln_total, cudaMemcpyDeviceToHost, h->st));
      BK_CUDA(cudaMemcpyAsync(aln_len, P.aln_len, n_pairs * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    }
    BK_CUDA(stream_wait(h));
    if (want_aln) {
      // the device walks the traceback from the end cell, so the strings arrive
      // end-first (olc.py:92-102 prepends); put them in reading order
      for (int64_t p = 0; p < n_pairs; ++p) {
        std::reverse(aln1 + aln_off[p], aln1 + aln_off[p] + aln_len[p]);
        std::reverse(aln2 + aln_off[p], aln2 + aln_off[p] + aln_len[p]);
      }
    }
  }
}

}  // namespace

extern "C" {

int bk_nw_batch(bk_handle_t h, const char* seqs, const int64_t* seq_off, int64_t n_seq, const int32_t* pair_a,
                const int32_t* pair_b, int64_t n_pairs, int32_t* out, int want_aln, char* aln1, char* aln2,
                const int64_t* aln_off, int32_t* aln_len) {
  return guarded(h, [&] {
    nw_batch_run(h, seqs, seq_off, n_seq, pair_a, pair_b, n_pairs, out, want_aln, aln1, aln2, aln_off, aln_len, nullptr);
  });
}

// read_batch.check_mer_read of the reference's older assembler variant (sv_assembly_mm2.py:290-355) for whole batches:
// the alignments the decision chains need go through nw_batch_kernel a round at a time for all batches together, and
// the chains are replayed on the host from the score table (csrc/dedup.cuh).
int bk_dedup_reads(bk_handle_t h, const char* seqs, const int64_t* seq_off, int64_t n_reads, const int32_t* mer_pos,
                   const int64_t* batch_off, int64_t n_batches, double subseq_frac, uint8_t* check, uint8_t* flags,
                   int64_t* n_pairs_out, int32_t* n_launches_out) {
  if (!h) return BK_ERR_ARG;
  int rc = guarded(h, [&] {
    if (n_reads < 0 || n_batches < 0 || (n_reads > 0 && (!seqs || !seq_off || !mer_pos || !check || !flags)) ||
        (n_batches > 0 && !batch_off) || (n_batches == 0 && n_reads != 0))
      fail(BK_ERR_ARG, "bk_dedup_reads: null argument");
    if (!(subseq_frac > 0.0 && subseq_frac <= 1.0)) fail(BK_ERR_ARG, "bk_dedup_reads: subseq_frac must be in (0, 1]");
    if (n_reads >= (int64_t(1) << 31)) fail(BK_ERR_CAPACITY, "bk_dedup_reads: more than 2^31 reads in one call");
    for (int64_t b = 0; b < n_batches; ++b) {
      const int64_t lo = batch_off[b], hi = batch_off[b + 1];
      if (lo < 0 || hi < lo || hi > n_reads || (b == 0 && lo != 0) || (b + 1 == n_batches && hi != n_reads))
        fail(BK_ERR_ARG, "bk_dedup_reads: batch_off must partition the reads");
      if (hi == lo) fail(BK_ERR_ARG, "bk_dedup_reads: batch %lld is empty (a batch is opened by its first read)", (long long)b);
    }
  });
  if (rc != BK_OK) return rc;
  if (n_pairs_out) *n_pairs_out = 0;
  if (n_launches_out) *n_launches_out = 0;
  if (n_batches == 0) return BK_OK;
  int rounds = 0;
  NwResident keep;                                   // reads uploaded once, reused by every round's launch
  rc = guarded(h, [&] {
    h->err.clear();
    h->dev.reset();
    h->pin.reset();
  });
  if (rc != BK_OK) return rc;
  rc = dedup_run(seq_off, mer_pos, batch_off, n_batches, subseq_frac, check, flags, n_pairs_out, &rounds,
                 [&](const int32_t* pa, const int32_t* pb, int64_t n, int32_t* out) {
                   return guarded(h, [&] {
                     nw_batch_run(h, seqs, seq_off, n_reads, pa, pb, n, out, 0, nullptr, nullptr, nullptr, nullptr, &keep);
                   });
                 });
  if (n_launches_out) *n_launches_out = rounds;
  if (rc == BK_ERR_CAPACITY && h->err.empty()) h->err = "bk_dedup_reads: too many read pairs in one launch";
  return rc;
}

int bk_count_kmers(bk_handle_t h, const char* bases, const int64_t* rec_off, int64_t n_rec, const uint32_t* rec_mult,
                   int k, const uint64_t** mers, const uint32_t** counts, int64_t* n_out) {
  return guarded(h, [&] {
    if (!mers || !counts || !n_out || n_rec < 0 || (n_rec > 0 && (!bases || !rec_off)))
      fail(BK_ERR_ARG, "bk_count_kmers: null argument");
    if (k < 1 || k > 31) fail(BK_ERR_ARG, "bk_count_kmers: k must be in 1..31");
    h->dev.reset();
    h->pin.reset();
    *mers = nullptr; *counts = nullptr; *n_out = 0;
    // drop empty records (they hold no window) so record starts are distinct
    std::vector<int64_t> off;
    std::vector<uint32_t> mult;
    off.reserve(n_rec + 1);
    for (int64_t r = 0; r < n_rec; ++r) {
      if (rec_off[r + 1] < rec_off[r]) fail(BK_ERR_ARG, "bk_count_kmers: rec_off not monotone");
      if (rec_off[r + 1] > rec_off[r]) {
        off.push_back(rec_off[r] - rec_off[0]);
        if (rec_mult) mult.push_back(rec_mult[r]);
      }
    }
    const int64_t n_bases = n_rec ? rec_off[n_rec] - rec_off[0] : 0;
    if (n_bases >= (int64_t(1) << 31)) fail(BK_ERR_CAPACITY, "bk_count_kmers: more than 2^31 bases in one call");
    off.push_back(n_bases);
    if (n_bases == 0) return;
    EmitParams E{};
    E.bases = (const uint8_t*)to_device(h, h->dev, bases + rec_off[0], (size_t)n_bases);
    E.n_bases = n_bases;
    E.rec_off = to_device(h, h->dev, off.data(), off.size());
    E.n_rec = (int64_t)off.size() - 1;
    E.rec_mult = rec_mult ? to_device(h, h->dev, mult.data(), mult.size()) : nullptr;
    E.k = k; E.tag = 0; E.emit_rc = 0;
    E.keys = h->dev.get<uint64_t>(n_bases);
    E.vals = h->dev.get<uint32_t>(n_bases);
    {
      TimedLaunch t(h->timers, h->st, KF_EMIT);
      kmer_emit_kernel<<<(unsigned)((n_bases + EMIT_TILE - 1) / EMIT_TILE), EMIT_THREADS, 0, h->st>>>(E);
    }
    SelectOut so = sort_and_select(h, E.keys, E.vals, n_bases, k, 0, SELECT_ALL, 0, n_bases);
    const int64_t n_sel = select_count(h, so);
    uint64_t* hm = h->pin.get<uint64_t>(n_sel ? n_sel : 1);
    uint32_t* hc = h->pin.get<uint32_t>(n_sel ? n_sel : 1);
    if (n_sel) {
      BK_CUDA(cudaMemcpyAsync(hm, so.mers, n_sel * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->st));
      BK_CUDA(cudaMemcpyAsync(hc, so.counts, n_sel * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    }
    BK_CUDA(stream_wait(h));
    *mers = hm; *counts = hc; *n_out = n_sel;
  });
}

int bk_sample_only(bk_handle_t h, int k, const uint64_t* case_mers, const uint32_t* case_counts, int64_t n_case,
                   const uint64_t* sc_mers, int64_t n_sc, const uint64_t* ref_mers, int64_t n_ref,
                   const uint64_t* normal_mers, int64_t n_normal, const uint64_t** mers, const uint32_t** counts,
                   int64_t* n_out) {
  return guarded(h, [&] {
    if (!mers || !counts || !n_out) fail(BK_ERR_ARG, "bk_sample_only: null output");
    if (k < 1 || k > 31) fail(BK_ERR_ARG, "bk_sample_only: k must be in 1..31");
    if ((n_case && (!case_mers || !case_counts)) || (n_sc && !sc_mers) || (n_ref && !ref_mers) || (n_normal && !normal_mers))
      fail(BK_ERR_ARG, "bk_sample_only: null input");
    h->dev.reset();
    h->pin.reset();
    *mers = nullptr; *counts = nullptr; *n_out = 0;
    const int64_t n = n_case + n_sc + n_ref + n_normal;
    if (n == 0) return;
    // one key per (mer, set); the device sorts them so that the sets of a mer
    // become adjacent, then run_select applies (case & sc) - ref - normal
    uint64_t* hk = h->pin.get<uint64_t>(n);
    uint32_t* hv = h->pin.get<uint32_t>(n);
    int64_t w = 0;
    for (int64_t i = 0; i < n_case; ++i, ++w) {
      if (case_counts[i] >= (1u << 30)) fail(BK_ERR_CAPACITY, "bk_sample_only: a count exceeds 2^30");
      hk[w] = case_mers[i]; hv[w] = case_counts[i] | ((uint32_t)TAG_CASE << 30);
    }
    for (int64_t i = 0; i < n_sc; ++i, ++w) { hk[w] = sc_mers[i]; hv[w] = 1u | ((uint32_t)TAG_SC << 30); }
    for (int64_t i = 0; i < n_ref; ++i, ++w) { hk[w] = ref_mers[i]; hv[w] = 1u | ((uint32_t)TAG_REF << 30); }
    for (int64_t i = 0; i < n_normal; ++i, ++w) { hk[w] = normal_mers[i]; hv[w] = 1u | ((uint32_t)TAG_NORMAL << 30); }
    uint64_t* dk = to_device(h, h->dev, hk, (size_t)n);
    uint32_t* dv = to_device(h, h->dev, hv, (size_t)n);
    SelectOut so = sort_and_select(h, dk, dv, n, k, 0, SELECT_SAMPLE_ONLY, 0, n_case);
    const int64_t n_sel = select_count(h, so);
    uint64_t* hm = h->pin.get<uint64_t>(n_sel ? n_sel : 1);
    uint32_t* hc = h->pin.get<uint32_t>(n_sel ? n_sel : 1);
    if (n_sel) {
      BK_CUDA(cudaMemcpyAsync(hm, so.mers, n_sel * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->st));
      BK_CUDA(cudaMemcpyAsync(hc, so.counts, n_sel * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    }
    BK_CUDA(stream_wait(h));
    *mers = hm; *counts = hc; *n_out = n_sel;
  });
}

// On a failed submit the stream may hold work that uses the arenas: drain it so that the handle is reusable.
static int submit_guarded(bk_handle_t h, const bk_batch_input* in, LongMode mode) {
  if (h && h->pending.active) {                     // refused without touching the batch that is in flight
    h->err = "a batch is already in flight on this handle (call bk_batch_wait first)";
    return BK_ERR_ARG;
  }
  const int rc = guarded(h, [&] { pipeline_submit(h, in, mode); });
  if (rc != BK_OK && h) { cudaStreamSynchronize(h->st); cudaGetLastError(); h->pending.active = false; }
  return rc;
}
static int wait_guarded(bk_handle_t h, bk_batch_result* out) {
  if (h && !h->pending.active) { h->err = "bk_batch_wait: no batch in flight on this handle"; return BK_ERR_ARG; }
  const int rc = guarded(h, [&] { pipeline_wait(h, out); });
  if (rc != BK_OK && h) { cudaStreamSynchronize(h->st); cudaGetLastError(); h->pending.active = false; }
  return rc;
}

int bk_batch_submit(bk_handle_t h, const bk_batch_input* in) {
  if (h && !in && !h->pipe) { h->err = "bk_batch_submit: null input and no batch uploaded"; return BK_ERR_ARG; }
  return submit_guarded(h, in, option_mode(h));
}

int bk_batch_wait(bk_handle_t h, bk_batch_result* out) {
  if (h && !out) { h->err = "bk_batch_wait: null argument"; return BK_ERR_ARG; }
  return wait_guarded(h, out);
}

int bk_compare_kmers_batch(bk_handle_t h, const bk_batch_input* in, bk_batch_result* out) {
  if (h && (!in || !out)) { h->err = "bk_compare_kmers_batch: null argument"; return BK_ERR_ARG; }
  const int rc = submit_guarded(h, in, option_mode(h));
  return rc != BK_OK ? rc : wait_guarded(h, out);
}

int bk_compare_kmers_long(bk_handle_t h, const bk_batch_input* in, bk_batch_result* out) {
  if (h && (!in || !out)) { h->err = "bk_compare_kmers_long: null argument"; return BK_ERR_ARG; }
  const int rc = submit_guarded(h, in, LONG_ALL);
  return rc != BK_OK ? rc : wait_guarded(h, out);
}

int bk_batch_upload(bk_handle_t h, const bk_batch_input* in) {
  return guarded(h, [&] {
    if (!in) fail(BK_ERR_ARG, "bk_batch_upload: null argument");
    pipeline_upload(h, in);
  });
}

int bk_compare_kmers_resident(bk_handle_t h, bk_batch_result* out) {
  if (h && !out) { h->err = "bk_compare_kmers_resident: null argument"; return BK_ERR_ARG; }
  if (h && !h->pipe) { h->err = "bk_compare_kmers_resident: no batch uploaded"; return BK_ERR_ARG; }
  const int rc = submit_guarded(h, nullptr, option_mode(h));
  return rc != BK_OK ? rc : wait_guarded(h, out);
}

int bk_ref_cache_build(bk_handle_t h, const char* ref_bases, const int64_t* ref_off, int32_t n_regions, int32_t k) {
  return guarded(h, [&] {
    if (!ref_off || n_regions < 0 || (n_regions > 0 && ref_off[n_regions] > 0 && !ref_bases)) fail(BK_ERR_ARG, "bk_ref_cache_build: null argument");
    if (k < 2 || k > 31) fail(BK_ERR_ARG, "bk_ref_cache_build: k must be in 2..31");
    ref_cache_build(h, ref_bases, ref_off, n_regions, k);
  });
}

int bk_ref_cache_clear(bk_handle_t h) {
  return guarded(h, [&] {
    BK_CUDA(stream_wait(h));
    h->cache.reset();
    h->ref_cache_mers = nullptr; h->ref_cache_koff = nullptr; h->ref_cache_regions = 0; h->ref_cache_k = 0;
  });
}

int bk_set_option(bk_handle_t h, const char* name, int64_t value) {
  return guarded(h, [&] {
    if (!name) fail(BK_ERR_ARG, "bk_set_option: null name");
    if (strcmp(name, "spec_width") == 0) {
      if (value != 0 && value != 1 && value != 2 && value != 4 && value != 8) fail(BK_ERR_ARG, "spec_width must be 0 (auto), 1, 2, 4 or 8");
      h->spec_width = (int)value;
    } else if (strcmp(name, "blocking_sync") == 0) {
      h->spin_sync = value == 0;
    } else if (strcmp(name, "long_regions") == 0) {
      if (value != 0 && value != 1) fail(BK_ERR_ARG, "long_regions must be 0 or 1");
      h->long_regions = (int)value;
    } else {
      fail(BK_ERR_ARG, "bk_set_option: unknown option %s", name);
    }
  });
}

static_assert(RR_FIELDS == BK_RR_FIELDS && RR_REASON == BK_RR_REASON && RR_PASS == BK_RR_PASS &&
                  RR_FIRST_REASON == BK_RR_FIRST_REASON && RR_SEEDS == BK_RR_SEEDS && RR_FIND_READS == BK_RR_FIND_READS &&
                  RR_CHECK_ALIGN == BK_RR_CHECK_ALIGN && RR_GROWN == BK_RR_GROWN && RR_REJ_SUPPORT == BK_RR_REJ_SUPPORT &&
                  RR_REJ_LENGTH == BK_RR_REJ_LENGTH,
              "report fields of common.cuh and include/breakmer_b200.h differ");
static_assert(RR_OK == BK_RR_OK && RR_READ_TOO_LONG == BK_RR_READ_TOO_LONG && RR_CONTIG_TOO_LONG == BK_RR_CONTIG_TOO_LONG &&
                  RR_KMER_LIST_FULL == BK_RR_KMER_LIST_FULL && RR_TOO_MANY_CONTIGS == BK_RR_TOO_MANY_CONTIGS &&
                  RR_OUTPUT_ARENA == BK_RR_OUTPUT_ARENA && RR_PASS_NONE == BK_RR_PASS_NONE &&
                  RR_PASS_BATCHED == BK_RR_PASS_BATCHED && RR_PASS_LONG == BK_RR_PASS_LONG,
              "report codes of common.cuh and include/breakmer_b200.h differ");

int bk_region_report(bk_handle_t h, const int32_t** table, int32_t* n_fields) {
  return guarded(h, [&] {
    if (!table || !n_fields) fail(BK_ERR_ARG, "bk_region_report: null argument");
    *table = region_report(h);
    *n_fields = RR_FIELDS;
  });
}

int bk_kernel_times(bk_handle_t h, const char** names, const double** ms, const int64_t** launches, int32_t* n) {
  return guarded(h, [&] {
    h->timers.collect();
    for (int i = 0; i < KF_COUNT_; ++i) { h->kt_ms[i] = h->timers.ms[i]; h->kt_launches[i] = h->timers.launches[i]; }
    if (names) *names = kKernelFamilyNames;
    if (ms) *ms = h->kt_ms;
    if (launches) *launches = h->kt_launches;
    if (n) *n = KF_COUNT_;
  });
}

int bk_kernel_times_reset(bk_handle_t h, int enable) {
  return guarded(h, [&] {
    BK_CUDA(stream_wait(h));
    h->timers.reset();
    h->timers.enabled = enable != 0;
  });
}

}  // extern "C"

// ---- ingest (host threads; see ingest.cuh) ---------------------------------------------------
struct bk_ingest_s {
  Ingest g;
};

namespace {
template <typename F>
int guarded_ingest(bk_ingest_t g, F&& f) {
  if (!g) return BK_ERR_ARG;
  try {
    f();
    return BK_OK;
  } catch (const ApiError& e) {
    g->g.err = e.msg;
    return e.code;
  } catch (const CudaError& e) {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at ingest line %d: %s", (int)e.e, cudaGetErrorString(e.e), e.line, e.what);
    g->g.err = buf;
    cudaGetLastError();
    return BK_ERR_CUDA;
  } catch (const std::bad_alloc&) {
    g->g.err = "host allocation failed";
    return BK_ERR_NOMEM;
  }
}
void fill_text(const IngestText& t, bk_ingest_text* out) {
  if (!out) return;
  out->id_bytes = t.id_bytes; out->id_off = t.id_off;
  out->qual_bytes = t.qual_bytes; out->qual_off = t.qual_off;
  out->n_reads = t.n_reads; out->read_flags = t.read_flags;
}
}  // namespace

extern "C" {

int bk_ingest_create(int n_threads, int pinned, bk_ingest_t* out) {
  if (!out) return BK_ERR_ARG;
  *out = nullptr;
  if (pinned) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); return BK_ERR_CUDA; }
  }
  bk_ingest_s* g = new (std::nothrow) bk_ingest_s();
  if (!g) return BK_ERR_NOMEM;
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  g->g.n_threads = std::max(1, std::min(n_threads, 256));
  g->g.pinned = pinned != 0;
  g->g.buf.pinned = g->g.pinned;
  *out = g;
  return BK_OK;
}

int bk_ingest_destroy(bk_ingest_t g) {
  if (!g) return BK_ERR_ARG;
  delete g;
  return BK_OK;
}

const char* bk_ingest_last_error(bk_ingest_t g) { return g ? g->g.err.c_str() : "null ingest handle"; }

int bk_ingest_buffers(bk_ingest_t g, int32_t n_regions, const bk_text* ref_fa, const bk_text* reads_fq,
                      const bk_text* sc_fa, const bk_text* normal_fq, bk_batch_input* in, bk_ingest_text* text) {
  return guarded_ingest(g, [&] {
    if (n_regions < 0 || !in) fail(BK_ERR_ARG, "bk_ingest_buffers: bad arguments");
    auto views = [&](const bk_text* t, std::vector<TextView>& v) -> const TextView* {
      if (!t) return nullptr;
      v.resize((size_t)n_regions);
      for (int r = 0; r < n_regions; ++r) v[r] = TextView{t[r].p, t[r].p ? (size_t)t[r].n : 0};
      return v.data();
    };
    std::vector<TextView> a, b, c, d;
    IngestText t{};
    ingest_texts(g->g, n_regions, views(ref_fa, a), views(reads_fq, b), views(sc_fa, c), views(normal_fq, d), in, &t);
    fill_text(t, text);
  });
}

int bk_ingest_files(bk_ingest_t g, int32_t n_regions, const char* const* ref_fa, const char* const* reads_fq,
                    const char* const* sc_fa, const char* const* normal_fq, bk_batch_input* in, bk_ingest_text* text) {
  return guarded_ingest(g, [&] {
    if (n_regions < 0 || !in) fail(BK_ERR_ARG, "bk_ingest_files: bad arguments");
    Ingest& G = g->g;
    const char* const* lists[4] = {ref_fa, reads_fq, sc_fa, normal_fq};
    G.file_text.assign((size_t)n_regions * 4, std::string());
    std::vector<TextView> v[4];
    std::vector<int> bad((size_t)n_regions, -1);
    for (int s = 0; s < 4; ++s) if (lists[s]) v[s].assign((size_t)n_regions, TextView{nullptr, 0});
    G.parallel_for(n_regions, [&](int r) {
      for (int s = 0; s < 4; ++s) {
        if (!lists[s] || !lists[s][r] || !lists[s][r][0]) continue;
        std::string& txt = G.file_text[(size_t)r * 4 + s];
        if (!read_whole_file(lists[s][r], txt)) { bad[r] = s; return; }
        v[s][r] = TextView{txt.data(), txt.size()};
      }
    });
    for (int r = 0; r < n_regions; ++r)
      if (bad[r] >= 0) fail(BK_ERR_IO, "cannot read %s", lists[bad[r]][r]);
    IngestText t{};
    ingest_texts(G, n_regions, lists[0] ? v[0].data() : nullptr, lists[1] ? v[1].data() : nullptr,
                 lists[2] ? v[2].data() : nullptr, lists[3] ? v[3].data() : nullptr, in, &t);
    fill_text(t, text);
    G.file_text.clear();
  });
}

int bk_write_contigs(bk_ingest_t g, const bk_batch_result* res, const bk_batch_input* in, const bk_ingest_text* text,
                     const char* const* contigs_dir, const char* const* cluster_fn, int64_t* n_files) {
  return guarded_ingest(g, [&] {
    if (!res || !in || !text || !contigs_dir) fail(BK_ERR_ARG, "bk_write_contigs: bad arguments");
    if (in->k < 1 || in->k > 31) fail(BK_ERR_ARG, "bk_write_contigs: in->k must be the k of the batch");
    IngestText t{text->id_bytes, text->id_off, text->qual_bytes, text->qual_off, text->n_reads, text->read_flags};
    const int64_t n = write_contig_files(g->g, res, in, &t, contigs_dir, cluster_fn, in->k);
    if (n_files) *n_files = n;
  });
}

int bk_write_sample_kmers(bk_ingest_t g, const bk_batch_result* res, int32_t k, const char* const* paths, int64_t* n_files) {
  return guarded_ingest(g, [&] {
    if (!res || !paths || k < 1 || k > 31) fail(BK_ERR_ARG, "bk_write_sample_kmers: bad arguments");
    const int64_t n = write_sample_kmer_files(g->g, res, paths, k);
    if (n_files) *n_files = n;
  });
}

}  // extern "C"
