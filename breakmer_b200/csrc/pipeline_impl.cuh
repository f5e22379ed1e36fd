// Host orchestration of the batched whole-path pipeline (bk_batch_submit / bk_batch_wait, and the one-call forms
// bk_compare_kmers_batch, bk_batch_upload + bk_compare_kmers_resident, bk_compare_kmers_long).  Included into api.cu.
//
// Stage order on the handle's stream (every stage is a kernel in this directory):
//   1. group identical reads            prep.cuh   read_hash -> radix sort -> leaders -> scan -> scatter
//   2. k-mer stage                      kmers.cuh  emit (reads, soft clips) -> radix sort -> run_select (count + case & case_sc)
//                                                  -> candidate table -> probe (reference fwd + rc, normal) -> survivors
//   3. k-mer -> read inverted index     prep.cuh   index_emit -> two radix sorts -> post_off / post_split
//   4. work order                       prep.cuh   regions by descending cost class (one block)
//   5. assembly                         assemble.cuh  one CTA per region slot, dynamic region queue; in the long modes
//                                                     (LongMode) then route_long_kernel and assemble_long_kernel
//   6. results to pinned host memory
//
// The host never waits for the device between stages: every intermediate count (unique reads, candidates, sample-only
// k-mers, postings) stays in device memory, arrays are allocated for upper bounds known from the input offsets alone,
// and kernels whose extent is data dependent are launched over the bound and read the count themselves.  submit()
// therefore only enqueues (copies + ~60 launches) and returns; wait() blocks once for the counters, checks the output
// arena, copies the results and blocks a second time.  One host thread can keep several handles (streams) busy.
#pragma once
#include <chrono>

#include "pipeline.cuh"

namespace {

void upload_record_set(bk_handle_t h, Arena<false>& A, const char* bases, const int64_t* off, const int64_t* reg_off,
                       int n_regions, RecordSet& rs, int64_t& h2d, const char* what) {
  rs = RecordSet();
  if (!off || !reg_off) {
    if (bases) fail(BK_ERR_ARG, "batch: %s offsets missing", what);
    int64_t zero = 0;
    rs.off = to_device(h, A, &zero, 1);
    rs.koff = rs.off;
    return;
  }
  const int64_t n_rec = reg_off[n_regions];
  if (reg_off[0] != 0) fail(BK_ERR_ARG, "batch: %s region offsets must start at 0", what);
  if (off[0] != 0) fail(BK_ERR_ARG, "batch: %s record offsets must start at 0", what);
  std::vector<int32_t> seg(n_rec ? n_rec : 1), kseg;
  std::vector<int64_t> koff;
  koff.reserve(n_rec + 1);
  kseg.reserve(n_rec + 1);
  rs.reg_base.assign(n_regions + 1, 0);
  rs.reg_krec.assign(n_regions + 1, 0);
  for (int r = 0; r < n_regions; ++r) {
    if (reg_off[r + 1] < reg_off[r]) fail(BK_ERR_ARG, "batch: %s region offsets not monotone", what);
    rs.reg_base[r] = off[reg_off[r]];
    rs.reg_krec[r] = (int64_t)koff.size();
    for (int64_t i = reg_off[r]; i < reg_off[r + 1]; ++i) {
      seg[i] = r;
      if (off[i + 1] < off[i]) fail(BK_ERR_ARG, "batch: %s record offsets not monotone", what);
      if (off[i + 1] > off[i]) { koff.push_back(off[i]); kseg.push_back(r); }
    }
    rs.max_reg_bases = std::max(rs.max_reg_bases, off[reg_off[r + 1]] - off[reg_off[r]]);
  }
  const int64_t n_bases = off[n_rec];
  rs.reg_base[n_regions] = n_bases;
  rs.reg_krec[n_regions] = (int64_t)koff.size();
  koff.push_back(n_bases);
  if (n_bases > 0 && !bases) fail(BK_ERR_ARG, "batch: %s bases missing", what);
  rs.n_bases = n_bases;
  rs.n_rec = n_rec;
  rs.bases = (const uint8_t*)to_device(h, A, bases, (size_t)n_bases);
  rs.off = to_device(h, A, off, (size_t)n_rec + 1);
  rs.seg = to_device(h, A, seg.data(), (size_t)n_rec);
  rs.kn_rec = (int64_t)koff.size() - 1;
  rs.koff = to_device(h, A, koff.data(), koff.size());
  rs.kseg = to_device(h, A, kseg.data(), kseg.size());
  rs.d_reg_base = to_device(h, A, rs.reg_base.data(), rs.reg_base.size());
  rs.d_reg_krec = to_device(h, A, rs.reg_krec.data(), rs.reg_krec.size());
  h2d += n_bases + (n_rec + 1) * 8;
}

// Regions with a read above NW_MAX_LEN (ASM_LONG_MAX_LEN in the long modes) are left out; LONG_ROUTE marks those with a
// read above NW_MAX_LEN for assemble_long_kernel.
void pipeline_upload_into(bk_handle_t h, Arena<false>& A, const bk_batch_input* in, Pipeline& p, LongMode mode) {
  p = Pipeline();
  p.long_mode = mode;
  p.keep_rejected = h->rejected_contigs != 0;
  p.keep_normal = h->normal_kmers != 0;
  const int max_len = mode == LONG_OFF ? NW_MAX_LEN : ASM_LONG_MAX_LEN;
  if (in->n_regions < 0 || in->n_regions > 65535) fail(BK_ERR_ARG, "batch: n_regions must be in 0..65535 per call");
  if (in->k < 2 || in->k > 31) fail(BK_ERR_ARG, "batch: k must be in 2..31");
  const int R = in->n_regions;
  p.n_regions = R; p.k = in->k; p.rc_thresh = in->rc_thresh; p.have_mers = in->have_mers;
  p.n_short = mode == LONG_ALL ? 0 : R;
  if (!in->read_off || !in->read_reg_off) fail(BK_ERR_ARG, "batch: read arrays missing");
  // per-region read statistics; a region holding a read the assembler cannot take is left out of the device pass (its
  // region_status becomes BK_ERR_CAPACITY) instead of failing the call: the other regions are unaffected
  std::vector<int32_t> rl(R ? R : 1, 0);
  std::vector<uint8_t> routed;
  int mx = 0, mx_short = 0;
  int64_t n_skipped = 0;
  for (int r = 0; r < R; ++r) {
    if (in->read_reg_off[r + 1] < in->read_reg_off[r]) fail(BK_ERR_ARG, "batch: read region offsets not monotone");
    int m = 0;
    for (int64_t i = in->read_reg_off[r]; i < in->read_reg_off[r + 1]; ++i)
      m = std::max<int>(m, (int)std::min<int64_t>(in->read_off[i + 1] - in->read_off[i], int64_t(1) << 30));
    rl[r] = in->read_len ? in->read_len[r] : m;                    // utils.py:236
    if (m > max_len) {
      if (p.region_skipped.empty()) p.region_skipped.assign(R, 0);
      p.region_skipped[r] = 1;
      ++n_skipped;
    } else {
      mx = std::max(mx, m);
      if (m <= NW_MAX_LEN) {
        mx_short = std::max(mx_short, m);
      } else if (mode == LONG_ROUTE) {
        if (routed.empty()) routed.assign(R, 0);
        routed[r] = 1;
        --p.n_short;
      }
      p.max_reg_records = std::max(p.max_reg_records, in->read_reg_off[r + 1] - in->read_reg_off[r]);
    }
  }
  p.max_read_len = mx;
  p.max_short_read_len = mx_short;
  if (!routed.empty()) p.d_routed = to_device(h, A, routed.data(), (size_t)R);
  const char* read_bases = in->read_bases;
  const int64_t* read_off = in->read_off;
  const int64_t* read_reg_off = in->read_reg_off;
  const uint8_t* read_flags = in->read_flags;
  if (n_skipped) {
    // rare path: host copies of the read arrays without the records of the skipped regions
    p.rec_shift.assign(R + 1, 0);
    p.filt_reg_off.assign(R + 1, 0);
    p.filt_off.assign(1, 0);
    for (int r = 0; r < R; ++r) {
      const int64_t a = in->read_reg_off[r], b = in->read_reg_off[r + 1];
      p.rec_shift[r] = a - p.filt_reg_off[r];
      if (!p.region_skipped[r]) {
        const int64_t b0 = in->read_off[a], b1 = in->read_off[b];
        const int64_t at = (int64_t)p.filt_bases.size();
        p.filt_bases.insert(p.filt_bases.end(), in->read_bases + b0, in->read_bases + b1);
        for (int64_t i = a; i < b; ++i) p.filt_off.push_back(at + in->read_off[i + 1] - b0);
        if (in->read_flags) p.filt_flags.insert(p.filt_flags.end(), in->read_flags + a, in->read_flags + b);
      }
      p.filt_reg_off[r + 1] = (int64_t)p.filt_off.size() - 1;
    }
    read_bases = p.filt_bases.data(); read_off = p.filt_off.data(); read_reg_off = p.filt_reg_off.data();
    read_flags = in->read_flags ? p.filt_flags.data() : nullptr;
  }
  upload_record_set(h, A, read_bases, read_off, read_reg_off, R, p.reads, p.h2d_bytes, "read");
  p.read_reg_off = to_device(h, A, read_reg_off, (size_t)R + 1);
  p.total_read_bytes = p.reads.n_bases;
  p.read_len = to_device(h, A, rl.data(), (size_t)(R ? R : 1));
  if (read_flags) p.read_flags = to_device(h, A, read_flags, (size_t)p.reads.n_rec);
  p.h2d_bytes += p.reads.n_rec;
  if (in->have_mers) {
    if (!in->in_mers_off) fail(BK_ERR_ARG, "batch: in_mers_off missing");
    p.n_in_mers = in->in_mers_off[R];
    for (int r = 0; r < R; ++r) {
      if (in->in_mers_off[r + 1] < in->in_mers_off[r]) fail(BK_ERR_ARG, "batch: in_mers_off not monotone");
      p.max_reg_mers = std::max(p.max_reg_mers, in->in_mers_off[r + 1] - in->in_mers_off[r]);
    }
    p.in_mers = to_device(h, A, in->in_mers, (size_t)p.n_in_mers);
    p.in_counts = to_device(h, A, in->in_counts, (size_t)p.n_in_mers);
    p.in_mers_off = to_device(h, A, in->in_mers_off, (size_t)R + 1);
    p.h2d_bytes += p.n_in_mers * 12;
  } else {
    if (in->ref_off) {
      std::vector<int64_t> ident(R + 1);
      std::iota(ident.begin(), ident.end(), 0);
      upload_record_set(h, A, in->ref_bases, in->ref_off, ident.data(), R, p.ref, p.h2d_bytes, "ref");
    } else {
      // no reference sequence in this batch: the handle's reference k-mer cache stands in for it
      if (!h->ref_cache_mers) fail(BK_ERR_ARG, "batch: ref arrays missing and no reference k-mer cache on the handle");
      if (h->ref_cache_regions != R || h->ref_cache_k != in->k)
        fail(BK_ERR_ARG, "batch: the reference k-mer cache was built for %d regions, k=%d", h->ref_cache_regions, h->ref_cache_k);
      p.use_ref_cache = true;
    }
    upload_record_set(h, A, in->sc_bases, in->sc_off, in->sc_reg_off, R, p.sc, p.h2d_bytes, "soft-clip");
    upload_record_set(h, A, in->normal_bases, in->normal_off, in->normal_reg_off, R, p.normal, p.h2d_bytes, "normal");
    p.max_reg_mers = p.sc.max_reg_bases;        // every sample-only mer of a region is a soft-clip window of it
    // k-mer stage tables: a power of two of slots > the region's soft-clip windows (its distinct k-mers can never fill
    // it), in shared memory when that is at most RK_SMEM_CAP_MAX slots, else a slice of the global table
    std::vector<uint32_t> cap(R ? R : 1, 1024);
    std::vector<int64_t> goff(R ? R : 1, -1);
    for (int r = 0; r < R; ++r) {
      const int64_t n_sc = p.sc.reg_base.empty() ? 0 : p.sc.reg_base[r + 1] - p.sc.reg_base[r];
      uint64_t c = 1024;
      while (c <= (uint64_t)n_sc) c <<= 1;
      if (c > (uint64_t(1) << 31)) fail(BK_ERR_CAPACITY, "batch: a region has more than 2^31 soft-clip bases");
      cap[r] = (uint32_t)c;
      if (c <= (uint64_t)RK_SMEM_CAP_MAX) p.rk_smem_cap = std::max<int>(p.rk_smem_cap, (int)c);
      else { goff[r] = p.rk_gtab_slots; p.rk_gtab_slots += (int64_t)c; }
    }
    p.d_tab_cap = to_device(h, A, cap.data(), cap.size());
    p.d_gtab_off = to_device(h, A, goff.data(), goff.size());
  }
}

// the mode of the batched entries: the handle's "long_regions" option, read when their inputs are uploaded
LongMode option_mode(bk_handle_t h) { return h && h->long_regions ? LONG_ROUTE : LONG_OFF; }

void pipeline_upload(bk_handle_t h, const bk_batch_input* in) {
  h->resident.reset();
  h->pipe.reset(new Pipeline());
  pipeline_upload_into(h, h->resident, in, *h->pipe, option_mode(h));
  BK_CUDA(stream_wait(h));
}

template <typename T>
T* dev_zero(bk_handle_t h, size_t n) {
  T* p = h->dev.get<T>(n ? n : 1);
  BK_CUDA(cudaMemsetAsync(p, 0, (n ? n : 1) * sizeof(T), h->st));
  return p;
}

template <typename T>
T* to_host(bk_handle_t h, const T* d, size_t n) {
  T* p = h->pin.get<T>(n ? n : 1);
  if (n) BK_CUDA(cudaMemcpyAsync(p, d, n * sizeof(T), cudaMemcpyDeviceToHost, h->st));
  return p;
}

inline unsigned nblk(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

// k-mer windows of the records of regions [r0, r1) of one input set
void emit_set(bk_handle_t h, const RecordSet& rs, int r0, int r1, int k, int tag, bool rc, uint64_t* keys, uint32_t* vals,
              int64_t base, int64_t base_rc) {
  if (rs.reg_base.empty()) return;
  const int64_t b0 = rs.reg_base[r0], b1 = rs.reg_base[r1];
  if (b1 == b0) return;
  const int64_t kr0 = rs.reg_krec[r0], kr1 = rs.reg_krec[r1];
  EmitParams E{};
  E.bases = rs.bases + b0; E.n_bases = b1 - b0; E.rec_off = rs.koff + kr0; E.n_rec = kr1 - kr0; E.rec_seg = rs.kseg + kr0;
  E.rec_mult = nullptr; E.k = k; E.tag = tag; E.emit_rc = rc ? 1 : 0; E.off_shift = b0; E.seg_shift = r0;
  E.keys = keys; E.vals = vals; E.out_base = base; E.out_base_rc = base_rc;
  TimedLaunch t(h->timers, h->st, KF_EMIT);
  kmer_emit_kernel<<<nblk(E.n_bases, EMIT_TILE), EMIT_THREADS, 0, h->st>>>(E);
}

// Persistent reference k-mer cache: forward + reverse-complement k-mers of every target window, counted once,
// kept as sorted per-region mer arrays (the analogue of the marker-file cache of the reference dumps, utils.py:157).
void ref_cache_build(bk_handle_t h, const char* ref_bases, const int64_t* ref_off, int R, int k) {
  cudaStream_t st = h->st;
  h->dev.reset();
  h->pin.reset();
  h->cache.reset();
  h->ref_cache_mers = nullptr; h->ref_cache_koff = nullptr; h->ref_cache_regions = 0; h->ref_cache_k = 0;
  std::vector<int64_t> ident(R + 1);
  std::iota(ident.begin(), ident.end(), 0);
  RecordSet ref;
  int64_t h2d = 0;
  upload_record_set(h, h->dev, ref_bases, ref_off, ident.data(), R, ref, h2d, "ref");
  const int max_seg_bits = 63 - 2 * k;
  const int chunk = (int)std::min<int64_t>(R > 0 ? R : 1, int64_t(1) << std::min(max_seg_bits, 16));
  struct ChunkOut { SelectOut so; int64_t n; };
  std::vector<ChunkOut> outs;
  uint32_t* seg_counts_all = dev_zero<uint32_t>(h, (size_t)R + 1);
  int64_t total = 0;
  for (int r0 = 0; r0 < R; r0 += chunk) {
    const int r1 = std::min(R, r0 + chunk);
    const int64_t nr = ref.reg_base[r1] - ref.reg_base[r0];
    const int64_t nk = 2 * nr;
    if (nk >= (int64_t(1) << 31)) fail(BK_ERR_CAPACITY, "ref cache: more than 2^31 k-mer windows in one chunk");
    uint64_t* keys = h->dev.get<uint64_t>(nk);
    uint32_t* vals = h->dev.get<uint32_t>(nk);
    emit_set(h, ref, r0, r1, k, TAG_REF, true, keys, vals, 0, nr);
    SelectOut so = sort_and_select(h, keys, vals, nk, k, bits_for((uint64_t)(r1 - r0)), SELECT_ALL, r1 - r0, nk);
    BK_CUDA(cudaMemcpyAsync(seg_counts_all + r0, so.seg_counts, (size_t)(r1 - r0) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    const int64_t n = select_count(h, so);              // one-time build: a host round trip per chunk is fine here
    outs.push_back({so, n});
    total += n;
  }
  uint64_t* mers = h->cache.get<uint64_t>(total);
  int64_t* koff = h->cache.get<int64_t>(R + 1);
  int64_t at = 0;
  for (auto& c : outs) {
    if (c.n) BK_CUDA(cudaMemcpyAsync(mers + at, c.so.mers, c.n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    at += c.n;
  }
  uint32_t* seg_excl = h->dev.get<uint32_t>(R + 1);
  uint32_t* d_tot = h->dev.get<uint32_t>(1);
  uint32_t* stmp = h->dev.get<uint32_t>(scan_tmp_elems(R));
  exclusive_scan_u32(seg_counts_all, seg_excl, R, stmp, d_tot, st);
  widen_scan_kernel<<<nblk(R + 1, 256), 256, 0, st>>>(seg_excl, d_tot, R, koff);
  BK_CUDA(cudaGetLastError());
  BK_CUDA(stream_wait(h));
  h->ref_cache_mers = mers; h->ref_cache_koff = koff; h->ref_cache_regions = R; h->ref_cache_k = k;
}

// CTAs of assemble_long_kernel.  How many regions will overgrow in assemble_kernel is known only on the device, so the
// grid is the regions routed at upload plus this allowance, within the SM count and R (with LONG_ALL: min(R, SM count));
// the CTAs are persistent, so a small grid is only slower.
constexpr int LONG_ROUTE_SPARE_CTAS = 4;

// assemble_long_kernel's grid, queue and per-CTA scratch: contig-sized arrays for AsmCapLong (about 11 MB per CTA), the
// staged read for the longest read of the call.  The work counter lives in the zeroed block (pipeline_submit).
void long_assembly_scratch(bk_handle_t h, LongAssembly& S, const Pipeline& p) {
  using C = AsmCapLong;
  const int R = p.n_regions;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)(R - p.n_short) + LONG_ROUTE_SPARE_CTAS, (int64_t)h->sm_count, (int64_t)R}));
  S.grid = grid;
  S.read_cap = (int)((std::max<int64_t>(NW_MAX_LEN + 1, p.max_read_len + 2) + 15) / 16 * 16);
  S.w_cseq = h->dev.get<uint8_t>((size_t)grid * C::BUF);
  S.w_cnt = h->dev.get<int32_t>((size_t)grid * 4 * C::BUF);
  S.w_K = h->dev.get<int32_t>((size_t)grid * 4 * C::KCAP);
  S.w_NK = h->dev.get<int32_t>((size_t)grid * 4 * C::KCAP);
  S.w_wcode = h->dev.get<uint64_t>((size_t)grid * C::CAP);
  S.w_diff = h->dev.get<int32_t>((size_t)grid * (C::CAP + 1));
  S.w_edge = h->dev.get<int2>((size_t)grid * 2 * ASM_CAP);         // the warp DP's scratch (pairs within NW_MAX_LEN)
  S.w_lastcol = h->dev.get<uint2>((size_t)grid * ASM_LASTCOL);
  S.w_tab = h->dev.get<uint8_t>((size_t)grid * NW_TAB_BYTES);
  S.L.reads = h->dev.get<uint8_t>((size_t)grid * S.read_cap);
  S.L.contig = h->dev.get<uint8_t>((size_t)grid * C::CAP);
  S.L.diag = h->dev.get<int32_t>((size_t)grid * 9 * (C::CAP + 1));
  S.queue = h->dev.get<int32_t>(R ? R : 1);
}

// assemble_long_kernel's AsmParams: A with the long kernel's scratch, its queue as the work order and its own work
// counter; the inputs, the per-region state and the output arena are A's
AsmParams long_params(AsmParams A, const LongAssembly& S) {
  A.read_cap = S.read_cap;
  A.w_cseq = S.w_cseq; A.w_cnt = S.w_cnt; A.w_K = S.w_K; A.w_NK = S.w_NK; A.w_wcode = S.w_wcode; A.w_diff = S.w_diff;
  A.w_edge = S.w_edge; A.w_lastcol = S.w_lastcol; A.w_tab = S.w_tab;
  A.work_order = S.queue; A.work_counter = S.counter;
  return A;
}

// assemble_kernel<W> at the width, residency and shared memory chosen at submit
cudaError_t launch_assembly_batched(const PendingBatch& B, const AsmParams& A, cudaStream_t st) {
  // shared-memory carve-out: just enough for the resident CTAs, the rest of the 256 KB stays L1
  int carve = (int)((100 * (size_t)B.ctas_per_sm * ((size_t)B.dyn_smem + 1024) + 228 * 1024 - 1) / (228 * 1024));
  if (const char* e = getenv("BK_ASM_CARVEOUT")) carve = atoi(e);
  carve = std::min(100, std::max(0, carve));
  if (B.spec_w == 8) return launch_assemble_w8(A, B.grid, B.dyn_smem, carve, st);
  if (B.spec_w == 4 && B.ctas_per_sm >= 5) return launch_assemble_w4c5(A, B.grid, B.dyn_smem, carve, st);
  if (B.spec_w == 4 && B.ctas_per_sm == 4) return launch_assemble_w4c4(A, B.grid, B.dyn_smem, carve, st);
  if (B.spec_w == 4) return launch_assemble_w4(A, B.grid, B.dyn_smem, carve, st);
  if (B.spec_w == 2) return launch_assemble_w2(A, B.grid, B.dyn_smem, carve, st);
  return launch_assemble_w1(A, B.grid, B.dyn_smem, carve, st);
}

// (re)launch the assembler of a submitted batch: zero the mutable state, allocate the output arena for the current
// capacity, launch, and queue the copies of the counters wait() looks at first
void launch_assembly(bk_handle_t h, PendingBatch& B) {
  cudaStream_t st = h->st;
  AsmParams& A = B.A;
  const int R = A.n_regions;
  A.cap_seq = B.cap_seq; A.cap_cnt = B.cap_seq; A.cap_reads = B.cap_seq; A.cap_kmers = 2 * B.cap_seq;
  A.cap_ctg = std::max<unsigned long long>(1024, B.cap_seq / 64);
  A.o_seq = h->dev.get<uint8_t>(A.cap_seq); A.o_locs = h->dev.get<int32_t>(A.cap_seq);
  A.o_io = h->dev.get<int32_t>(A.cap_cnt); A.o_ot = h->dev.get<int32_t>(A.cap_cnt);
  A.o_reads = h->dev.get<int32_t>(A.cap_reads);
  A.o_kmer_mer = h->dev.get<uint64_t>(A.cap_kmers); A.o_kmer_pos = h->dev.get<int32_t>(A.cap_kmers);
  A.o_kmer_meta = h->dev.get<int32_t>(A.cap_kmers);
  A.o_desc = h->dev.get<int64_t>(A.cap_ctg * 10);
  BK_CUDA(cudaMemsetAsync(B.zero_lo, 0, B.zero_bytes, st));
  const int n_short = B.p->n_short;
  if (n_short > 0) {
    AsmParams S = A;                                       // assemble_kernel takes only the first n_short of the work order
    S.n_regions = n_short;
    TimedLaunch t(h->timers, st, KF_ASSEMBLE);
    BK_CUDA(launch_assembly_batched(B, S, st));
  }
  if (R > 0 && B.route) {
    {
      TimedLaunch t(h->timers, st, KF_PREP);
      route_long_kernel<<<1, ROUTE_THREADS, 0, st>>>(A.work_order, n_short, R, A.region_status, A.out_cursor, B.LA.queue, B.n_queue,
                                                     B.ctg_snapshot, A.region_report,
                                                     B.p->long_mode == LONG_ROUTE ? RR_READ_TOO_LONG : RR_OK);
    }
    TimedLaunch t(h->timers, st, KF_ASSEMBLE);
    BK_CUDA(launch_assemble_long(long_params(A, B.LA), B.LA.L, B.LA.grid, st));
  }
  BK_CUDA(cudaGetLastError());
  if (B.route) {
    B.h_queue = to_host(h, B.LA.queue, (size_t)R);
    B.h_n_queue = to_host(h, B.n_queue, 1);
    B.h_snapshot = to_host(h, B.ctg_snapshot, 1);
  }
  B.h_cursor = to_host(h, A.out_cursor, 5);
  B.h_stats = to_host(h, A.stats, 32);
  B.h_status = to_host(h, A.region_status, (size_t)(R ? R : 1));
  B.h_cells = to_host(h, A.region_cells, (size_t)(R ? R : 1));
}

// Enqueue the whole device pass of one batch.  in == nullptr: the batch uploaded with bk_batch_upload, in the mode it was
// uploaded with.  Otherwise mode: LONG_ALL for bk_compare_kmers_long (assemble_kernel gets no regions and is not
// launched), option_mode(h) for the batched entries.
void pipeline_submit(bk_handle_t h, const bk_batch_input* in, LongMode mode) {
  cudaStream_t st = h->st;
  if (h->pending.active) fail(BK_ERR_ARG, "a batch is already in flight on this handle (call bk_batch_wait first)");
  h->dev.reset();
  h->pin.reset();
  PendingBatch& B = h->pending;
  B = PendingBatch();
  BK_CUDA(cudaEventRecord(h->ev0, st));
  if (!in) {
    if (!h->pipe) fail(BK_ERR_ARG, "bk_compare_kmers_resident: no batch uploaded");
    B.p = h->pipe.get();
  } else {
    pipeline_upload_into(h, h->dev, in, B.local, mode);
    B.p = &B.local;
  }
  const Pipeline& p = *B.p;
  const int R = p.n_regions;
  const int k = p.k;
  if (p.reads.n_bases >= (int64_t(1) << 31) || p.n_in_mers >= (int64_t(1) << 31))
    fail(BK_ERR_CAPACITY, "batch: more than 2^31 read bases or k-mers in one call; use fewer regions per call");
  uint32_t* d_counts = dev_zero<uint32_t>(h, 4);   // [0] unique reads, [1] sample-only k-mers, [2] postings, [3] normal k-mers
  B.d_counts = d_counts;
  uint32_t* d_NU = d_counts, *d_S = d_counts + 1, *d_npost = d_counts + 2, *d_N = d_counts + 3;

  // field widths of the packed sort keys, from bounds the input offsets give (no device round trip)
  const int s_bits = std::max(1, bits_for((uint64_t)std::max<int64_t>(1, p.max_reg_mers)));
  const int u_bits = std::max(1, bits_for((uint64_t)std::max<int64_t>(1, p.max_reg_records)));
  if (s_bits > 24 || u_bits > 24) fail(BK_ERR_CAPACITY, "a region has more than 2^24 reads or soft-clip bases");

  // ---- 1. group identical reads -------------------------------------------------------
  const int64_t n_rec = p.reads.n_rec;                   // also the bound of the number of unique reads
  const int64_t NUB = n_rec;
  int32_t* u_rec = h->dev.get<int32_t>(NUB); uint32_t* u_mult = h->dev.get<uint32_t>(NUB);
  uint8_t* u_io = h->dev.get<uint8_t>(NUB); int32_t* u_len = h->dev.get<int32_t>(NUB);
  int64_t* u_off = h->dev.get<int64_t>(R + 1);
  if (n_rec > 0) {
    uint64_t* hk = h->dev.get<uint64_t>(n_rec);
    uint32_t* hv = h->dev.get<uint32_t>(n_rec);
    {
      TimedLaunch t(h->timers, st, KF_GROUP);
      read_hash_kernel<<<nblk(n_rec * 32, 128), 128, 0, st>>>(p.reads.bases, p.reads.off, p.reads.seg, n_rec, hk, hv);
    }
    const int64_t tiles = rs_num_tiles(n_rec);
    RadixSortScratch sc;
    sc.keys_alt = h->dev.get<uint64_t>(n_rec);
    sc.vals_alt = h->dev.get<uint32_t>(n_rec);
    sc.table = h->dev.get<uint32_t>(256 * tiles);
    sc.scan_tmp = h->dev.get<uint32_t>(scan_tmp_elems(256 * tiles));
    uint64_t* sk; uint32_t* sv;
    radix_sort_pairs(hk, hv, n_rec, 32, sc, st, &sk, &sv, h->timers, true);   // low 32 hash bits; runs are verified byte-wise
    int32_t* leader_of = h->dev.get<int32_t>(n_rec);
    uint32_t* mult_by_rec = dev_zero<uint32_t>(h, n_rec);
    uint32_t* flag = h->dev.get<uint32_t>(n_rec);
    uint32_t* u_index = h->dev.get<uint32_t>(n_rec);
    uint32_t* stmp = h->dev.get<uint32_t>(scan_tmp_elems(n_rec));
    {
      TimedLaunch t(h->timers, st, KF_GROUP, 2);
      group_leader_kernel<<<nblk(n_rec, 128), 128, 0, st>>>(sk, sv, n_rec, p.reads.bases, p.reads.off, p.reads.seg, leader_of,
                                                            mult_by_rec);
      leader_flag_kernel<<<nblk(n_rec, 256), 256, 0, st>>>(leader_of, n_rec, flag);
    }
    {
      TimedLaunch t(h->timers, st, KF_SCAN, 3);
      exclusive_scan_u32(flag, u_index, n_rec, stmp, d_NU, st);
    }
    {
      TimedLaunch t(h->timers, st, KF_GROUP, 2);
      unique_scatter_kernel<<<nblk(n_rec, 256), 256, 0, st>>>(leader_of, u_index, n_rec, mult_by_rec, p.read_flags, p.reads.off, u_rec,
                                                              u_mult, u_io, u_len);
      region_uoff_kernel<<<nblk(R + 1, 256), 256, 0, st>>>(p.read_reg_off, R, u_index, n_rec, d_NU, u_off);
    }
  } else {
    BK_CUDA(cudaMemsetAsync(u_off, 0, (R + 1) * sizeof(int64_t), st));
  }

  // ---- 2. k-mer stage ---------------------------------------------------------------------
  // SB = upper bound of the number of sample-only k-mers of the batch
  const int64_t SB = p.have_mers ? p.n_in_mers : std::min(p.sc.n_bases, p.reads.n_bases);
  const uint64_t* so_mer = nullptr; const uint32_t* so_cnt = nullptr;
  int64_t* so_off = h->dev.get<int64_t>(R + 1);
  if (p.have_mers) {
    so_mer = p.in_mers; so_cnt = p.in_counts;
    BK_CUDA(cudaMemcpyAsync(so_off, p.in_mers_off, (R + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    set_u32_kernel<<<1, 1, 0, st>>>(d_S, (uint32_t)p.n_in_mers);
  } else {
    const int64_t n_keys = 2 * p.ref.n_bases + p.reads.n_bases + p.sc.n_bases + p.normal.n_bases;
    B.n_keys = n_keys;
    uint64_t* all_m = h->dev.get<uint64_t>(SB ? SB : 1);
    uint32_t* all_c = h->dev.get<uint32_t>(SB ? SB : 1);
    uint32_t* seg_counts = dev_zero<uint32_t>(h, (size_t)R + 1);
    B.kmer_stage = true;
    B.keep_normal = p.keep_normal;
    int64_t* nm_off = p.keep_normal ? h->dev.get<int64_t>(R + 1) : nullptr;
    if (R > 0 && p.sc.n_bases > 0) {
      // one CTA per region: shared-memory hash table of its soft-clip k-mers, reads counted into it, reference and
      // normal windows streamed past it (region_kmers.cuh).  It runs without reads too: the report counts the candidates.
      RegionKmerParams K{};
      K.n_regions = R; K.k = k;
      auto view = [](const RecordSet& rs) { return RkSet{rs.n_bases > 0 ? rs.bases : nullptr, rs.koff, rs.d_reg_base, rs.d_reg_krec}; };
      K.sc = view(p.sc); K.reads = view(p.reads); K.normal = view(p.normal);
      if (p.use_ref_cache) { K.ref_mers = h->ref_cache_mers; K.ref_koff = h->ref_cache_koff; }
      else K.ref = view(p.ref);
      K.smem_cap = p.rk_smem_cap; K.tab_cap = p.d_tab_cap; K.gtab_off = p.d_gtab_off;
      K.gkeys = h->dev.get<uint64_t>(p.rk_gtab_slots ? p.rk_gtab_slots : 1);
      K.gcnt = h->dev.get<uint32_t>(p.rk_gtab_slots ? p.rk_gtab_slots : 1);
      K.st_mer = h->dev.get<uint64_t>(p.sc.n_bases); K.st_cnt = h->dev.get<uint32_t>(p.sc.n_bases);
      K.seg_counts = seg_counts;
      K.kmer_report = h->dev.get<int32_t>((size_t)R * KR_FIELDS);
      B.kmer_report = K.kmer_report;
      if (p.keep_normal) {                                 // a second staging slice, sorted and compacted the same way
        K.nm_mer = h->dev.get<uint64_t>(p.sc.n_bases); K.nm_cnt = h->dev.get<uint32_t>(p.sc.n_bases);
        K.nm_counts = h->dev.get<uint32_t>((size_t)R + 1);
      }
      const size_t smem = (size_t)K.smem_cap * 12 + RK_TILE + 64;
      const int per_sm = std::max<int>(1, (int)((220 * 1024) / (smem + 1024)));
      const int grid_k = (int)std::min<int64_t>(R, (int64_t)h->sm_count * std::min(per_sm, 4) * 2);
      {
        TimedLaunch t(h->timers, st, KF_REGION_KMERS);
        std::lock_guard<std::mutex> hold(launch_attr_mutex());     // (the limit is per kernel, the size per batch)
        BK_CUDA(cudaFuncSetAttribute(region_kmer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        region_kmer_kernel<<<grid_k, RK_THREADS, smem, st>>>(K);
        BK_CUDA(cudaGetLastError());
      }
      // the per-region counts -> offsets, and the staged k-mers -> dense arrays at those offsets
      auto compact = [&](const uint32_t* counts, uint32_t* d_total, int64_t* off, const uint64_t* st_m, const uint32_t* st_c,
                         uint64_t* m, uint32_t* c) {
        if (SB == 0) {                                     // no reads in the batch: no region has any
          BK_CUDA(cudaMemsetAsync(off, 0, (R + 1) * sizeof(int64_t), st));
          return;
        }
        uint32_t* excl = h->dev.get<uint32_t>(R + 1);
        uint32_t* stmp = h->dev.get<uint32_t>(scan_tmp_elems(R));
        {
          TimedLaunch t(h->timers, st, KF_SCAN, 4);
          exclusive_scan_u32(counts, excl, R, stmp, d_total, st);
          widen_scan_kernel<<<nblk(R + 1, 256), 256, 0, st>>>(excl, d_total, R, off);
        }
        {
          TimedLaunch t(h->timers, st, KF_REGION_KMERS);
          region_compact_kernel<<<(unsigned)std::min<int64_t>(R, (int64_t)h->sm_count * 16), 256, 0, st>>>(st_m, st_c, p.sc.d_reg_base, off, R,
                                                                                                         m, c);
        }
        BK_CUDA(cudaGetLastError());
      };
      compact(seg_counts, d_S, so_off, K.st_mer, K.st_cnt, all_m, all_c);
      if (p.keep_normal) {
        uint64_t* nm_m = h->dev.get<uint64_t>(SB ? SB : 1);   // (every one is a k-mer of the reads, as a sample-only one is)
        uint32_t* nm_c = h->dev.get<uint32_t>(SB ? SB : 1);
        compact(K.nm_counts, d_N, nm_off, K.nm_mer, K.nm_cnt, nm_m, nm_c);
        B.nm_mer = nm_m; B.nm_cnt = nm_c;
      }
    } else {
      BK_CUDA(cudaMemsetAsync(so_off, 0, (R + 1) * sizeof(int64_t), st));
      if (p.keep_normal) BK_CUDA(cudaMemsetAsync(nm_off, 0, (R + 1) * sizeof(int64_t), st));
    }
    B.nm_off = nm_off;
    so_mer = all_m; so_cnt = all_c;
  }

  // ---- 3. inverted index ------------------------------------------------------------------------------
  int64_t* post_off = h->dev.get<int64_t>(SB + 1);
  int64_t* rk_off = h->dev.get<int64_t>(NUB + 1);
  const int64_t cap = std::max<int64_t>(1, p.reads.n_bases);      // at most one posting per window
  int32_t* post_read = h->dev.get<int32_t>(cap); int32_t* post_pos = h->dev.get<int32_t>(cap);
  int32_t* rk_s = h->dev.get<int32_t>(cap); int32_t* rk_pos = h->dev.get<int32_t>(cap);
  if (SB > 0 && NUB > 0) {
    uint64_t* ik = h->dev.get<uint64_t>(cap);
    uint32_t* iv = h->dev.get<uint32_t>(cap);
    uint64_t* ik2 = h->dev.get<uint64_t>(cap);
    uint32_t* iv2 = h->dev.get<uint32_t>(cap);
    {
      TimedLaunch t(h->timers, st, KF_INDEX);
      const int ws_stride = ((p.max_read_len + 31) / 32) * 32 + 32;
      // window table of a warp's read: shared memory up to NW_MAX_LEN bases; longer reads (bk_compare_kmers_long) use a
      // global table, one window per read base at the read's own offset
      int32_t* ws_global = p.max_read_len > NW_MAX_LEN ? h->dev.get<int32_t>((size_t)cap) : nullptr;
      const size_t idx_smem = ws_global ? 0 : (size_t)IDX_WARPS * ws_stride * sizeof(int32_t);
      std::lock_guard<std::mutex> hold(launch_attr_mutex());
      if (idx_smem > 48 * 1024) BK_CUDA(cudaFuncSetAttribute(index_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)idx_smem));
      index_emit_kernel<<<nblk(NUB, IDX_WARPS), 32 * IDX_WARPS, idx_smem, st>>>(p.reads.bases, p.reads.off, u_off, u_rec, R, d_NU, so_off,
                                                                                so_mer, k, ik, iv, ik2, iv2, u_bits, s_bits, ws_stride,
                                                                                ws_global, d_npost, (uint32_t)std::min<int64_t>(cap, 0xFFFFFFFFll));
    }
    const int64_t tiles = rs_num_tiles(cap);
    RadixSortScratch sc;
    sc.keys_alt = h->dev.get<uint64_t>(cap);
    sc.vals_alt = h->dev.get<uint32_t>(cap);
    sc.table = h->dev.get<uint32_t>(256 * tiles);
    sc.scan_tmp = h->dev.get<uint32_t>(scan_tmp_elems(256 * tiles));
    uint64_t* sk; uint32_t* sv; uint64_t* sk2; uint32_t* sv2;
    radix_sort_pairs(ik, iv, cap, u_bits + bits_for((uint64_t)SB + 1), sc, st, &sk, &sv, h->timers, true, d_npost);
    RadixSortScratch sc2 = sc;
    sc2.keys_alt = h->dev.get<uint64_t>(cap);
    sc2.vals_alt = h->dev.get<uint32_t>(cap);
    radix_sort_pairs(ik2, iv2, cap, s_bits + bits_for((uint64_t)NUB + 1), sc2, st, &sk2, &sv2, h->timers, true, d_npost);
    TimedLaunch t(h->timers, st, KF_INDEX, 4);
    post_off_kernel<<<nblk(SB + 1, 256), 256, 0, st>>>(sk, d_npost, d_S, u_bits, post_off);
    post_off_kernel<<<nblk(NUB + 1, 256), 256, 0, st>>>(sk2, d_npost, d_NU, s_bits, rk_off);
    post_split_kernel<<<nblk(cap, 256), 256, 0, st>>>(sk, sv, d_npost, u_bits, post_read, post_pos);
    post_split_kernel<<<nblk(cap, 256), 256, 0, st>>>(sk2, sv2, d_npost, s_bits, rk_s, rk_pos);
  } else {
    BK_CUDA(cudaMemsetAsync(post_off, 0, (SB + 1) * sizeof(int64_t), st));
    BK_CUDA(cudaMemsetAsync(rk_off, 0, (NUB + 1) * sizeof(int64_t), st));
  }

  // ---- 4. work order: most expensive regions first (longest processing time) -----------------------------------
  int32_t* order = h->dev.get<int32_t>(R ? R : 1);
  if (R > 0) {
    TimedLaunch t(h->timers, st, KF_PREP);
    work_order_kernel<<<1, 1024, 0, st>>>(so_off, u_off, R, p.d_routed, order);
  }

  // ---- 5. assembly ----------------------------------------------------------------------------------------
  AsmParams& A = B.A;
  memset(&A, 0, sizeof A);
  A.n_regions = R; A.k = k; A.rc_thresh = p.rc_thresh; A.keep_rejected = p.keep_rejected ? 1 : 0;
  A.rbases = p.reads.bases; A.roff = p.reads.off;
  A.u_off = u_off; A.u_rec = u_rec; A.u_mult = u_mult; A.u_io = u_io; A.u_len = u_len; A.read_len = p.read_len;
  A.rk_off = rk_off; A.rk_s = rk_s; A.rk_pos = rk_pos;
  A.so_off = so_off; A.so_mer = so_mer; A.so_cnt = so_cnt;
  A.post_off = post_off; A.post_read = post_read; A.post_pos = post_pos;
  A.work_order = order;
  if (p.n_short > 0) {
    // speculation width and residency of the assembler (see assemble_kernel).  Auto = 4: one aligning warp per SM
    // sub-partition; 8 warps share the four ALU pipes of the SM and finish a round no sooner (measured on C4).
    int spec_w = h->spec_width;
    if (const char* e = getenv("BK_SPEC_W")) spec_w = atoi(e);
    if (spec_w <= 0) spec_w = 4;
    spec_w = spec_w >= 8 ? 8 : (spec_w >= 4 ? 4 : (spec_w >= 2 ? 2 : 1));
    int ctas_per_sm = spec_w == 8 ? 1 : (spec_w == 4 ? 3 : (spec_w == 2 ? 6 : 8));
    if (const char* e = getenv("BK_ASM_CTAS_PER_SM")) ctas_per_sm = std::max(1, atoi(e));
    const int grid = (int)std::min<int64_t>(p.n_short, (int64_t)h->sm_count * ctas_per_sm);
    // dynamic shared memory: exactly what the kernel needs (padding it to bound residency starves L1: 15 % slower)
    A.read_cap = (int)std::min<int64_t>(ASM_CAP, std::max<int64_t>(64, (p.max_short_read_len + 2 + 15) / 16 * 16));
    B.spec_w = spec_w; B.ctas_per_sm = ctas_per_sm; B.grid = grid;
    B.dyn_smem = (int)assemble_smem_bytes(spec_w, A.read_cap);
    if (getenv("BK_ASM_PAD")) B.dyn_smem = std::max(B.dyn_smem, (int)((227 * 1024) / ctas_per_sm) - 1024);
    A.w_cseq = h->dev.get<uint8_t>((size_t)grid * ASM_BUF);
    A.w_cnt = h->dev.get<int32_t>((size_t)grid * 4 * ASM_BUF);
    A.w_K = h->dev.get<int32_t>((size_t)grid * 4 * ASM_KCAP);
    A.w_NK = h->dev.get<int32_t>((size_t)grid * 4 * ASM_KCAP);
    A.w_wcode = h->dev.get<uint64_t>((size_t)grid * ASM_CAP);
    A.w_diff = h->dev.get<int32_t>((size_t)grid * (ASM_CAP + 1));
    A.w_edge = p.max_short_read_len > 256 ? h->dev.get<int2>((size_t)grid * spec_w * 2 * ASM_CAP) : nullptr;
    A.w_lastcol = h->dev.get<uint2>((size_t)grid * spec_w * ASM_LASTCOL);
    A.w_tab = getenv("BK_NW_PACKED") ? nullptr : h->dev.get<uint8_t>((size_t)grid * spec_w * NW_TAB_BYTES);   // (env: the packed-cell DP everywhere, for A/B runs)
  }
  B.route = p.long_mode != LONG_OFF;
  if (B.route) long_assembly_scratch(h, B.LA, p);
  A.region_status = h->dev.get<int32_t>(R ? R : 1);
  A.region_ncontigs = h->dev.get<int32_t>(R ? R : 1);
  A.region_cells = h->dev.get<unsigned long long>(R ? R : 1);
  A.m_alive = h->dev.get<uint8_t>(SB ? SB : 1);            // set by the kernel (bind_region)
  A.seed_a = h->dev.get<uint64_t>(SB ? SB : 1);            // seed order of each region, sorted by the kernel (bind_region)
  A.seed_b = h->dev.get<uint64_t>(SB ? SB : 1);
  A.l_mused = h->dev.get<int32_t>(SB ? SB : 1);
  // everything else starts zeroed (per attempt)
  size_t zero_bytes = 0;
  auto zalloc = [&](size_t bytes) { bytes = (bytes + 255) & ~size_t(255); size_t o = zero_bytes; zero_bytes += bytes; return o; };
  const size_t o_mused = zalloc(SB), o_checked = zalloc(SB * 4), o_taken = zalloc(SB * 4), o_first = zalloc(SB * 4);
  const size_t o_rused = zalloc(NUB), o_rdel = zalloc(NUB), o_rq = zalloc(NUB), o_rbuf = zalloc(NUB * 4), o_rin = zalloc(NUB * 4);
  const size_t o_work = zalloc(sizeof(int)), o_cursor = zalloc(5 * sizeof(unsigned long long)), o_stats = zalloc(32 * sizeof(unsigned long long));
  const size_t o_report = zalloc((size_t)R * RR_FIELDS * sizeof(int32_t));
  const size_t o_route = B.route ? zalloc(2 * sizeof(int) + sizeof(unsigned long long)) : 0;   // long counter, queue length, snapshot
  uint8_t* zero_lo = h->dev.get<uint8_t>(zero_bytes);
  if (B.route) {
    B.LA.counter = (int*)(zero_lo + o_route);
    B.n_queue = B.LA.counter + 1;
    B.ctg_snapshot = (unsigned long long*)(B.LA.counter + 2);
    B.LA.L.n_queue = B.n_queue;
  }
  B.zero_lo = zero_lo; B.zero_bytes = zero_bytes;
  A.m_used = zero_lo + o_mused; A.m_checked = (uint32_t*)(zero_lo + o_checked); A.m_taken = (uint32_t*)(zero_lo + o_taken); A.m_first = (uint32_t*)(zero_lo + o_first);
  A.r_used = zero_lo + o_rused; A.r_deleted = zero_lo + o_rdel; A.r_queued = zero_lo + o_rq;
  A.r_buf = (uint32_t*)(zero_lo + o_rbuf); A.r_inreads = (uint32_t*)(zero_lo + o_rin);
  A.work_counter = (int*)(zero_lo + o_work);
  A.out_cursor = (unsigned long long*)(zero_lo + o_cursor);
  A.stats = (unsigned long long*)(zero_lo + o_stats);
  A.region_report = (int32_t*)(zero_lo + o_report);
  A.q_read = h->dev.get<int32_t>(NUB ? NUB : 1); A.q_seed = h->dev.get<int32_t>(NUB ? NUB : 1);
  A.l_alt = h->dev.get<int32_t>(NUB ? NUB : 1); A.l_del = h->dev.get<int32_t>(NUB ? NUB : 1);
  A.hit_u = h->dev.get<int32_t>(NUB ? NUB : 1); A.hit_pos = h->dev.get<int32_t>(NUB ? NUB : 1);
  A.hit2_u = h->dev.get<int32_t>(NUB ? NUB : 1); A.hit2_pos = h->dev.get<int32_t>(NUB ? NUB : 1);
  A.sort_a = h->dev.get<uint64_t>(NUB ? NUB : 1); A.sort_b = h->dev.get<uint64_t>(NUB ? NUB : 1);
  A.prof_regions = getenv("BK_PHASE_PRINT") ? dev_zero<unsigned long long>(h, (size_t)R * 12 + 12) : nullptr;
  B.cap_seq = (unsigned long long)std::max<int64_t>(1 << 20, 8 * p.total_read_bytes);
  B.so_mer = so_mer; B.so_cnt = so_cnt; B.so_off = so_off; B.u_off = u_off; B.u_rec = u_rec; B.u_mult = u_mult;
  launch_assembly(h, B);
  B.h_counts = to_host(h, d_counts, 4);
  B.h_so_off = to_host(h, so_off, (size_t)R + 1);
  B.h_u_off = to_host(h, u_off, (size_t)R + 1);
  B.active = true;
}

void phase_print(bk_handle_t h, const PendingBatch& B);

// Block until the submitted batch is done and hand out its results.
void pipeline_wait(bk_handle_t h, bk_batch_result* out) {
  cudaStream_t st = h->st;
  PendingBatch& B = h->pending;
  if (!B.active) fail(BK_ERR_ARG, "bk_batch_wait: no batch in flight on this handle");
  B.active = false;                                        // whatever happens below, the handle is free again
  memset(out, 0, sizeof *out);
  const Pipeline& p = *B.p;
  const AsmParams& A = B.A;
  const int R = p.n_regions;
  out->n_regions = R;
  out->n_kmer_occurrences = B.n_keys;
  out->n_sorted_keys = B.n_sorted;
  const auto t_enter = std::chrono::steady_clock::now();
  double blocked_ms = 0;
  auto timed_wait = [&] {
    const auto a = std::chrono::steady_clock::now();
    const cudaError_t e = stream_wait(h);
    blocked_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
    return e;
  };
  for (int attempt = 0;; ++attempt) {
    BK_CUDA(timed_wait());                                 // first wait: counters of the whole pass
    const bool overflow = B.h_cursor[0] > A.cap_seq || B.h_cursor[1] > A.cap_cnt || B.h_cursor[2] > A.cap_reads ||
                          B.h_cursor[3] > A.cap_kmers || B.h_cursor[4] > A.cap_ctg;
    if (!overflow) break;
    if (attempt >= 3) fail(BK_ERR_CAPACITY, "assembly output arena overflow");
    B.cap_seq *= 8;                                        // rare: rerun the assembly with a larger arena
    launch_assembly(h, B);
  }
  const int64_t NU = B.h_counts[0], S_total = B.h_counts[1];
  const unsigned long long* h_cursor = B.h_cursor;
  const int64_t n_desc = (int64_t)h_cursor[4];
  out->n_check_align = (int64_t)B.h_stats[0];
  out->n_dp_cells = (int64_t)B.h_stats[1];
  if (getenv("BK_PHASE_PRINT")) phase_print(h, B);
  out->so_off = B.h_so_off;
  out->so_mers = to_host(h, B.so_mer, (size_t)S_total);
  out->so_counts = to_host(h, B.so_cnt, (size_t)S_total);
  out->uniq_reg_off = B.h_u_off;
  int32_t* h_urec = to_host(h, B.u_rec, (size_t)NU);
  out->uniq_rec = h_urec;
  out->uniq_mult = to_host(h, B.u_mult, (size_t)NU);
  out->region_status = B.h_status;
  out->region_dp_cells = (const int64_t*)B.h_cells;
  const int64_t* h_desc = to_host(h, A.o_desc, (size_t)n_desc * 10);
  out->ctg_seq = (const char*)to_host(h, A.o_seq, (size_t)h_cursor[0]);
  out->ctg_kmer_locs = to_host(h, A.o_locs, (size_t)h_cursor[0]);
  out->ctg_indel_only = to_host(h, A.o_io, (size_t)h_cursor[1]);
  out->ctg_others = to_host(h, A.o_ot, (size_t)h_cursor[1]);
  int32_t* h_reads = to_host(h, A.o_reads, (size_t)h_cursor[2]);
  out->ctg_reads = h_reads;
  out->ctg_kmer_mer = to_host(h, A.o_kmer_mer, (size_t)h_cursor[3]);
  out->ctg_kmer_pos = to_host(h, A.o_kmer_pos, (size_t)h_cursor[3]);
  const int32_t* h_meta = to_host(h, A.o_kmer_meta, (size_t)h_cursor[3]);
  BK_CUDA(cudaEventRecord(h->ev1, st));
  BK_CUDA(timed_wait());                                   // second wait: the result arrays
  float ms = 0;
  BK_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  out->gpu_ms = ms;

  // contigs left the device in completion order; the tables below put them in (region, growth order) -- payload arrays
  // stay where they are.  The accepted contigs come first; rejected ones (keep_rejected) follow them, at n_contigs ..
  std::vector<int64_t> idx(n_desc);
  std::iota(idx.begin(), idx.end(), 0);
  if (B.route) {
    // a region assemble_long_kernel took over keeps only that kernel's contigs (descriptors from the snapshot on), and
    // none if it failed there too (LONG_ALL: the snapshot is 0); the dropped descriptors' payloads stay unreferenced
    std::vector<uint8_t> rerouted(R ? R : 1, 0);
    for (int i = 0; i < *B.h_n_queue; ++i) rerouted[B.h_queue[i]] = 1;
    const int64_t snap = (int64_t)*B.h_snapshot;
    idx.erase(std::remove_if(idx.begin(), idx.end(), [&](int64_t c) {
                const int64_t r = h_desc[c * 10];
                return rerouted[r] && (c < snap || B.h_status[r] != ST_OK);
              }), idx.end());
  }
  auto reason_of = [&](int64_t c) { return (int32_t)(h_desc[c * 10 + 1] >> 32); };
  if (p.keep_rejected)                                     // a region that stopped has no rejected contigs
    idx.erase(std::remove_if(idx.begin(), idx.end(), [&](int64_t c) {
                return reason_of(c) != REJ_NONE && B.h_status[h_desc[c * 10]] != ST_OK;
              }), idx.end());
  const auto first_rej = std::stable_partition(idx.begin(), idx.end(), [&](int64_t c) { return reason_of(c) == REJ_NONE; });
  const int64_t n_ctg = first_rej - idx.begin(), n_all = (int64_t)idx.size();
  out->n_contigs = n_ctg;
  auto growth_order = [&](int64_t a, int64_t b) {
    const int64_t* da = h_desc + a * 10; const int64_t* db = h_desc + b * 10;
    return da[0] != db[0] ? da[0] < db[0] : (uint32_t)da[1] < (uint32_t)db[1];
  };
  std::sort(idx.begin(), first_rej, growth_order);
  std::sort(first_rej, idx.end(), growth_order);
  int64_t* t_reg = h->pin.get<int64_t>(R + 1);
  int64_t* t_seq = h->pin.get<int64_t>(2 * n_all + 2);
  int64_t* t_cnt = h->pin.get<int64_t>(2 * n_all + 2);
  int64_t* t_rd = h->pin.get<int64_t>(2 * n_all + 2);
  int64_t* t_km = h->pin.get<int64_t>(2 * n_all + 2);
  for (int r = 0; r <= R; ++r) t_reg[r] = 0;
  B.keep_rejected = p.keep_rejected;
  B.rej_reg_off.assign(p.keep_rejected ? R + 1 : 0, 0);
  B.rej_reason.clear();
  for (int64_t c = 0; c < n_all; ++c) {
    const int64_t* d = h_desc + idx[c] * 10;
    if (c < n_ctg) {
      t_reg[d[0] + 1] += 1;
    } else {
      B.rej_reg_off[d[0] + 1] += 1;
      B.rej_reason.push_back(reason_of(idx[c]));
    }
    t_seq[2 * c] = d[2]; t_seq[2 * c + 1] = d[3];
    t_cnt[2 * c] = d[4]; t_cnt[2 * c + 1] = d[5];
    t_rd[2 * c] = d[6]; t_rd[2 * c + 1] = d[7];
    t_km[2 * c] = d[8]; t_km[2 * c + 1] = d[9];
  }
  for (int r = 0; r < R; ++r) t_reg[r + 1] += t_reg[r];
  for (int r = 0; r < (int)B.rej_reg_off.size() - 1; ++r) B.rej_reg_off[r + 1] += B.rej_reg_off[r];
  out->ctg_reg_off = t_reg;
  out->ctg_seq_off = t_seq; out->ctg_cnt_off = t_cnt; out->ctg_reads_off = t_rd; out->ctg_kmers_off = t_km;
  // split the packed tuple meta word into the three fields of the 5-tuple
  int32_t* lth = h->pin.get<int32_t>(h_cursor[3] + 1);
  int32_t* dist = h->pin.get<int32_t>(h_cursor[3] + 1);
  int32_t* ord = h->pin.get<int32_t>(h_cursor[3] + 1);
  for (unsigned long long e = 0; e < h_cursor[3]; ++e) {
    lth[e] = h_meta[e] & 1; ord[e] = (h_meta[e] >> 1) & 3; dist[e] = h_meta[e] >> 3;
  }
  out->ctg_kmer_lth = lth; out->ctg_kmer_dist = dist; out->ctg_kmer_order = ord;
  struct HostTimes {                                       // filled on every normal exit
    bk_batch_result* out; std::chrono::steady_clock::time_point t0; double* blocked;
    ~HostTimes() {
      const double total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      out->host_wait_ms = *blocked; out->host_post_ms = total - *blocked;
    }
  } host_times{out, t_enter, &blocked_ms};
  B.h_reason.assign(B.h_status, B.h_status + R);          // the device's status of a stopped region is the reason
  for (int r = 0; r < R; ++r)
    if (B.h_status[r] != ST_OK) B.h_status[r] = BK_ERR_CAPACITY;
  B.long_queue.assign(B.route ? B.h_queue : nullptr, B.route ? B.h_queue + *B.h_n_queue : nullptr);
  if (!p.region_skipped.empty()) {
    // regions that were left out: report them, and give record indices in the caller's numbering again
    for (int r = 0; r < R; ++r) {
      if (p.region_skipped[r]) { B.h_status[r] = BK_ERR_CAPACITY; B.h_cells[r] = 0; }
      const int32_t shift = (int32_t)p.rec_shift[r];
      if (!shift) continue;
      for (int64_t u = B.h_u_off[r]; u < B.h_u_off[r + 1]; ++u) h_urec[u] += shift;
      auto shift_reads = [&](int64_t c0, int64_t c1) {
        for (int64_t c = c0; c < c1; ++c)
          for (int64_t e = t_rd[2 * c]; e < t_rd[2 * c] + t_rd[2 * c + 1]; ++e) h_reads[e] += shift;
      };
      shift_reads(t_reg[r], t_reg[r + 1]);
      if (p.keep_rejected) shift_reads(n_ctg + B.rej_reg_off[r], n_ctg + B.rej_reg_off[r + 1]);
    }
  }
  B.report_skipped = p.region_skipped;                     // (the resident Pipeline may be replaced before the report is read)
  B.result_epoch = h->dev.resets();
  B.has_result = true;
}

// bk_region_report: the report of the last result.  The device's table holds the counters and RR_FIRST_REASON; the reason
// (the device's region_status) and the pass (the long kernel's queue) are added here, and regions left out at upload get
// their row here, as their region_status does in pipeline_wait
const int32_t* region_report(bk_handle_t h) {
  PendingBatch& B = h->pending;
  if (B.active) fail(BK_ERR_ARG, "bk_region_report: a batch is in flight on this handle (call bk_batch_wait first)");
  if (!B.has_result || B.result_epoch != h->dev.resets()) fail(BK_ERR_ARG, "bk_region_report: no result on this handle");
  const int R = B.A.n_regions;
  B.h_report.assign((size_t)(R ? R : 1) * RR_FIELDS, 0);
  if (R) {
    BK_CUDA(cudaMemcpyAsync(B.h_report.data(), B.A.region_report, (size_t)R * RR_FIELDS * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    BK_CUDA(stream_wait(h));
  }
  for (int r = 0; r < R; ++r) {
    int32_t* row = B.h_report.data() + (size_t)r * RR_FIELDS;
    row[RR_REASON] = B.h_reason[r];
    row[RR_PASS] = RR_PASS_BATCHED;
  }
  for (int32_t r : B.long_queue) B.h_report[(size_t)r * RR_FIELDS + RR_PASS] = RR_PASS_LONG;
  for (int r = 0; r < (int)B.report_skipped.size(); ++r) {
    if (!B.report_skipped[r]) continue;
    int32_t* row = B.h_report.data() + (size_t)r * RR_FIELDS;
    std::fill(row, row + RR_FIELDS, 0);
    row[RR_REASON] = RR_READ_TOO_LONG;
  }
  return B.h_report.data();
}

// bk_rejected_contigs: the rejected contigs of the last result, as pipeline_wait split them off
void rejected_contigs(bk_handle_t h, const int64_t** reg_off, const int32_t** reason, int64_t* n) {
  PendingBatch& B = h->pending;
  if (B.active) fail(BK_ERR_ARG, "bk_rejected_contigs: a batch is in flight on this handle (call bk_batch_wait first)");
  if (!B.has_result || B.result_epoch != h->dev.resets()) fail(BK_ERR_ARG, "bk_rejected_contigs: no result on this handle");
  if (!B.keep_rejected) fail(BK_ERR_ARG, "bk_rejected_contigs: the last result was made with the \"rejected_contigs\" option off");
  *reg_off = B.rej_reg_off.data();
  *reason = B.rej_reason.empty() ? nullptr : B.rej_reason.data();
  *n = (int64_t)B.rej_reason.size();
}

// the refusals bk_kmer_report and bk_normal_kmers share: a batch in flight, no result (or its memory reused), a result
// without a k-mer stage (have_mers)
void check_kmer_stage_result(bk_handle_t h, const char* what) {
  const PendingBatch& B = h->pending;
  if (B.active) fail(BK_ERR_ARG, "%s: a batch is in flight on this handle (call bk_batch_wait first)", what);
  if (!B.has_result || B.result_epoch != h->dev.resets()) fail(BK_ERR_ARG, "%s: no result on this handle", what);
  if (!B.kmer_stage) fail(BK_ERR_ARG, "%s: the last result was given its sample-only k-mers (have_mers): no k-mer stage ran", what);
}

// bk_kmer_report: the k-mer stage's report of the last result; regions left out at upload get an all-zero row
const int32_t* kmer_report(bk_handle_t h) {
  check_kmer_stage_result(h, "bk_kmer_report");
  PendingBatch& B = h->pending;
  const int R = B.A.n_regions;
  B.h_kmer_report.assign((size_t)(R ? R : 1) * KR_FIELDS, 0);
  if (R && B.kmer_report) {
    BK_CUDA(cudaMemcpyAsync(B.h_kmer_report.data(), B.kmer_report, (size_t)R * KR_FIELDS * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    BK_CUDA(stream_wait(h));
  }
  for (int r = 0; r < (int)B.report_skipped.size(); ++r)
    if (B.report_skipped[r]) std::fill_n(B.h_kmer_report.data() + (size_t)r * KR_FIELDS, KR_FIELDS, 0);
  return B.h_kmer_report.data();
}

// bk_normal_kmers: the k-mers the normal sample removed from the last result (the "normal_kmers" option)
void normal_kmers(bk_handle_t h, const int64_t** reg_off, const uint64_t** mers, const uint32_t** counts, int64_t* n) {
  check_kmer_stage_result(h, "bk_normal_kmers");
  PendingBatch& B = h->pending;
  if (!B.keep_normal) fail(BK_ERR_ARG, "bk_normal_kmers: the last result was made with the \"normal_kmers\" option off");
  const int R = B.A.n_regions;
  B.h_nm_off.assign((size_t)R + 1, 0);
  BK_CUDA(cudaMemcpyAsync(B.h_nm_off.data(), B.nm_off, ((size_t)R + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->st));
  BK_CUDA(stream_wait(h));
  const int64_t total = B.h_nm_off[R];
  B.h_nm_mer.assign((size_t)(total ? total : 1), 0);
  B.h_nm_cnt.assign((size_t)(total ? total : 1), 0);
  if (total) {
    BK_CUDA(cudaMemcpyAsync(B.h_nm_mer.data(), B.nm_mer, (size_t)total * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->st));
    BK_CUDA(cudaMemcpyAsync(B.h_nm_cnt.data(), B.nm_cnt, (size_t)total * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    BK_CUDA(stream_wait(h));
  }
  *reg_off = B.h_nm_off.data();
  *mers = B.h_nm_mer.data();
  *counts = B.h_nm_cnt.data();
  *n = total;
}

void phase_print(bk_handle_t h, const PendingBatch& B) {
  const AsmParams& A = B.A;
  const int R = A.n_regions;
  const unsigned long long* h_stats = B.h_stats;
  const int64_t* h_u_off = B.h_u_off; const int64_t* h_so_off = B.h_so_off;
  static const char* nm[] = {"nw", "find_reads", "kmers", "finalize", "emit", "predict", "total", "max_region",
                             "apply", "refresh", "seed", "valid", "dp", "stage", "init", "bind"};
  for (int i = 0; i < 16; ++i) fprintf(stderr, "phase %-10s %12llu cycles\n", nm[i], h_stats[8 + i]);
  fprintf(stderr, "find_reads calls %llu seeds %llu check_align %llu rounds %llu slots %llu\n", h_stats[2], h_stats[3], h_stats[0],
          h_stats[4], h_stats[5]);
  if (!A.prof_regions) return;
  std::vector<unsigned long long> pr((size_t)R * 12);
  BK_CUDA(cudaMemcpy(pr.data(), A.prof_regions, pr.size() * 8, cudaMemcpyDeviceToHost));
  std::vector<int> ids(R);
  std::iota(ids.begin(), ids.end(), 0);
  std::sort(ids.begin(), ids.end(), [&](int a, int b) { return pr[(size_t)a * 12 + 6] > pr[(size_t)b * 12 + 6]; });
  unsigned long long t0 = ~0ull, t1 = 0, sum = 0;
  for (int r = 0; r < R; ++r) {
    const unsigned long long a = pr[(size_t)r * 12 + 8], b = pr[(size_t)r * 12 + 9];
    if (a < t0) t0 = a;
    if (b > t1) t1 = b;
    sum += b - a;
  }
  fprintf(stderr, "TIMELINE handle %p regions_start_ns %llu end_ns %llu span_ms %.3f sum_region_ms %.3f avg_concurrency %.1f\n", (void*)h,
          t0, t1, (t1 - t0) / 1e6, sum / 1e6, (double)sum / (double)(t1 - t0 + 1));
  if (getenv("BK_REGION_DUMP")) {
    FILE* f = fopen(getenv("BK_REGION_DUMP"), "w");
    if (f) {
      for (int r = 0; r < R; ++r)
        fprintf(f, "%d %lld %lld %llu %llu %llu\n", r, (long long)(h_u_off[r + 1] - h_u_off[r]), (long long)(h_so_off[r + 1] - h_so_off[r]),
                pr[(size_t)r * 12 + 6], pr[(size_t)r * 12 + 0], pr[(size_t)r * 12 + 8] - t0);
      fclose(f);
    }
  }
  if (getenv("BK_TIMELINE_DUMP")) {
    FILE* f = fopen(getenv("BK_TIMELINE_DUMP"), "a");
    if (f) {
      for (int r = 0; r < R; ++r)
        fprintf(f, "%p %d %llu %llu %llu\n", (void*)h, r, pr[(size_t)r * 12 + 8], pr[(size_t)r * 12 + 9], pr[(size_t)r * 12 + 10]);
      fclose(f);
    }
  }
  for (int t = 0; t < 4 && t < R; ++t) {
    const unsigned long long* q = &pr[(size_t)ids[t] * 12];
    fprintf(stderr, "region %d (U=%lld S=%lld): total %llu nw %llu find %llu kmers %llu finalize %llu emit %llu predict %llu\n", ids[t],
            (long long)(h_u_off[ids[t] + 1] - h_u_off[ids[t]]), (long long)(h_so_off[ids[t] + 1] - h_so_off[ids[t]]), q[6], q[0], q[1],
            q[2], q[3], q[4], q[5]);
  }
}

}  // namespace
