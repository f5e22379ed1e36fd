// Per-region greedy k-mer assembler: the reference's `init_assembly` and all it
// drives (sv_assembly.py:11-63, 102-155, 160-267, 272-366, 379-411, 416-649),
// executed by ONE WARP PER TARGET REGION, many regions per launch.
//
// The algorithm is a sequential, stateful state machine (SURVEY.md section 3.3);
// the device version keeps the reference's order of events exactly and spends
// the warp's 32 lanes inside each step: the overlap DP (nw.cuh), scanning
// posting lists, enumerating contig k-mers, vector updates.  All control flow is
// warp-uniform; scalars are replicated in registers, shared state lives in
// global memory (L1/L2 resident, a few hundred KB per region) and is written by
// lane-strided loops or by lane 0, with __syncwarp() between producer and
// consumer phases.
//
// Line citations are into /root/reference/sv_assembly.py; Q-numbers refer to
// SURVEY.md section 8.1.  The CPU restatement of the same behaviour is
// oracle/assembler_py.py (pinned to the reference); tests compare the two.
//
// Order policy for the two hash-order dependent spots (SURVEY.md 8.4): reads are
// numbered in fq_recs insertion order and ties keep that order (Q9); the
// alt-read candidate set is walked in ascending mer order (Q13).
#pragma once
#include "common.cuh"
#include "nw.cuh"
#ifndef BK_SIM
#include "nw_sweep.cuh"
#endif

namespace bk {

constexpr int ASM_CAP = 4096;          // contig / count-vector capacity (NW_MAX_LEN + 1)
constexpr int ASM_BUF = 3 * ASM_CAP;   // gap buffers: data starts at ASM_CAP, may grow both ways
constexpr int ASM_KCAP = 2 * ASM_CAP;  // contig k-mer tuple list capacity
constexpr int ASM_LASTCOL = ASM_CAP / 2 + 1;   // row pairs of one sweep
constexpr int ORDER_FOR = 0, ORDER_REV = 1, ORDER_MID = 2;

// Capacity of the state machine, a template argument of everything below that touches a contig.  BITS is the width of
// a position in the packed keys: find_reads sorts [pos : BITS | CAP - 1 - len : BITS], m_first holds
// [contig serial : 32 - BITS | CAP - 1 - window : BITS].
//   AsmCap      assemble_kernel: reads and contigs up to 4,095 bases (the warp DP's limit, NW_MAX_LEN), contig and
//               staged reads in shared memory, 2^20 contigs per region
//   AsmCapLong  assemble_long_kernel: reads and contigs up to 65,535 bases, contig and staged read in global scratch,
//               2^16 contigs per region
struct AsmCap {
  static constexpr int BITS = 12;
  static constexpr int CAP = 1 << BITS;        // as ASM_CAP
  static constexpr int MAX_LEN = CAP - 1;       // longest read / contig
  static constexpr int BUF = 3 * CAP;           // as ASM_BUF
  static constexpr int KCAP = 2 * CAP;          // as ASM_KCAP
  static constexpr bool LONG = false;
  using Key = int;
};
struct AsmCapLong {
  static constexpr int BITS = 16;
  static constexpr int CAP = 1 << BITS;
  static constexpr int MAX_LEN = CAP - 1;
  static constexpr int BUF = 3 * CAP;
  static constexpr int KCAP = 2 * CAP;
  static constexpr bool LONG = true;
  using Key = unsigned;
};
constexpr int ASM_LONG_MAX_LEN = AsmCapLong::CAP - 1;                          // 65,535

// Speculation width: the next ASM_SPEC_W reads of a contig's read stream are aligned
// concurrently, one warp each (the CTA has up to ASM_SPEC_W warps per region; warp 0
// also runs the state machine).  Slot 0 aligns against the current contig; slot w > 0
// aligns against a PREDICTED contig -- the current one with the predicted effects of
// slots 0..w-1 applied (gapless overlap at the shared k-mer: prepend / append /
// replace / no change).  Results are committed in stream order, and a slot's result
// is used only if the actual contig at that moment is byte-identical to the contig
// the slot was aligned against; otherwise a new round starts there.  The outcome is
// therefore identical to checking the reads one by one (the prediction is a hint).
#ifndef ASM_W4_CTAS
#define ASM_W4_CTAS 3
#endif
#ifndef ASM_W1_CTAS
#define ASM_W1_CTAS 13
#endif
#ifndef ASM_SPEC_W
#define ASM_SPEC_W 8     // maximum width (array sizes); the width of a launch is a kernel template argument
#endif

struct SpecShared {               // command + results of one speculation round (shared memory)
  int n;                          // reads in this round, -1 = workers exit
  int region;
  int u[ASM_SPEC_W];              // local unique-read indices
  int lr[ASM_SPEC_W];             // their lengths
  int abuf[ASM_SPEC_W];           // which contig buffer slot w aligns against: 0 = the current contig,
                                  // b > 0 = predicted contig buffer b - 1
  int la[ASM_SPEC_W];             // length of that contig
  NwOut v1[ASM_SPEC_W];           // nw(contig, read)
  NwOut v2[ASM_SPEC_W];           // nw(read, contig)
};

// optional phase timing (-DBK_PHASE_PROF, experiments only): cycles per phase, summed over regions
enum { PH_NW = 0, PH_FIND, PH_KMERS, PH_FINALIZE, PH_EMIT, PH_PREDICT, PH_TOTAL, PH_MAXREGION,
       PH_APPLY, PH_REFRESH, PH_SEED, PH_VALID, PH_DP, PH_STAGE, PH_INIT, PH_BIND, PH_COUNT_ };
#if defined(BK_PHASE_PROF) && !defined(BK_SIM)
#define BK_PH_BEGIN long long _ph_t0 = clock64();
#define BK_PH_END(c, ph) (c).ph_cycles[ph] += clock64() - _ph_t0;
#else
#define BK_PH_BEGIN
#define BK_PH_END(c, ph)
#endif

// ---- batch-wide inputs / state (device pointers) -----------------------------
struct AsmParams {
  int n_regions;
  int k;
  int rc_thresh;
  int read_cap;                    // bytes of one staged-read buffer in shared memory: >= longest read + 2, multiple of 16
  // reads: raw records + unique-read table (fq_recs, utils.py:239-244, Q28)
  const uint8_t* rbases;
  const int64_t* roff;             // n_rec + 1
  const int64_t* u_off;            // n_regions + 1 : unique reads of a region
  const int32_t* u_rec;            // representative (first) record of each unique read
  const uint32_t* u_mult;          // len(fq_recs[seq])
  const uint8_t* u_io;             // reads[0].indel_only
  const int32_t* u_len;            // length of each unique read
  const int32_t* read_len;         // per region: max record length (utils.py:236)
  // sample-only k-mers (ascending per region) and derived tables
  const int64_t* so_off;           // n_regions + 1
  const uint64_t* so_mer;
  const uint32_t* so_cnt;
  const int64_t* post_off;         // total mers + 1 : k-mer -> read posting lists
  const int32_t* post_read;        // local unique-read index, ascending within a list
  const int32_t* post_pos;         // first position of the mer in that read
  const int64_t* rk_off;           // total unique reads + 1 : read -> sample-only k-mers it holds (ascending local index)
  const int32_t* rk_s;
  const int32_t* rk_pos;           // first position of that mer in the read
  // mutable per-mer / per-read state (zero-initialised except m_alive)
  uint8_t* m_alive;                // akmers.mers membership (set by bind_region: homopolymers start dead, Q5)
  uint64_t* seed_a;                // two buffers of [count : 32 | local index : 32] per mer: the region's seed order is
  uint64_t* seed_b;                // sorted into one of them by bind_region (Q7)
  uint8_t* m_used;                 // buffer.used_mers
  uint32_t* m_checked;             // contig serial in whose checked_kmers the mer is
  uint32_t* m_taken;               // finalize serial (check_alt_reads' mer_set)
  uint32_t* m_first;               // [contig serial : 32 - BITS | CAP - 1 - first window : BITS] of the mer in the contig being emitted
  uint8_t* r_used;                 // fq_read.used
  uint8_t* r_deleted;              // key removed from fq_recs
  uint8_t* r_queued;               // 1: contig pending in buffer.contigs, 2: left it
  uint32_t* r_buf;                 // contig serial whose .buffer holds the read
  uint32_t* r_inreads;             // contig serial whose .reads holds the read
  int32_t* q_read;                 // buffer.contigs FIFO (per region slice of size U)
  int32_t* q_seed;
  int32_t* l_alt;                  // read_batch.alt / .delete, find_reads results (size U each)
  int32_t* l_del;
  int32_t* hit_u; int32_t* hit_pos; int32_t* hit2_u; int32_t* hit2_pos;
  uint64_t* sort_a; uint64_t* sort_b;  // size U each: sort buffers of find_reads
  int32_t* l_mused;                    // size S: list form of buffer.used_mers
  // per-warp scratch, slot = global warp index; sizes for AsmCap (AsmCapLong: the same formulas with its CAP)
  uint8_t* w_cseq;                 // ASM_BUF bytes
  int32_t* w_cnt;                  // 4 * ASM_BUF ints: io[2], ot[2]
  int32_t* w_K;                    // 4 * ASM_KCAP ints: s, x, meta, buffer coordinate of the window
  int32_t* w_NK;                   // 4 * ASM_KCAP ints: s, stream end, meta, buffer coordinate
  uint64_t* w_wcode;               // ASM_CAP
  int32_t* w_diff;                 // ASM_CAP + 1
  int2* w_edge;                    // 2 * ASM_CAP int2, or null if no read is longer than 256
  uint2* w_lastcol;                // ASM_LASTCOL uint2 per warp: last DP column of the sweep in flight (nw.cuh)
  uint8_t* w_tab;                  // NW_TAB_BYTES per warp: low bytes of the score table of the sweep in flight (nw.cuh)
  // work distribution
  int* work_counter;
  const int32_t* work_order;       // regions, most expensive first
  // output arena (bump allocated)
  unsigned long long* out_cursor;  // [0]=seq bytes [1]=count ints [2]=read ints [3]=kmer tuples [4]=contigs
  unsigned long long cap_seq, cap_cnt, cap_reads, cap_kmers, cap_ctg;
  uint8_t* o_seq; int32_t* o_locs;
  int32_t* o_io; int32_t* o_ot;
  int32_t* o_reads;
  uint64_t* o_kmer_mer; int32_t* o_kmer_pos; int32_t* o_kmer_meta;
  int64_t* o_desc;                 // per contig 10 x int64: region, ordinal, seq_off, seq_len, cnt_off, cnt_len,
                                   //                        reads_off, n_reads, kmers_off, n_kmers
  int32_t* region_status;          // per region: its status (ST_OK or the RR_* reason it stopped for)
  int32_t* region_ncontigs;
  unsigned long long* region_cells;  // per region: sum over its check_align calls of len(contig) * len(read)
  int32_t* region_report;          // per region: RR_FIELDS ints (common.cuh, bk_region_report), or null: no report
  unsigned long long* stats;       // [0] check_align calls, [1] DP cells, [2] find_reads, [3] seeds, [8..] phase cycles
  unsigned long long* prof_regions; // BK_PHASE_PROF: n_regions x 8 phase cycles (or null)
};

// ---- small warp helpers -----------------------------------------------------------------
BK_DEV unsigned lane_lt_mask() { return (1u << lane()) - 1u; }
BK_DEV int warp_min_i(int v) {
#ifndef BK_SIM
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
#endif
  return v;
}
BK_DEV int warp_max_i(int v) {
#ifndef BK_SIM
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
#endif
  return v;
}

// Sort n UNIQUE 64-bit keys (all > 0) in descending order with one warp; a and b are two buffers of n keys, the input
// is in a, the result is in the buffer returned.  Chunks of a warp are sorted in registers (bitonic over the lanes),
// then merged pass by pass: every element finds its place in the merged run by a binary search in the neighbouring
// run.  O(n log^2 n / 32) steps.
#ifdef BK_SIM
inline
#else
static __device__ __noinline__                           // (rarely executed, several call sites: keep one copy out of line)
#endif
uint64_t* warp_sort_desc(uint64_t* a, uint64_t* b, int n) {
#ifndef BK_SIM
  for (int base = 0; base < n; base += WARP) {
    const int i = base + lane();
    unsigned long long v = i < n ? (unsigned long long)a[i] : 0ull;
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, j);
        const bool desc = (lane() & k) == 0, lower = (lane() & j) == 0;
        v = (lower == desc) ? (v > o ? v : o) : (v < o ? v : o);
      }
    if (i < n) a[i] = v;
  }
#endif
  syncwarp();
  uint64_t* src = a; uint64_t* dst = b;
  for (int L = WARP; L < n; L <<= 1) {
    for (int i = lane(); i < n; i += WARP) {
      const int a0 = (i / (2 * L)) * 2 * L;
      const int a1 = (a0 + L) < n ? (a0 + L) : n, b1 = (a0 + 2 * L) < n ? (a0 + 2 * L) : n;
      const uint64_t key = src[i];
      const bool left = i < a1;
      int lo = left ? a1 : a0, hi = left ? b1 : a1;      // the other run (descending): count its elements > key
      const int o0 = lo;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (src[mid] > key) lo = mid + 1; else hi = mid;
      }
      dst[a0 + (left ? i - a0 : i - a1) + (lo - o0)] = key;
    }
    syncwarp();
    uint64_t* t = src; src = dst; dst = t;
  }
  return src;
}

// 2-bit code of the k-mer starting at seq[x]; false if it holds a non-ACGT byte
BK_DEV bool window_code(const uint8_t* seq, int x, int k, uint64_t& code) {
  uint64_t c = 0;
  bool ok = true;
  for (int t = 0; t < k; ++t) {
    const int b = base_code_strict(seq[x + t]);
    ok = ok && (b < 4);
    c = (c << 2) | (uint64_t)(b & 3);
  }
  code = c;
  return ok;
}

template <class T>
struct RegionCtxT {
  const AsmParams* P;
  int region, k;
  // mers
  int S; int64_t gm0;
  const uint64_t* mer; const uint32_t* cnt;
  const uint64_t* seed_keys; int seed_cursor;   // mers by (count, mer) descending; first position not yet consumed
  uint8_t* alive; uint8_t* mused; uint32_t* checked; uint32_t* taken; uint32_t* first;
  int32_t* s_hash; bool hash_on;   // shared-memory hash of the region's mer table (find_mer)
  // reads
  int U; int64_t gu0;
  const int32_t* u_rec; const uint32_t* u_mult; const uint8_t* u_io; const int32_t* u_len;
  uint8_t* r_used; uint8_t* r_deleted; uint8_t* r_queued; uint32_t* r_buf; uint32_t* r_inreads;
  int32_t* q_read; int32_t* q_seed; int q_head, q_tail;
  int32_t* l_alt; int32_t* l_del; int n_alt, n_del;
  int32_t* hit_u; int32_t* hit_pos; int32_t* hit2_u; int32_t* hit2_pos;
  uint64_t* sort_a; uint64_t* sort_b;   // find_reads: sort buffers for long posting lists (U keys each)
  int32_t* l_mused; int n_mused;        // mers in buffer.used_mers since the last remove_kmers
  // read stream of the current snapshot (st_u aliases hit_u) and speculation state
  int st_n;
  int rnd_base, rnd_cnt;          // stream range the last round covers
  unsigned seq_ver;               // bumped whenever the contig SEQUENCE changes
  unsigned rnd_ver;               // seq_ver when the last round started
  int spec_w;                     // speculation width of this launch (1..ASM_SPEC_W)
  SpecShared* sp;
  uint8_t* s_reads;               // ASM_SPEC_W staging buffers of ASM_CAP bytes; [0] doubles as s_read
  uint8_t* s_pred;                // ASM_SPEC_W - 1 predicted-contig buffers of ASM_CAP bytes
  int round_seed;                 // >= 0: every slot of the stream belongs to this mer (setup); -1: look up the entry
  int seed_anchor;                // setup: gap-buffer coordinate of the seed mer in the contig
  int cur_e;                      // grow: entry of the snapshot being committed
  int2* edge_all;                 // ASM_SPEC_W x (2 * ASM_CAP) int2 or null
  uint2* lastcol;                 // warp 0's last-column scratch
  uint8_t* tab;                   // warp 0's score-table scratch
  int32_t* nwl_diag;              // AsmCapLong: diagonals of the CTA's anti-diagonal sweep (nw_long.cuh), 9 * (CAP + 1) ints
  // contig under construction
  uint8_t* cseq; int c0, clen;
  int32_t* cnt_buf; int cur, k0, klen;
  int32_t* K; int nK;
  int32_t* NK; int nNK;
  uint64_t* wcode; int32_t* diff; int2* edge;
  uint32_t serial, fin_serial;
  bool ct_setup, ct_finalized;
  bool setup_queued;              // setup_contigs: the new contig went into buffer.contigs
  int ct_init_read;
  int status;                     // ST_OK, or the reason (RR_*) the region stopped for
  int n_out;
  unsigned long long n_align, n_cells;   // work counters of the region (flushed once at its end)
#if defined(BK_PHASE_PROF) && !defined(BK_SIM)
  long long ph_cycles[PH_COUNT_];
#endif
  // staging (shared memory on the device; global scratch in the long kernel)
  uint8_t* s_read; uint8_t* s_contig;

  BK_DEV int32_t* io_vec(int which) const { return cnt_buf + (size_t)which * T::BUF; }
  BK_DEV int32_t* ot_vec(int which) const { return cnt_buf + (size_t)(2 + which) * T::BUF; }
  BK_DEV int read_len_of(int u) const { return u_len[u]; }
  BK_DEV const uint8_t* read_ptr(int u) const { return P->rbases + P->roff[u_rec[u]]; }
};
using RegionCtx = RegionCtxT<AsmCap>;

// ---- per-region report (bk_region_report) ------------------------------------------------------------------------------
// A region that stops keeps the reason in c.status (ST_OK while it runs), which becomes its region_status.  Its counters
// are kept in s_report, a shared-memory row of the CTA at a fixed address, while it runs (lane 0 of the warp that runs the
// state machine writes it: one CTA owns a region), and copied to P.region_report when it ends, with its check_align
// calls.  Neither the counters nor the table's address live in registers, and the copy-in and copy-out are out of line:
// assemble_kernel<W> compiles to the same registers, stack and spills as without the report.  RR_REASON and RR_PASS are
// filled in on the host from region_status and the long kernel's queue; RR_FIRST_REASON is route_long_kernel's.
#if defined(BK_SIM)
static int s_report[RR_FIELDS];
#define BK_DEV_OUTLINE inline
#elif defined(BK_SIMT)
__shared__ int s_report[RR_FIELDS];
#define BK_DEV_OUTLINE inline
#else
__shared__ int s_report[RR_FIELDS];
#define BK_DEV_OUTLINE static __device__ __noinline__
#endif
BK_DEV void report_add(int field, int v) {
  if (lane() == 0) s_report[field] += v;
}
BK_DEV_OUTLINE void report_begin() {                                    // (bind_region syncs the warp after it)
  for (int f = lane(); f < RR_FIELDS; f += WARP) s_report[f] = 0;
}
// table is null in the single-region harnesses of tests/sim
BK_DEV_OUTLINE void report_end(int32_t* table, int region, unsigned long long n_align) {
  syncwarp();                                                            // lane 0's counters are visible to the warp
  for (int f = lane(); f < RR_FIELDS; f += WARP)
    if (table && f >= RR_SEEDS) table[(size_t)region * RR_FIELDS + f] = f == RR_CHECK_ALIGN ? (int32_t)n_align : s_report[f];
}

// lookup of a code in the region's ascending mer table; -1 if absent.  Regions with up
// to MER_HASH_MAX mers use an open-addressed table in shared memory (entry =
// [tag:15 | index:16]); larger ones fall back to a binary search.
constexpr int MER_HASH_SIZE = 2048;
constexpr int MER_HASH_MAX = 1400;
BK_DEV unsigned mer_hash(uint64_t code) { return (unsigned)((code * 0x9E3779B97F4A7C15ull) >> 53); }        // 11 bits
BK_DEV int mer_tag(uint64_t code) { return (int)((code * 0xC2B2AE3D27D4EB4Full) >> 49); }                 // 15 bits

template <class T>
BK_DEV void build_mer_hash(RegionCtxT<T>& c) {
  c.hash_on = c.S > 0 && c.S <= MER_HASH_MAX;
  if (!c.hash_on) return;
  syncwarp();
  for (int i = lane(); i < MER_HASH_SIZE; i += WARP) c.s_hash[i] = -1;
  syncwarp();
  for (int s = lane(); s < c.S; s += WARP) {
    const uint64_t code = c.mer[s];
    const int entry = (mer_tag(code) << 16) | s;
    unsigned slot = mer_hash(code);
    while (atomic_cas(&c.s_hash[slot], -1, entry) != -1) slot = (slot + 1) & (MER_HASH_SIZE - 1);
  }
  syncwarp();
}

template <class T>
BK_DEV int find_mer(const RegionCtxT<T>& c, uint64_t code) {
  if (c.hash_on) {
    const int tag = mer_tag(code);
    unsigned slot = mer_hash(code);
    for (;;) {
      const int e = c.s_hash[slot];
      if (e < 0) return -1;
      if ((e >> 16) == tag) {
        const int idx = e & 0xffff;
        if (c.mer[idx] == code) return idx;
      }
      slot = (slot + 1) & (MER_HASH_SIZE - 1);
    }
  }
  int lo = 0, hi = c.S;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const uint64_t v = c.mer[mid];
    if (v < code) lo = mid + 1; else hi = mid;
  }
  return (lo < c.S && c.mer[lo] == code) ? lo : -1;
}

template <class T>
BK_DEV int stage_read(RegionCtxT<T>& c, int u) {
  const int n = c.read_len_of(u);
  const uint8_t* src = c.read_ptr(u);
  syncwarp();
  for (int x = lane(); x < n; x += WARP) c.s_read[x] = src[x];
  syncwarp();
  return n;
}
template <class T>
BK_DEV void sync_contig_to_smem(RegionCtxT<T>& c) {
  syncwarp();
  for (int x = lane(); x < c.clen; x += WARP) c.s_contig[x] = c.cseq[c.c0 + x];
  syncwarp();
}

// ---- get_read_kmers_ordered (:126-143; Q8 skips the last window, Q26 floor) ----
// windows of seq[base .. base+nlen) that are live sample-only mers, appended to
// the contig's k-mer tuple list in the requested order
// pass A of every "which windows are live sample-only mers" question: lane l owns a
// contiguous run of windows and rolls the 2-bit code along it (k loads for the first
// window, one per further window); win[x] = local mer index or -1
template <class T>
BK_DEV void lookup_windows(RegionCtxT<T>& c, const uint8_t* seq, int nwin, int32_t* win) {
  const int k = c.k;
  const int per = (nwin + WARP - 1) / WARP;
  const int x0 = lane() * per;
  const int x1 = (x0 + per) < nwin ? (x0 + per) : nwin;
  const uint64_t mask = (k == 32) ? ~0ull : ((1ull << (2 * k)) - 1ull);
  uint64_t code = 0;
  int bad = 0;                                  // windows (counting from x) still poisoned by a non-ACGT byte
  for (int x = x0; x < x1; ++x) {
    if (x == x0) {
      for (int t = 0; t < k; ++t) {
        const int bc = base_code_strict(seq[x + t]);
        code = (code << 2) | (uint64_t)(bc & 3);
        if (bc >= 4) bad = t + 1;
      }
    } else {
      const int bc = base_code_strict(seq[x + k - 1]);
      code = ((code << 2) | (uint64_t)(bc & 3)) & mask;
      bad = bc >= 4 ? k : (bad > 0 ? bad - 1 : 0);
    }
    int sidx = -1;
    if (bad == 0) sidx = find_mer(c, code);
    win[x] = sidx;
  }
  syncwarp();
}

template <class T>
BK_DEV void append_kmers(RegionCtxT<T>& c, const uint8_t* seq, int base, int nlen, int order) {
  const int k = c.k;
  const int nwin = nlen - k;              // range(0, len - l)
  if (nwin <= 0) return;
  BK_PH_BEGIN
  const int m = nlen / 2;
  const unsigned lt = lane_lt_mask();
  constexpr int KCAP = T::KCAP;
  int32_t* Ks = c.K; int32_t* Kx = c.K + KCAP; int32_t* Km = c.K + 2 * KCAP; int32_t* Kb = c.K + 3 * KCAP;
  int32_t* win = reinterpret_cast<int32_t*>(c.wcode);
  lookup_windows(c, seq + base, nwin, win);
  // pass 0: ascending x over [lo0, hi0) ; pass 1: descending x over [lo1, hi1)
  int lo0 = 0, hi0 = 0, lo1 = 0, hi1 = 0;
  if (order == ORDER_FOR) { lo0 = 0; hi0 = nwin; }
  else if (order == ORDER_REV) { lo1 = 0; hi1 = nwin; }
  else { lo0 = m < nwin ? m : nwin; hi0 = nwin; lo1 = 0; hi1 = m < nwin ? m : nwin; }   // sorted by (x<m, |x-m|) (:142)
  for (int pass = 0; pass < 2; ++pass) {
    const int lo = pass == 0 ? lo0 : lo1, hi = pass == 0 ? hi0 : hi1;
    for (int b = 0; b < hi - lo; b += WARP) {
      const int t = b + lane();
      const int x = pass == 0 ? lo + t : hi - 1 - t;
      int sidx = -1;
      if (t < hi - lo) {
        sidx = win[x];
        if (sidx >= 0 && !c.alive[sidx]) sidx = -1;
      }
      const unsigned mk = ballot(sidx >= 0);
      if (sidx >= 0) {
        const int dst = c.nK + popc(mk & lt);
        if (dst < KCAP) {
          Ks[dst] = sidx; Kx[dst] = x;
          const int lth = x < m ? 1 : 0, dist = x < m ? m - x : x - m;
          Km[dst] = lth | (order << 1) | (dist << 3);
          Kb[dst] = c.c0 + base + x;         // where the window sits in the gap buffer (stable under prepend/append)
        }
      }
      c.nK += popc(mk);
    }
  }
  if (c.nK > KCAP) { c.nK = KCAP; c.status = RR_KMER_LIST_FULL; }
  syncwarp();
  BK_PH_END(c, PH_KMERS)
}

template <class T>
BK_DEV void set_kmers(RegionCtxT<T>& c) {                               // :548-550
  c.ct_setup = true;
  c.nK = 0;
  append_kmers(c, c.s_contig, 0, c.clen, ORDER_MID);
}

// ---- assembly_counts (:160-221) ---------------------------------------------------
template <class T>
BK_DEV void set_counts(RegionCtxT<T>& c, int start, int end, int n, bool io) {      // :195-199
  int32_t* v = (io ? c.io_vec(c.cur) : c.ot_vec(c.cur)) + c.k0;
  if (end > c.klen) end = c.klen;                                   // python slice clipping
  for (int x = start + lane(); x < end; x += WARP) v[x] += n;
  syncwarp();
}
template <class T>
BK_DEV void extend_counts(RegionCtxT<T>& c, int l, int n, bool io, bool post) {     // :201-221
  int32_t* vi = c.io_vec(c.cur);
  int32_t* vo = c.ot_vec(c.cur);
  const int at = post ? c.k0 + c.klen : c.k0 - l;
  for (int x = lane(); x < l; x += WARP) { vi[at + x] = io ? n : 0; vo[at + x] = io ? 0 : n; }
  if (!post) c.k0 -= l;
  c.klen += l;
  syncwarp();
}
// contig replaced by read u; old counts re-added at [start, end) with python's
// zip-truncate / slice-assign semantics (:181-193, Q17).  s_read holds read u.
template <class T>
BK_DEV void set_superseq(RegionCtxT<T>& c, int u, const uint8_t* rd, int lr, int start, int end) {
  const int n = (int)c.u_mult[u];
  const bool io = c.u_io[u] != 0;
  const int bio = io ? n : 0, bot = io ? 0 : n;
  const int32_t* oi = c.io_vec(c.cur) + c.k0;
  const int32_t* oo = c.ot_vec(c.cur) + c.k0;
  int32_t* ni = c.io_vec(c.cur ^ 1) + T::CAP;
  int32_t* no = c.ot_vec(c.cur ^ 1) + T::CAP;
  const int span = end - start;
  const int mid = span < c.klen ? span : c.klen;
  const int tail = lr - end;
  const int nl = start + mid + tail;
  for (int x = lane(); x < nl; x += WARP) {
    int a = bio, b = bot;
    if (x >= start && x < start + mid) { a += oi[x - start]; b += oo[x - start]; }
    ni[x] = a; no[x] = b;
  }
  c.cur ^= 1; c.k0 = T::CAP; c.klen = nl;
  c.c0 = T::CAP; c.clen = lr;
  for (int x = lane(); x < lr; x += WARP) { const uint8_t ch = rd[x]; c.cseq[T::CAP + x] = ch; c.s_contig[x] = ch; }
  c.seq_ver += 1;
  syncwarp();
}

// first occurrence of mer `code` in seq[a, b) (str.find on the slice); -1 if none
#ifdef BK_SIM
inline
#else
static __device__ __noinline__                           // (rare paths, five call sites)
#endif
int find_in_slice(const uint8_t* seq, int a, int b, int k, uint64_t code) {
  const int nwin = b - a - k + 1;
  int best = 0x7fffffff;
  for (int t = 0; t < nwin; t += WARP) {
    const int x = t + lane();
    bool hit = false;
    if (x < nwin) {
      uint64_t w;
      hit = window_code(seq, a + x, k, w) && w == code;
    }
    const unsigned mk = ballot(hit);
    if (mk) { best = t + ffs(mk) - 1; break; }
  }
  return best == 0x7fffffff ? -1 : best;
}

// ---- contig.__init__ (:417-426) ---------------------------------------------------------
template <class T>
BK_DEV void contig_init(RegionCtxT<T>& c, int seed_s, int u) {
  BK_PH_BEGIN
  c.serial += 1;
  if (c.serial >= (1u << (32 - T::BITS))) { c.status = RR_TOO_MANY_CONTIGS; return; }   // tag width of m_first
  const int lr = stage_read(c, u);
  c.c0 = T::CAP; c.clen = lr;
  c.cur = 0; c.k0 = T::CAP; c.klen = lr;
  const int n = (int)c.u_mult[u];
  const bool io = c.u_io[u] != 0;
  int32_t* vi = c.io_vec(0) + T::CAP;
  int32_t* vo = c.ot_vec(0) + T::CAP;
  for (int x = lane(); x < lr; x += WARP) {
    const uint8_t ch = c.s_read[x];
    c.cseq[T::CAP + x] = ch; c.s_contig[x] = ch;
    vi[x] = io ? n : 0; vo[x] = io ? 0 : n;
  }
  c.nK = 0; c.nNK = 0;
  c.ct_setup = false; c.ct_finalized = false; c.ct_init_read = u;
  c.n_alt = 0; c.n_del = 0;
  if (lane() == 0) { c.checked[seed_s] = c.serial; c.r_buf[u] = c.serial; }    // checked_kmers=[seed] (Q24), buffer={read}
  syncwarp();
  BK_PH_END(c, PH_INIT)
}

// (contig.check_align and its two overlap cases, :449-546, are apply_align below: decision first, then ONE site per action)

// ---- the two olc.nw calls of check_align (:451-452), one warp per read ------------------------------
// Executed by every warp of the CTA (warp w takes stream slot w of the round).
BK_DEV void spec_stage(const AsmParams& P, SpecShared* sp, uint8_t* s_reads, int w) {
  const int64_t gu0 = P.u_off[sp->region];
  const int rec = P.u_rec[gu0 + sp->u[w]];
  const int64_t a = P.roff[rec];
  const int lr = (int)(P.roff[rec + 1] - a);
  uint8_t* rd = s_reads + (size_t)w * P.read_cap;
  const uint8_t* src = P.rbases + a;
  for (int x = lane(); x < lr; x += WARP) rd[x] = src[x];
  if (lane() == 0) sp->lr[w] = lr;
  syncwarp();
}
#if defined(BK_SIM)
inline
#else
static __device__ __noinline__                           // one copy of the sweeps: the controller and the aligner warps share it
#endif
void spec_dp(SpecShared* sp, const uint8_t* s_reads, int read_cap, const uint8_t* s_contig, const uint8_t* s_pred, int w,
             int2* edge, uint2* lastcol, uint8_t* tab) {
  const uint8_t* rd = s_reads + (size_t)w * read_cap;
  const int lr = sp->lr[w];
  const int b = sp->abuf[w];
  const uint8_t* ct = b == 0 ? s_contig : s_pred + (size_t)(b - 1) * ASM_CAP;
  const int lc = sp->la[w];
  NwDual r;
  // columns = read, rows = contig: dev-frame A = nw(read, contig) = v2, B = nw(contig, read) = v1
  nw_dual_dispatch<true>(rd, lr, ct, lc, edge, edge ? edge + ASM_CAP : nullptr, lastcol, tab, r);
  if (lane() == 0) { sp->v1[w] = r.b; sp->v2[w] = r.a; }
  syncwarp();
}


// mer (local index) that stream slot `pos` belongs to, and where that mer sits in the
// contig's gap buffer (a hint for the predictor; may be stale after a replacement)
template <class T>
BK_DEV int slot_mer(const RegionCtxT<T>& c, int pos, int* anchor_buf) {
  if (c.round_seed >= 0) { *anchor_buf = c.seed_anchor; return c.round_seed; }
  const int32_t* Ns = c.NK; const int32_t* Nend = c.NK + T::KCAP; const int32_t* Nb = c.NK + 3 * T::KCAP;
  int e = c.cur_e;
  while (pos >= Nend[e]) ++e;
  *anchor_buf = Nb[e];
  return Ns[e];
}

// Predicted contig after read slot w-1 is committed against contig buffer (src, la):
// gapless overlap anchored at the shared k-mer.  Writes the prediction to dst (if it
// differs) and returns its length; *same is set when the prediction is "unchanged".
template <class T>
BK_DEV int predict_contig(const RegionCtxT<T>& c, const uint8_t* src, int la, const uint8_t* rd, int lr, int pos_r, int mer_s,
                          int xc_hint, uint8_t* dst, bool* same, int* shift) {
  *same = true;
  const int k = c.k;
  if (pos_r < 0 || pos_r + k > lr) return la;
  // anchor: the hinted position if the k-mer really is there, else the first occurrence
  int xc = xc_hint;
  bool ok = xc >= 0 && xc + k <= la;
  if (ok) {
    bool diff = false;
    for (int t = lane(); t < k; t += WARP) diff = diff || (src[xc + t] != rd[pos_r + t]);
    ok = ballot(diff) == 0u;
  }
  if (!ok) xc = find_in_slice(src, 0, la, k, c.mer[mer_s]);
  if (xc < 0) return la;
  const int oL = pos_r - xc, oR = (lr - pos_r) - (la - xc);
  const int r0 = oL > 0 ? oL : 0, r1 = lr - (oR > 0 ? oR : 0), c0 = oL < 0 ? -oL : 0;
  const int ov = r1 - r0;
  if (ov <= 0) return la;
  int mm = 0;
  for (int t = lane(); t < ov; t += WARP) mm += (rd[r0 + t] != src[c0 + t]) ? 1 : 0;
#ifndef BK_SIM
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mm += __shfl_xor_sync(0xffffffffu, mm, o);
#endif
  const int sc = ov - 3 * mm;
  const int mn = la < lr ? la : lr;
  if (200 * sc < 179 * ov || 4 * sc < mn) return la;            // predicted: no match
  if (oL <= 0 && oR <= 0) return la;                            // contained: only the counts change
  int nl;
  if (oL > 0 && oR > 0) {                                       // the read replaces the contig
    nl = lr;
    for (int x = lane(); x < lr; x += WARP) dst[x] = rd[x];
    *shift = 0x40000000;                                        // coordinates of the old contig are void
  } else if (oL > 0) {                                          // prepend read[0:oL]
    nl = la + oL;
    if (nl > T::MAX_LEN) return la;
    for (int x = lane(); x < nl; x += WARP) dst[x] = x < oL ? rd[x] : src[x - oL];
    *shift += oL;
  } else {                                                      // append read[lr-oR:]
    nl = la + oR;
    if (nl > T::MAX_LEN) return la;
    for (int x = lane(); x < nl; x += WARP) dst[x] = x < la ? src[x] : rd[lr - oR + (x - la)];
  }
  *same = false;
  syncwarp();
  return nl;
}

#ifndef BK_SIM
// The long kernel's pair (slot 0 of a width-1 round: staged read, current contig) through the anti-diagonal sweep of
// nw_long.cuh, both directions, by every thread of the CTA.  v1 = nw(contig, read): columns = contig.
__device__ __forceinline__ void long_pair_dp(SpecShared* sp, const uint8_t* rd, const uint8_t* ct, int32_t* diag) {
  const int lr = sp->lr[0], lc = sp->la[0];
  constexpr size_t stride = AsmCapLong::CAP + 1;
  NwlEnd e = nwl_sweep(ct, lc, rd, lr, diag, stride, nullptr);
  if (e.owner) sp->v1[0] = NwOut{lc, e.oj, e.i, e.oi, e.v};
  e = nwl_sweep(rd, lr, ct, lc, diag, stride, nullptr);
  if (e.owner) sp->v2[0] = NwOut{lr, e.oj, e.i, e.oi, e.v};
}

// DP of a long-kernel round: the warp DP of nw.cuh when both sequences are within its 4,095 bases (the staged read
// and contig buffers hold at least NW_MAX_LEN + 1 bytes, as nw.cuh reads the row sequence that far), else the CTA
// sweep; the other warps of the CTA wait for that command in assemble_long_kernel
template <class T>
BK_DEV void long_round_dp(RegionCtxT<T>& c) {
  SpecShared* sp = c.sp;
  if (sp->lr[0] <= NW_MAX_LEN && c.clen <= NW_MAX_LEN) {
    spec_dp(sp, c.s_reads, c.P->read_cap, c.s_contig, nullptr, 0, c.edge_all, c.lastcol, c.tab);
    return;
  }
  __syncthreads();                                   // command published (sp->n, lr[0], la[0])
  long_pair_dp(sp, c.s_reads, c.s_contig, c.nwl_diag);
  __syncthreads();                                   // results published
}
#endif

// one speculation round over stream slots [pos, pos + cnt)
template <class T>
BK_DEV void nw_round(RegionCtxT<T>& c, int pos, int cnt) {
  BK_PH_BEGIN
  SpecShared* sp = c.sp;
  syncwarp();
  if (lane() == 0) {
    sp->n = cnt; sp->region = c.region;
    for (int w = 0; w < cnt; ++w) sp->u[w] = c.hit_u[pos + w];
  }
  syncwarp();
  const bool multi = c.spec_w > 1;
  // 1. every warp stages its read
#ifdef BK_SIM
  for (int w = 0; w < cnt; ++w) spec_stage(*c.P, sp, c.s_reads, w);
#else
  {
    BK_PH_BEGIN
    if (multi) __syncthreads();
    spec_stage(*c.P, sp, c.s_reads, 0);
    if (multi) __syncthreads();
    BK_PH_END(c, PH_STAGE)
  }
#endif
  // 2. warp 0 predicts the contig each later slot will see
  if (lane() == 0) { atomic_add(&c.P->stats[4], 1ull); atomic_add(&c.P->stats[5], (unsigned long long)cnt); }
  {
    BK_PH_BEGIN
    int buf = 0, la = c.clen;                                    // buffer 0 = the current contig
    const uint8_t* src = c.s_contig;
    if (lane() == 0) { sp->abuf[0] = 0; sp->la[0] = la; }
    int shift = 0;                                               // bases the predictions have prepended so far
    for (int w = 1; w < cnt; ++w) {
      uint8_t* dst = c.s_pred + (size_t)(w - 1) * ASM_CAP;
      bool same;
      int anchor_buf;
      const int mer_s = slot_mer(c, pos + w - 1, &anchor_buf);
      const int hint = shift >= 0x40000000 ? -1 : anchor_buf - c.c0 + shift;
      const int nl = predict_contig(c, src, la, c.s_reads + (size_t)(w - 1) * c.P->read_cap, sp->lr[w - 1], c.hit_pos[pos + w - 1],
                                    mer_s, hint, dst, &same, &shift);
      if (!same) { buf = w; la = nl; src = dst; }
      if (lane() == 0) { sp->abuf[w] = buf; sp->la[w] = la; }
    }
    syncwarp();
    BK_PH_END(c, PH_PREDICT)
  }
  // 3. every warp aligns its read against its contig
#ifdef BK_SIM
  for (int w = 0; w < cnt; ++w) spec_dp(sp, c.s_reads, c.P->read_cap, c.s_contig, c.s_pred, w, nullptr, nullptr, nullptr);
#else
  {
    BK_PH_BEGIN
    if constexpr (T::LONG) {
      long_round_dp(c);
    } else {
      if (multi) __syncthreads();
      spec_dp(sp, c.s_reads, c.P->read_cap, c.s_contig, c.s_pred, 0, c.edge_all, c.lastcol, c.tab);
      if (multi) __syncthreads();
    }
    BK_PH_END(c, PH_DP)
  }
#endif
  c.rnd_base = pos; c.rnd_cnt = cnt;
  BK_PH_END(c, PH_NW)
}

// ---- contig.check_align (:449-504), decision part: v1/v2 come from the round -------------------------------
template <class T>
BK_DEV bool apply_align_impl(RegionCtxT<T>& c, int u, int seed_s, bool grow, const uint8_t* rd, int lr, const NwOut& v1, const NwOut& v2);
template <class T>
BK_DEV bool apply_align(RegionCtxT<T>& c, int u, int seed_s, bool grow, const uint8_t* rd, int lr, const NwOut& v1, const NwOut& v2) {
  BK_PH_BEGIN
  const bool r = apply_align_impl(c, u, seed_s, grow, rd, lr, v1, v2);
  BK_PH_END(c, PH_APPLY)
  return r;
}
// contig.check_align (:449-504) with contig_overlap_read (:506-528) and read_overlap_contig (:530-546).  The decision
// tree is evaluated first and yields one action; every action's body exists once (instruction footprint).
enum { ACT_SUPERSEQ = 1, ACT_COUNTS, ACT_APPEND, ACT_PREPEND };
template <class T>
BK_DEV bool apply_align_impl(RegionCtxT<T>& c, int u, int seed_s, bool grow, const uint8_t* rd, int lr, const NwOut& v1, const NwOut& v2) {
  const int lc = c.clen;
  c.n_align += 1ull;
  c.n_cells += (unsigned long long)lc * (unsigned long long)lr;
  const int s1 = v1.score, s2 = v2.score;
  const int mn = lc < lr ? lc : lr;
  // :459-464 in integers (Q27)
  const bool bad1 = (4 * s1 < mn) || (200 * s1 < 179 * (v1.prej - v1.j0));
  const bool bad2 = (4 * s2 < mn) || (200 * s2 < 179 * (v2.prej - v2.j0));
  if (bad1 && bad2) return false;
  if (s1 == s2 && v1.j0 == 0 && v1.i0 == 0 && lc == lr) return true;            // :466 (Q16)
  // contig_overlap_read(v1): the read replaces the contig if the alignment starts at the contig's first base (:508; prej ==
  // len always, Q15), else its overhang is appended.  read_overlap_contig(v2): counts only if the alignment starts at the
  // read's first base (:531), else the read's head is prepended.
  const int act_cr = v1.j0 == 0 ? ACT_SUPERSEQ : ACT_APPEND;
  const int act_rc = v2.j0 == 0 ? ACT_COUNTS : ACT_PREPEND;
  int act;
  if (s1 == s2) {
    if (lc < lr || v1.j0 == 0) act = ACT_SUPERSEQ;                   // :471
    else if (lr < lc || v2.j0 == 0) act = ACT_COUNTS;                // :480
    else {
      // :485-496 -- alignment strings minus '-' are the aligned spans themselves
      const uint64_t code = c.mer[seed_s];
      const int i11 = find_in_slice(c.s_contig, v1.j0, lc, c.k, code);
      const int i12 = find_in_slice(rd, v1.i0, v1.prei, c.k, code);
      const int i21 = find_in_slice(rd, v2.j0, lr, c.k, code);
      const int i22 = find_in_slice(c.s_contig, v2.i0, v2.prei, c.k, code);
      const int d1 = i11 > i12 ? i11 - i12 : i12 - i11;
      const int d2 = i21 > i22 ? i21 - i22 : i22 - i21;
      act = 0;
      if (i11 > -1 && i12 > -1) {
        if ((i21 == -1 && i22 == -1) || d2 > d1) act = act_cr;
      } else if (i21 > -1 && i22 > -1) {
        if ((i11 == -1 && i12 == -1) || d2 < d1) act = act_rc;
      }
      if (act == 0) return false;
    }
  } else {
    act = s1 > s2 ? act_cr : act_rc;
  }
  const int n = (int)c.u_mult[u];
  const bool io = c.u_io[u] != 0;
  // k-mers to add to the contig's list afterwards (grow only): window range and order
  int k_base = 0, k_len = 0, k_order = ORDER_MID;
  bool k_reset = false;
  if (act == ACT_SUPERSEQ) {
    set_superseq(c, u, rd, lr, v1.i0, v1.prei);
    k_reset = true; k_len = c.clen;                                  // set_kmers (:548-550)
  } else if (act == ACT_COUNTS) {
    set_counts(c, v2.i0, v2.prei, n, io);
    return true;
  } else if (act == ACT_APPEND) {
    const int plen = lr - v1.prei;                                    // post_seq = read[aln[4]:]
    if (lc + plen > T::MAX_LEN) { c.status = RR_CONTIG_TOO_LONG; return true; }
    for (int x = lane(); x < plen; x += WARP) {
      const uint8_t ch = rd[v1.prei + x];
      c.cseq[c.c0 + lc + x] = ch; c.s_contig[lc + x] = ch;
    }
    c.clen = lc + plen;
    if (plen > 0) c.seq_ver += 1;
    syncwarp();
    set_counts(c, v1.j0, lc, n, io);                                  // add_postseq :243-250
    extend_counts(c, plen, n, io, true);
    k_base = lc - (c.k - 1); k_len = (c.k - 1) + plen; k_order = ORDER_FOR;   // :521,525-527
  } else {
    const int plen = v2.j0;                                           // pre_seq = read[0:aln[3]]
    if (lc + plen > T::MAX_LEN) { c.status = RR_CONTIG_TOO_LONG; return true; }
    for (int x = lane(); x < plen; x += WARP) c.cseq[c.c0 - plen + x] = rd[x];
    c.c0 -= plen; c.clen = lc + plen;
    c.seq_ver += 1;
    sync_contig_to_smem(c);
    set_counts(c, v2.i0, v2.prei, n, io);                             // add_preseq :255-262 (old coordinates)
    extend_counts(c, plen, n, io, false);
    const int head = (c.k - 1) < lc ? (c.k - 1) : lc;
    k_base = 0; k_len = plen + head; k_order = ORDER_REV;             // :539,543-545
  }
  if (grow) {
    if (k_reset) { c.ct_setup = true; c.nK = 0; }
    append_kmers(c, c.s_contig, k_base, k_len, k_order);
  }
  return true;
}

// ---- contig.check_read (:552-566, Q30) for stream slot `pos` -----------------------------------------------
// Uses the slot's result from the last round if the contig it was aligned against
// is byte-identical to the contig now; otherwise runs a new round starting here.
template <class T>
BK_DEV bool round_slot_valid(const RegionCtxT<T>& c, int w) {
  const SpecShared* sp = c.sp;
  const int b = sp->abuf[w];
  if (sp->la[w] != c.clen) return false;
  if (b == 0) return c.seq_ver == c.rnd_ver;                          // aligned against the contig of the round start
  const uint8_t* pr = c.s_pred + (size_t)(b - 1) * ASM_CAP;
  bool diff = false;
  for (int x = lane(); x < c.clen; x += WARP) diff = diff || (pr[x] != c.s_contig[x]);
  return ballot(diff) == 0u;
}

template <class T>
BK_DEV bool check_read(RegionCtxT<T>& c, int seed_s, int pos, bool grow) {
  bool have = pos < c.rnd_base + c.rnd_cnt;
  if (have) {
    BK_PH_BEGIN
    have = round_slot_valid(c, pos - c.rnd_base);
    BK_PH_END(c, PH_VALID)
  }
  if (!have) {
    int cnt = c.st_n - pos;
    if (cnt > c.spec_w) cnt = c.spec_w;
    c.rnd_ver = c.seq_ver;
    nw_round(c, pos, cnt);
  }
  const int w = pos - c.rnd_base;
  const int u = c.hit_u[pos];
  const NwOut v1 = c.sp->v1[w], v2 = c.sp->v2[w];
  const bool match = apply_align(c, u, seed_s, grow, c.s_reads + (size_t)w * c.P->read_cap, c.sp->lr[w], v1, v2);
  if (match) {
    if (lane() == 0) { c.r_used[u] = 1; c.r_inreads[u] = c.serial; }  // committed by the finalize that follows
  } else if (c.cnt[seed_s] > 2 && !c.r_used[u]) {
    if (lane() == 0) c.l_alt[c.n_alt] = u;
    c.n_alt += 1;
  } else {
    if (lane() == 0) c.l_del[c.n_del] = u;
    c.n_del += 1;
  }
  syncwarp();
  return match;
}

// ---- buffer.add_contig (:337-340) ----------------------------------------------------------------
template <class T>
BK_DEV bool add_contig(RegionCtxT<T>& c, int u, int seed_s) {
  const bool used = c.r_used[u];            // (a queued read is always used, so `id in contigs` is implied)
  syncwarp();                               // every lane has read the flag before lane 0 sets it
  if (used) return false;
  if (lane() == 0) {
    c.q_read[c.q_tail] = u; c.q_seed[c.q_tail] = seed_s;
    c.r_used[u] = 1; c.r_queued[u] = 1;
  }
  c.q_tail += 1;
  syncwarp();
  return true;
}

// ---- contig.check_alt_reads (:568-582, Q12, Q13) + finalize (:584-599) + rb.clean (:389-397, Q11) --
template <class T>
BK_DEV void finalize(RegionCtxT<T>& c, bool setup) {
  if (setup) set_kmers(c);
  BK_PH_BEGIN
  c.fin_serial += 1;
  const int k = c.k;
  for (int a = 0; a < c.n_alt; ++a) {
    const int u = c.l_alt[a];
    // the read's sample-only mers (ascending) with their first positions; get_read_kmers
    // skips the last window (Q8), i.e. keeps the mers whose first window starts before len-k
    const int64_t e0 = c.P->rk_off[c.gu0 + u], e1 = c.P->rk_off[c.gu0 + u + 1];
    const int32_t* ks = c.P->rk_s + e0;
    const int32_t* kp = c.P->rk_pos + e0;
    const int ne = (int)(e1 - e0);
    const int lim = c.u_len[u] - k;
    int best = -1;
    for (int t = 0; t < ne && best < 0; t += WARP) {
      const int i = t + lane();
      bool cand = false;
      if (i < ne && kp[i] < lim) {
        const int s = ks[i];
        cand = c.alive[s] && !c.mused[s] && c.taken[s] != c.fin_serial && c.cnt[s] > 1;
      }
      const unsigned mk = ballot(cand);
      if (mk) best = shfl(i < ne ? ks[i] : 0, ffs(mk) - 1);        // smallest candidate mer (order policy Q13)
    }
    if (best >= 0) {
      // new contig seeded there; the WHOLE candidate set joins mer_set (:580)
      for (int i = lane(); i < ne; i += WARP) {
        if (kp[i] < lim) {
          const int s = ks[i];
          if (c.alive[s] && !c.mused[s]) c.taken[s] = c.fin_serial;
        }
      }
      syncwarp();
      add_contig(c, u, best);
    }
  }
  if (!c.ct_finalized) {
    if (lane() == 0) c.r_inreads[c.ct_init_read] = c.serial;         // batch_reads[0] is aligned=True
    c.ct_finalized = true;
  }
  for (int d = lane(); d < c.n_del; d += WARP) c.r_deleted[c.l_del[d]] = 1;   // del fq_recs[read.seq]
  c.n_alt = 0; c.n_del = 0;
  syncwarp();
  BK_PH_END(c, PH_FINALIZE)
}

// ---- find_reads / read_search (:102-122; Q9, Q10, Q28) -------------------------------------------
// Appends the matching reads to the stream at [at, at + n), sorted by (pos, -len)
// or (-pos, -len) with ties in read order.  With filter_buffer the reads already in
// contig.buffer are skipped and the appended ones join it right away: they are
// all going to be checked by this contig, in this order, whatever the outcomes
// (the k-mer snapshot loop of grow has no early exit), so adding them early is
// unobservable.
template <class T>
BK_DEV int find_reads(RegionCtxT<T>& c, int s, bool filter_buffer, bool rev, int at) {
  BK_PH_BEGIN
  const int64_t a = c.P->post_off[c.gm0 + s], b = c.P->post_off[c.gm0 + s + 1];
  const int32_t* pr = c.P->post_read + a;
  const int32_t* pp = c.P->post_pos + a;
  const int n0 = (int)(b - a);
  const unsigned lt = lane_lt_mask();
  using Key = typename T::Key;
  constexpr unsigned KEY_MAX = T::BITS == 16 ? 0xFFFFFFFFu : (1u << (2 * T::BITS)) - 1u;
  int n = 0;
  if (n0 <= WARP) {
    // the whole posting list fits one warp pass: filter, rank and place from registers
    const int i = lane();
    bool keep = false;
    int u = 0, pos = 0;
    Key key = 0;
    if (i < n0) {
      u = pr[i]; pos = pp[i];
      keep = !c.r_deleted[u] && !(filter_buffer && c.r_buf[u] == c.serial);
      // sort key: primary pos (or -pos), secondary -len; both < CAP
      key = ((Key)(rev ? (T::CAP - 1 - pos) : pos) << T::BITS) | (Key)(T::CAP - 1 - c.u_len[u]);
    }
    const unsigned mk = ballot(keep);
    n = popc(mk);
    int rank = 0;
#ifdef BK_SIM
    (void)lt;
#else
    for (unsigned rest = mk; rest; rest &= rest - 1) {
      const int j = __ffs((int)rest) - 1;
      const Key kj = __shfl_sync(0xffffffffu, key, j);
      rank += (kj < key || (kj == key && j < i)) ? 1 : 0;          // stable: ties keep read order (Q9)
    }
#endif
    if (keep) {
      c.hit_u[at + rank] = u;
      c.hit_pos[at + rank] = pos;
      if (filter_buffer) c.r_buf[u] = c.serial;
    }
  } else {
    // long posting list (deep coverage): compact the kept reads, then sort [key | index] with the warp merge sort.
    // Ascending (key, list order) == descending of the complemented pair; ties keep read order (Q9).
    for (int t = 0; t < n0; t += WARP) {
      const int i = t + lane();
      bool keep = false;
      int u = 0, pos = 0;
      if (i < n0) {
        u = pr[i]; pos = pp[i];
        keep = !c.r_deleted[u] && !(filter_buffer && c.r_buf[u] == c.serial);
      }
      const unsigned mk = ballot(keep);
      if (keep) {
        const int dst = n + popc(mk & lt);
        const unsigned key = ((unsigned)(rev ? (T::CAP - 1 - pos) : pos) << T::BITS) | (unsigned)(T::CAP - 1 - c.u_len[u]);
        c.hit2_u[dst] = u;
        c.sort_a[dst] = ((unsigned long long)(KEY_MAX - key) << 32) | (unsigned)(0x7FFFFFFF - dst);
        if (filter_buffer) c.r_buf[u] = c.serial;
      }
      n += popc(mk);
    }
    syncwarp();
    const uint64_t* sorted = warp_sort_desc(c.sort_a, c.sort_b, n);
    for (int r = lane(); r < n; r += WARP) {
      const uint64_t kk = sorted[r];
      const int i = 0x7FFFFFFF - (int)(kk & 0xFFFFFFFFu);
      const int hi = (int)((KEY_MAX - (unsigned)(kk >> 32)) >> T::BITS);
      c.hit_u[at + r] = c.hit2_u[i];
      c.hit_pos[at + r] = rev ? (T::CAP - 1 - hi) : hi;
    }
  }
  syncwarp();
  if (lane() == 0) atomic_add(&c.P->stats[2], 1ull);
  report_add(RR_FIND_READS, 1);
  BK_PH_END(c, PH_FIND)
  return n;
}

// buffer.add_used_mer (:334-335): used_mers is a dict; the mers added since the last remove_kmers are also kept in a
// list so that remove_kmers (:358-360) touches those instead of sweeping the whole table once per seed
template <class T>
BK_DEV void add_used_mer(RegionCtxT<T>& c, int s) {
  if (!c.mused[s]) {                                                 // (warp-uniform: every lane reads the same byte)
    syncwarp();
    if (lane() == 0) { c.mused[s] = 1; c.l_mused[c.n_mused] = s; }
    c.n_mused += 1;
  }
  syncwarp();
}

// ---- set_kmer_locs (:434-438, Q25) + emit the accepted contig -------------------------------------------
template <class T>
BK_DEV void emit_contig(RegionCtxT<T>& c) {
  BK_PH_BEGIN
  const AsmParams& P = *c.P;
  const int k = c.k, len = c.clen;
  const int32_t* Ks = c.K; const int32_t* Kx = c.K + T::KCAP; const int32_t* Km = c.K + 2 * T::KCAP;
  // first window of every sample-only mer in the final contig (str.find), via a tagged
  // per-mer table: [serial | CAP - 1 - x] under atomicMax keeps the smallest x of this contig
  const int nwin = len - k + 1;
  for (int x = lane(); x <= len; x += WARP) c.diff[x] = 0;
  {
    int32_t* win = reinterpret_cast<int32_t*>(c.wcode);
    lookup_windows(c, c.s_contig, nwin, win);
    for (int x = lane(); x < nwin; x += WARP) {
      const int s = win[x];
      if (s >= 0) atomic_max(&c.first[s], (c.serial << T::BITS) | (unsigned)(T::CAP - 1 - x));
    }
  }
  syncwarp();
  for (int e = lane(); e < c.nK; e += WARP) {
    const unsigned v = c.first[Ks[e]];
    if ((v >> T::BITS) == c.serial) {                                // find() == -1 touches nothing (Q25)
      const int p = T::CAP - 1 - (int)(v & (unsigned)(T::CAP - 1));
      atomic_add(&c.diff[p], 1);
      atomic_add(&c.diff[(p + k) < len ? (p + k) : len], -1);
    }
  }
  syncwarp();
  // reads of the contig, ascending unique-read index
  int n_reads = 0;
  const unsigned lt = lane_lt_mask();
  for (int t = 0; t < c.U; t += WARP) {
    const int u = t + lane();
    const bool in = (u < c.U) && (c.r_inreads[u] == c.serial);
    const unsigned mk = ballot(in);
    if (in) c.hit_u[n_reads + popc(mk & lt)] = u;
    n_reads += popc(mk);
  }
  syncwarp();
  // reserve output space
  unsigned long long o_seq = 0, o_cnt = 0, o_rd = 0, o_km = 0, o_ct = 0;
  if (lane() == 0) {
    o_seq = atomic_add(&P.out_cursor[0], (unsigned long long)len);
    o_cnt = atomic_add(&P.out_cursor[1], (unsigned long long)c.klen);
    o_rd = atomic_add(&P.out_cursor[2], (unsigned long long)n_reads);
    o_km = atomic_add(&P.out_cursor[3], (unsigned long long)c.nK);
    o_ct = atomic_add(&P.out_cursor[4], 1ull);
  }
  o_seq = shfl(o_seq, 0); o_cnt = shfl(o_cnt, 0); o_rd = shfl(o_rd, 0); o_km = shfl(o_km, 0); o_ct = shfl(o_ct, 0);
  if (o_seq + len > P.cap_seq || o_cnt + c.klen > P.cap_cnt || o_rd + n_reads > P.cap_reads || o_km + c.nK > P.cap_kmers ||
      o_ct + 1 > P.cap_ctg) {
    c.status = RR_OUTPUT_ARENA;
    return;
  }
  // kmer_locs = prefix sum of diff (sequential over chunks of a warp)
  int carry = 0;
  for (int t = 0; t < len; t += WARP) {
    const int x = t + lane();
    int v = x < len ? c.diff[x] : 0;
#ifndef BK_SIM
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int w = __shfl_up_sync(0xffffffffu, v, o);
      if (lane() >= o) v += w;
    }
#endif
    if (x < len) {
      P.o_locs[o_seq + x] = carry + v;
      P.o_seq[o_seq + x] = c.s_contig[x];
    }
    carry += shfl(v, WARP - 1);
  }
  const int32_t* vi = c.io_vec(c.cur) + c.k0;
  const int32_t* vo = c.ot_vec(c.cur) + c.k0;
  for (int x = lane(); x < c.klen; x += WARP) { P.o_io[o_cnt + x] = vi[x]; P.o_ot[o_cnt + x] = vo[x]; }
  for (int x = lane(); x < n_reads; x += WARP) P.o_reads[o_rd + x] = c.u_rec[c.hit_u[x]];
  for (int e = lane(); e < c.nK; e += WARP) {
    P.o_kmer_mer[o_km + e] = c.mer[Ks[e]];
    P.o_kmer_pos[o_km + e] = Kx[e];
    P.o_kmer_meta[o_km + e] = Km[e];
  }
  if (lane() == 0) {
    int64_t* d = P.o_desc + o_ct * 10;
    d[0] = c.region; d[1] = c.n_out; d[2] = (int64_t)o_seq; d[3] = len; d[4] = (int64_t)o_cnt; d[5] = c.klen;
    d[6] = (int64_t)o_rd; d[7] = n_reads; d[8] = (int64_t)o_km; d[9] = c.nK;
  }
  c.n_out += 1;
  syncwarp();
  BK_PH_END(c, PH_EMIT)
}

// ---- setup_contigs (:11-26, Q20) and contig.grow (:616-649) ------------------------------------------------------------
// Both walk a read stream with contig.check_read and close every k-mer's reads with contig.finalize; they are one function
// here so that the (large) check_read / finalize / find_reads code exists once in the kernel -- the controller's
// instruction footprint is what its speed depends on most.
//   GROW_SETUP       the stream is the reads of the seed k-mer (slot 0 is the contig's own read); then the contig is
//                    grown (it was queued: it is the FIFO head)
//   GROW_SETUP_ONLY  same stream, but the contig was NOT queued (its first read was already used, Q20): check_read and
//                    finalize still run against it, then it is dropped
//   GROW_ONLY        a contig popped from the FIFO
enum { GROW_ONLY = 0, GROW_SETUP = 1, GROW_SETUP_ONLY = 2 };
template <class T>
BK_DEV void grow(RegionCtxT<T>& c, int mode, int seed_s) {
  bool setup = mode != GROW_ONLY;
  if (!setup && !c.ct_setup) set_kmers(c);
  const unsigned lt = lane_lt_mask();
  constexpr int KCAP = T::KCAP;
  int32_t* Ks = c.K; int32_t* Km = c.K + 2 * KCAP; int32_t* Kb = c.K + 3 * KCAP;
  int32_t* Ns = c.NK; int32_t* Nend = c.NK + KCAP; int32_t* Nm = c.NK + 2 * KCAP; int32_t* Nb = c.NK + 3 * KCAP;
  while (c.status == ST_OK) {
    int nn = 1;
    if (!setup) {
      // refresh_kmers (:601): tuples whose mer is not in checked_kmers, order kept
      BK_PH_BEGIN
      nn = 0;
      for (int t = 0; t < c.nK; t += WARP) {
        const int e = t + lane();
        bool keep = false;
        int s = 0, meta = 0, xb = 0;
        if (e < c.nK) { s = Ks[e]; meta = Km[e]; xb = Kb[e]; keep = c.checked[s] != c.serial; }
        const unsigned mk = ballot(keep);
        if (keep) { const int dst = nn + popc(mk & lt); Ns[dst] = s; Nm[dst] = meta; Nb[dst] = xb; }
        nn += popc(mk);
      }
      c.nNK = nn;
      syncwarp();
      BK_PH_END(c, PH_REFRESH)
      if (nn == 0) break;
    }
    // The read stream: setup -- find_reads(seed) over every remaining read (:14); grow -- get_mer_reads (:604-614) for
    // every tuple of the snapshot, in order.  It does not depend on how the alignments turn out (see find_reads).
    int st = 0;
    for (int e = 0; e < nn; ++e) {
#if !defined(BK_SIM) && !defined(BK_SIMT)   // (PTX; a hint only, absent from the host builds of tests/sim)
      if (!setup && e + 1 < nn) {       // warm L1/L2 for the next tuple's posting list while this one is processed
        const int64_t na = c.P->post_off[c.gm0 + Ns[e + 1]];
        asm volatile("prefetch.global.L2 [%0];" ::"l"(c.P->post_read + na + lane()));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(c.P->post_pos + na + lane()));
      }
#endif
      const int meta = setup ? 0 : Nm[e];
      const int lth = meta & 1, order = (meta >> 1) & 3;
      const bool rev = setup ? false : ((order == ORDER_MID) ? (lth == 0) : (order == ORDER_FOR));
      st += find_reads(c, setup ? seed_s : Ns[e], !setup, rev, st);
      if (!setup && lane() == 0) Nend[e] = st;
    }
    c.st_n = st;
    c.rnd_base = 0; c.rnd_cnt = 0;
    syncwarp();
    int pos = 0;
    if (setup) {
      add_used_mer(c, seed_s);                                         // buff.add_used_mer (:15)
      if (st == 0) { c.setup_queued = false; return; }                 // no read holds the seed: nothing to set up
      c.round_seed = seed_s;
      c.seed_anchor = T::CAP + c.hit_pos[0];                           // contig_init puts the first read at CAP
      c.rnd_cnt = 1;                                                   // slot 0 is the contig's own read: nothing to align
      const int u0 = c.hit_u[0];
      contig_init(c, seed_s, u0);
      const bool fresh = !c.r_used[u0];                                // (every lane reads the flag before lane 0 sets it)
      syncwarp();
      c.setup_queued = fresh;
      if (fresh) {                                                     // buff.add_contig(read, ct) (Q20)
        if (lane() == 0) c.r_used[u0] = 1;
        syncwarp();
      }
      pos = 1;
    } else {
      c.round_seed = -1;
    }
    for (int e = 0; e < nn && c.status == ST_OK; ++e) {
      c.cur_e = e;
      const int s = setup ? seed_s : Ns[e];
      const int end = setup ? st : Nend[e];
      if (!setup) add_used_mer(c, s);                                  // buff.add_used_mer (:632)
      syncwarp();
      for (; pos < end && c.status == ST_OK; ++pos) {
        const int u = c.hit_u[pos];
        if (setup && lane() == 0) c.r_buf[u] = c.serial;               // self.buffer.add(read.id) (:22)
        if (check_read(c, s, pos, !setup)) {
          const bool queued = !setup && c.r_queued[u] == 1;            // buff.remove_contig(read.id) :639
          syncwarp();                                                  // (every lane has read the flag before lane 0 changes it)
          if (queued) {
            if (lane() == 0) c.r_queued[u] = 2;
            syncwarp();
          }
        }
      }
      if (c.status != ST_OK) break;
      finalize(c, setup);
      if (!setup && lane() == 0) c.checked[s] = c.serial;
      syncwarp();
    }
    if (setup) {
      setup = false;
      if (!c.setup_queued) return;                                     // (Q20) the contig is not grown
    }
  }
}

template <class T>
BK_DEV int total_reads(const RegionCtxT<T>& c) {                         // :178-179
  const int32_t* vi = c.io_vec(c.cur) + c.k0;
  const int32_t* vo = c.ot_vec(c.cur) + c.k0;
  int a = -0x7fffffff, b = -0x7fffffff;
  for (int x = lane(); x < c.klen; x += WARP) { a = vi[x] > a ? vi[x] : a; b = vo[x] > b ? vo[x] : b; }
  return warp_max_i(a) + warp_max_i(b);
}

// after grow: accept or drop (:53-59, Q21)
template <class T>
BK_DEV void finish_contig(RegionCtxT<T>& c, int rc_thresh, int read_len) {
  if (c.status != ST_OK) return;
  report_add(RR_GROWN, 1);
  if (total_reads(c) < rc_thresh) { report_add(RR_REJ_SUPPORT, 1); return; }
  if (c.clen <= read_len) { report_add(RR_REJ_LENGTH, 1); return; }
  emit_contig(c);
}

// ---- akmers.has_mers + mers.items()[0] (:43-45, :318-322; seed order Q7) ----------------------------------------
// The reference keeps the mers in an OrderedDict sorted by (count, mer) descending and takes the first remaining one:
// the first live entry of the region's seed order.  Mers only ever leave akmers, so a cursor over the order suffices;
// 32 entries are tested per step.  Returns -1 when no live mer with count > 1 is left.
template <class T>
BK_DEV int next_seed(RegionCtxT<T>& c) {
  while (c.seed_cursor < c.S) {
    const int i = c.seed_cursor + lane();
    bool live = false;
    uint64_t key = 0;
    if (i < c.S) { key = c.seed_keys[i]; live = c.alive[(int)(key & 0xffffffffu)] != 0; }
    const unsigned mk = ballot(live);
    if (mk) {
      const int first = ffs(mk) - 1;
      c.seed_cursor += first;
      const uint64_t k0 = shfl(key, first);
      return (unsigned)(k0 >> 32) > 1u ? (int)(k0 & 0xffffffffu) : -1;
    }
    c.seed_cursor += WARP;
  }
  return -1;
}

// ---- init_assembly (:30-63) for one region ------------------------------------------------------------------
template <class T>
BK_DEV void assemble_region(RegionCtxT<T>& c) {
  const AsmParams& P = *c.P;
  const int read_len = P.read_len[c.region];
  c.serial = 0; c.fin_serial = 0; c.status = ST_OK; c.n_out = 0; c.n_align = 0; c.n_cells = 0;
  c.q_head = 0; c.q_tail = 0; c.n_alt = 0; c.n_del = 0;
  if (c.S == 0) return;                                              // :33-34
  while (c.status == ST_OK) {
    int seed;
    {
      BK_PH_BEGIN
      seed = next_seed(c);                                           // has_mers (:318-322): max count must be > 1
      BK_PH_END(c, PH_SEED)
    }
    if (seed < 0) break;
    if (lane() == 0) atomic_add(&P.stats[3], 1ull);
    report_add(RR_SEEDS, 1);
    // setup_contigs (:11-26) for the seed, then `while len(buff.contigs) > 0` (:50): the set-up contig first if it was
    // queued (the queue was empty, so it is the FIFO head), then whatever check_alt_reads queued
    int mode = GROW_SETUP;
    for (;;) {
      if (mode == GROW_ONLY) {
        while (c.q_head < c.q_tail && c.r_queued[c.q_read[c.q_head]] != 1) ++c.q_head;
        if (c.q_head >= c.q_tail) break;
        const int u = c.q_read[c.q_head], s = c.q_seed[c.q_head];
        ++c.q_head;
        syncwarp();                                                  // every lane is past its scan of the queue flags
        if (lane() == 0) c.r_queued[u] = 2;
        syncwarp();
        contig_init(c, s, u);
      }
      grow(c, mode, seed);
      if (c.status != ST_OK) break;
      if (mode == GROW_ONLY || c.setup_queued) finish_contig(c, P.rc_thresh, read_len);
      mode = GROW_ONLY;
    }
    // buff.remove_kmers (:358-360); remove_reads is a no-op (Q10)
    {
      BK_PH_BEGIN
      for (int i = lane(); i < c.n_mused; i += WARP) {                // the mers add_used_mer recorded since the last sweep
        const int s = c.l_mused[i];
        c.alive[s] = 0; c.mused[s] = 0;
      }
      c.n_mused = 0;
      syncwarp();
      BK_PH_END(c, PH_SEED)
    }
  }
}

// ---- kmers.get_all_kmer_values (:280-285, Q7): the region's mers by (count, mer) descending -----------------------
// Keys [count | local index] are unique, mers ascend with the index: one warp_sort_desc per region instead of a scan
// per seed.
template <class T>
BK_DEV void build_seed_order(RegionCtxT<T>& c, uint64_t* a, uint64_t* b) {
  for (int i = lane(); i < c.S; i += WARP) a[i] = ((unsigned long long)c.cnt[i] << 32) | (unsigned)i;
  syncwarp();
  c.seed_keys = warp_sort_desc(a, b, c.S);
  c.seed_cursor = 0;
}

template <class T>
BK_DEV void bind_region(RegionCtxT<T>& c, const AsmParams& P, int region, int64_t slot, uint8_t* s_reads, uint8_t* s_contig,
                        uint8_t* s_pred, int32_t* s_hash, SpecShared* sp, int spec_w) {
  c.s_hash = s_hash;
  c.spec_w = spec_w; c.s_pred = s_pred; c.round_seed = -1; c.cur_e = 0; c.rnd_ver = 0;
  c.P = &P; c.region = region; c.k = P.k;
  c.gm0 = P.so_off[region]; c.S = (int)(P.so_off[region + 1] - c.gm0);
  c.mer = P.so_mer + c.gm0; c.cnt = P.so_cnt + c.gm0;
  c.alive = P.m_alive + c.gm0; c.mused = P.m_used + c.gm0; c.checked = P.m_checked + c.gm0; c.taken = P.m_taken + c.gm0;
  c.first = P.m_first + c.gm0;
  c.gu0 = P.u_off[region]; c.U = (int)(P.u_off[region + 1] - c.gu0);
  c.u_rec = P.u_rec + c.gu0; c.u_mult = P.u_mult + c.gu0; c.u_io = P.u_io + c.gu0; c.u_len = P.u_len + c.gu0;
  c.r_used = P.r_used + c.gu0; c.r_deleted = P.r_deleted + c.gu0; c.r_queued = P.r_queued + c.gu0;
  c.r_buf = P.r_buf + c.gu0; c.r_inreads = P.r_inreads + c.gu0;
  c.q_read = P.q_read + c.gu0; c.q_seed = P.q_seed + c.gu0;
  c.l_alt = P.l_alt + c.gu0; c.l_del = P.l_del + c.gu0;
  c.hit_u = P.hit_u + c.gu0; c.hit_pos = P.hit_pos + c.gu0; c.hit2_u = P.hit2_u + c.gu0; c.hit2_pos = P.hit2_pos + c.gu0;
  c.sort_a = P.sort_a + c.gu0; c.sort_b = P.sort_b + c.gu0;
  c.l_mused = P.l_mused + c.gm0; c.n_mused = 0;
  c.cseq = P.w_cseq + slot * T::BUF;
  c.cnt_buf = P.w_cnt + slot * 4 * T::BUF;
  c.K = P.w_K + slot * 4 * T::KCAP;
  c.NK = P.w_NK + slot * 4 * T::KCAP;
  c.wcode = P.w_wcode + slot * T::CAP;
  c.diff = P.w_diff + slot * (T::CAP + 1);
  c.edge_all = P.w_edge ? P.w_edge + slot * spec_w * 2 * ASM_CAP : nullptr;
  c.lastcol = P.w_lastcol ? P.w_lastcol + (size_t)slot * spec_w * ASM_LASTCOL : nullptr;
  c.tab = P.w_tab ? P.w_tab + (size_t)slot * spec_w * NW_TAB_BYTES : nullptr;
  c.edge = c.edge_all;
  c.s_reads = s_reads; c.s_read = s_reads; c.s_contig = s_contig; c.sp = sp;
  report_begin();
  c.st_n = 0; c.rnd_base = 0; c.rnd_cnt = 0; c.seq_ver = 0;
  // kmers.add_kmer (:272-278, Q5): a homopolymer (len(set(mer)) == 1) never enters akmers
  for (int s = lane(); s < c.S; s += WARP) {
    const uint64_t m = c.mer[s];
    bool homo = true;
    for (int t = 1; t < c.k; ++t) homo = homo && (((m >> (2 * t)) & 3ull) == (m & 3ull));
    c.alive[s] = homo ? 0 : 1;
  }
  syncwarp();
  build_seed_order(c, P.seed_a + c.gm0, P.seed_b + c.gm0);
  build_mer_hash(c);
}

#ifndef BK_SIM
// One CTA of W warps per region slot: warp 0 runs the state machine and is worker 0 of
// every speculation round; warps 1..W-1 only align.  W = 4 minimises the latency of a
// region (used when a batch runs alone on the device), W = 1 spends no work on
// speculation and packs more regions per SM (used when several batches are in flight).
// dynamic shared memory of one CTA: W read buffers (sized by the longest read of the batch), the contig, W-1 predicted contigs,
// the mer hash, the round mailbox (then padding, see above)
inline size_t assemble_smem_bytes(int W, int read_cap) {
  return (size_t)W * read_cap + ASM_CAP + (size_t)(W - 1) * ASM_CAP + MER_HASH_SIZE * sizeof(int32_t) +
         ((sizeof(SpecShared) + 15) & ~size_t(15));
}

// CTAS = resident CTAs per SM the register allocation is bounded for (0: the default of the width)
template <int W, int CTAS = 0>
__global__ void __launch_bounds__(32 * W, (CTAS > 0 ? CTAS : (W >= 8 ? 1 : (W == 4 ? ASM_W4_CTAS : (W == 2 ? 5 : ASM_W1_CTAS))))) assemble_kernel(AsmParams P) {
  BK_DYN_SMEM(uint8_t, smem_raw);
  uint8_t* s_reads = smem_raw;
  uint8_t* s_contig = s_reads + (size_t)W * P.read_cap;
  uint8_t* s_pred = s_contig + ASM_CAP;
  int32_t* s_hash = reinterpret_cast<int32_t*>(s_pred + (size_t)(W - 1) * ASM_CAP);
  SpecShared& sp = *reinterpret_cast<SpecShared*>(s_hash + MER_HASH_SIZE);
  const int64_t slot = blockIdx.x;
  // Roles rotate with the CTA index: the controller (role 0: state machine + stream slot 0) is hardware warp
  // blockIdx % W, so the controllers of the CTAs resident on an SM do not all sit on the same sub-partition.
  const int warp = ((int)(threadIdx.x >> 5) + W - (int)(blockIdx.x % W)) % W;
  if (W > 1 && warp > 0) {
    int2* edge = P.w_edge ? P.w_edge + (slot * W + warp) * 2 * ASM_CAP : nullptr;
    uint2* lastcol = P.w_lastcol + (size_t)(slot * W + warp) * ASM_LASTCOL;
    uint8_t* tab = P.w_tab ? P.w_tab + (size_t)(slot * W + warp) * NW_TAB_BYTES : nullptr;
    for (;;) {
      __syncthreads();                                 // command published
      const int n = sp.n;
      if (n < 0) return;
      if (warp < n) spec_stage(P, &sp, s_reads, warp);
      __syncthreads();                                 // reads staged; warp 0 predicts
      __syncthreads();                                 // predictions published
      if (warp < n) spec_dp(&sp, s_reads, P.read_cap, s_contig, s_pred, warp, edge, lastcol, tab);
      __syncthreads();                                 // results published
    }
  }
  RegionCtx c;
  for (;;) {
    int w = 0;
    if (lane() == 0) w = atomicAdd(P.work_counter, 1);
    w = shfl(w, 0);
    if (w >= P.n_regions) break;
    const int region = P.work_order[w];
#if defined(BK_PHASE_PROF)
    const long long t_reg0 = clock64();
#endif
    bind_region(c, P, region, slot, s_reads, s_contig, s_pred, s_hash, &sp, W);
#if defined(BK_PHASE_PROF)
    for (int i = 0; i < PH_COUNT_; ++i) c.ph_cycles[i] = 0;
    c.ph_cycles[PH_BIND] = clock64() - t_reg0;
    unsigned long long gt0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt0));
#endif
    assemble_region(c);
#if defined(BK_PHASE_PROF)
    c.ph_cycles[PH_TOTAL] = clock64() - t_reg0;
    if (lane() == 0) {
      for (int i = 0; i < PH_MAXREGION; ++i) atomicAdd(&P.stats[8 + i], (unsigned long long)c.ph_cycles[i]);
      for (int i = PH_MAXREGION + 1; i < PH_COUNT_; ++i) atomicAdd(&P.stats[8 + i], (unsigned long long)c.ph_cycles[i]);
      atomicMax(&P.stats[8 + PH_MAXREGION], (unsigned long long)c.ph_cycles[PH_TOTAL]);
      if (P.prof_regions) {
        for (int i = 0; i < 8; ++i) P.prof_regions[(size_t)region * 12 + i] = (unsigned long long)c.ph_cycles[i];
        unsigned long long gt1; unsigned smid;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt1));
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        P.prof_regions[(size_t)region * 12 + 8] = gt0; P.prof_regions[(size_t)region * 12 + 9] = gt1;
        P.prof_regions[(size_t)region * 12 + 10] = smid;
      }
    }
#endif
    if (lane() == 0) {
      P.region_status[region] = c.status; P.region_ncontigs[region] = c.n_out;
      P.region_cells[region] = c.n_cells;
      atomicAdd(&P.stats[0], c.n_align);
      atomicAdd(&P.stats[1], c.n_cells);
    }
    report_end(P.region_report, region, c.n_align);
    syncwarp();
  }
  if (W > 1) {
    if (lane() == 0) sp.n = -1;                        // dismiss the workers
    __syncthreads();
  }
}

// ---- assemble_long_kernel: the same state machine with AsmCapLong (reads and contigs up to 65,535 bases) ----------
// Per-CTA scratch in global memory (the contig and the staged read do not fit shared memory at this capacity)
struct AsmLongScratch {
  uint8_t* reads;                  // read_cap bytes per CTA (>= longest read + 2 and > NW_MAX_LEN)
  uint8_t* contig;                 // AsmCapLong::CAP bytes per CTA
  int32_t* diag;                   // 9 * (AsmCapLong::CAP + 1) ints per CTA: the sweep's rolling diagonals
  const int* n_queue;              // device: length of P.work_order, written by route_long_kernel (null: P.n_regions)
};

#endif

}  // namespace bk
