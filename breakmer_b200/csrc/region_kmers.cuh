// K-mer stage of the batched pipeline, one CTA per target region (SURVEY.md rows K1-K4, kernels G1-G4).
//
// The reference counts four inputs per region with jellyfish (utils.py:151-179), loads the dumps into dicts
// (utils.py:287-297) and keeps  (case & case_sc) - ref  with the case counts (sv_processor.py:621-631); config 3
// also subtracts the normal sample's k-mers (K4).  Every key of that result is a soft-clip k-mer, so the region's
// whole set algebra fits an open-addressed hash table of its distinct soft-clip k-mers (atomicCAS insertion):
//
//   1. soft-clip windows    insert                                  (the candidate set: at most one slot per window)
//   2. read windows         look up, hit -> count += 1              (case counts: every record, duplicates included, Q3)
//   3. reference windows,   look up, hit -> candidate dead          (forward strand and its reverse complement, Q2;
//      normal windows                                                or the handle's cached reference k-mers)
//   4. survivors with count > 0 -> sorted by mer (A<C<G<T order) -> (mer, count) at the region's staging offset
//
// The table lives in SHARED memory (a region of a panel has a few thousand soft-clip windows), so the stage reads
// every input base once from HBM (1 B/base, coalesced, staged through a shared-memory tile) and writes only the
// sample-only k-mers: its HBM traffic is the algorithmic minimum of SURVEY.md 8.5, where the sort-based version moved
// every window ~10 times.  A region with more soft-clip windows than the shared table holds (deep amplicons) uses a
// slice of a global-memory table instead -- same code, L2 atomics.
//
// Jellyfish 1.1.11 semantics as restated in oracle/kmers_py.py: forward strand only (utils.py:160 has no -C), a window
// holding a non-ACGT base or crossing a record boundary is dropped, lower case folded.
//
// The stage also says where each candidate went (bk_kmer_report, one row of KR_FIELDS per region), in the order of the
// reference's set operations: the insertions that claim a slot count the candidates; a k-mer with count 0 never occurs
// in the reads; one killed with count > 0 was removed by the reference, unless the normal pass killed it (the one thread
// whose atomicOr set the dead bit knows); the rest are the sample-only k-mers.  None of this changes what the table
// holds, so the sample-only output is the same as without the report.  With the "normal_kmers" option the normal pass
// also stages the k-mers it removed (with their case counts) in a second slice at the region's soft-clip offset, sorted
// like the sample-only ones.
#pragma once
#include "common.cuh"
#include "kmers.cuh"

namespace bk {

constexpr int RK_THREADS = 512;
constexpr int RK_PER_THREAD = 4;
constexpr int RK_TILE = RK_THREADS * RK_PER_THREAD;
constexpr int RK_SMEM_CAP_MAX = 16384;          // slots of the shared-memory table (12 B each)
constexpr uint32_t RK_DEAD = 0x80000000u;

// the k-mer stage's per-region report (RegionKmerParams::kmer_report): the BK_KR_* fields of include/breakmer_b200.h,
// distinct k-mers each; KR_SOFT_CLIP = KR_NOT_IN_READS + KR_IN_REFERENCE + KR_IN_NORMAL + KR_SAMPLE_ONLY
constexpr int KR_SOFT_CLIP = 0, KR_NOT_IN_READS = 1, KR_IN_REFERENCE = 2, KR_IN_NORMAL = 3, KR_SAMPLE_ONLY = 4, KR_FIELDS = 5;

struct RkSet {                       // one input set of the batch (device arrays)
  const uint8_t* bases;
  const int64_t* koff;               // record offsets without empty records (+ terminator)
  const int64_t* reg_base;           // n_regions + 1 : base range of each region
  const int64_t* reg_krec;           // n_regions + 1 : range of each region in koff
};

struct RegionKmerParams {
  int n_regions, k;
  RkSet sc, reads, ref, normal;      // bases == nullptr: the set is absent
  const uint64_t* ref_mers;          // optional reference k-mer cache (sorted per region), instead of `ref`
  const int64_t* ref_koff;
  int smem_cap;                      // slots of the shared table of this launch (power of two)
  const uint32_t* tab_cap;           // per region: table slots (power of two > its soft-clip windows)
  const int64_t* gtab_off;           // per region: offset of its slice of the global table, -1 = shared memory
  uint64_t* gkeys; uint32_t* gcnt;   // global table slices
  uint64_t* st_mer; uint32_t* st_cnt;   // staging: region r writes at [sc.reg_base[r], + n)
  uint32_t* seg_counts;              // per region: number of sample-only k-mers
  int32_t* kmer_report;              // per region: KR_FIELDS counts; null: not written (and a region without reads is
                                     // skipped as before)
  uint64_t* nm_mer; uint32_t* nm_cnt;   // the "normal_kmers" option: the k-mers the normal sample removed, staged like
  uint32_t* nm_counts;                  // st_mer / st_cnt, and their number per region; null: not written
};

struct RkTable {
  uint64_t* keys; uint32_t* cnt; uint32_t mask;
  bool glob;                         // slice of the global table: plain loads could be served from a stale L1 line
  __device__ __forceinline__ uint64_t key_at(uint32_t i) const { return glob ? __ldcg(keys + i) : keys[i]; }
  __device__ __forceinline__ uint32_t cnt_at(uint32_t i) const { return glob ? __ldcg(cnt + i) : cnt[i]; }
};

// -> true for the one insertion that claimed the key's slot (the key was not in the table yet)
__device__ __forceinline__ bool rk_insert(const RkTable& T, uint64_t key) {
  uint32_t slot = (uint32_t)cand_hash(key) & T.mask;
  for (;;) {
    const unsigned long long old = atomicCAS((unsigned long long*)&T.keys[slot], (unsigned long long)KEY_INVALID, (unsigned long long)key);
    if (old == (unsigned long long)KEY_INVALID) return true;
    if (old == (unsigned long long)key) return false;
    slot = (slot + 1) & T.mask;
  }
}
__device__ __forceinline__ int rk_find(const RkTable& T, uint64_t key) {
  uint32_t slot = (uint32_t)cand_hash(key) & T.mask;
  for (;;) {
    const uint64_t t = T.key_at(slot);
    if (t == key) return (int)slot;
    if (t == KEY_INVALID) return -1;
    slot = (slot + 1) & T.mask;
  }
}

// Every valid window of region `r` of `set`, forward code (and reverse complement if `rc`), handed to f(code).
// Executed by the whole block; `code` is a shared tile buffer of RK_TILE + 32 bytes, `s_rfirst` one shared int64.
template <typename F>
__device__ __forceinline__ void rk_for_each_window(const RkSet& set, int r, int k, bool rc, uint8_t* code, int64_t* s_rfirst, F f) {
  const int64_t b0 = set.reg_base[r], b1 = set.reg_base[r + 1];
  const int64_t kr0 = set.reg_krec[r], kr1 = set.reg_krec[r + 1];
  if (b1 <= b0 || kr1 <= kr0) return;
  const int tid = threadIdx.x;
  const uint64_t kmask = (1ull << (2 * k)) - 1ull;
  for (int64_t p0 = b0; p0 < b1; p0 += RK_TILE) {
    __syncthreads();
    if (tid == 0) {
      int64_t lo = kr0, hi = kr1;            // koff[lo] <= p0 < koff[hi]: last record starting at or before the tile
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (set.koff[mid] <= p0) lo = mid; else hi = mid;
      }
      *s_rfirst = lo;
    }
    for (int x = tid; x < RK_TILE + k - 1; x += RK_THREADS) {
      const int64_t p = p0 + x;
      code[x] = (p < b1) ? (uint8_t)base_code(set.bases[p]) : (uint8_t)4;
    }
    __syncthreads();
    const int64_t lim = p0 + RK_TILE + k - 1;
    for (int64_t q = *s_rfirst + 1 + tid; q < kr1; q += RK_THREADS) {
      const int64_t o = set.koff[q];
      if (o >= lim) break;
      code[o - p0] |= 8;                     // a record starts here: no window may span it
    }
    __syncthreads();
    const int xb = tid * RK_PER_THREAD;
    uint64_t fwd = 0, rcv = 0;
    int bad = 0;
#pragma unroll
    for (int q = 0; q < RK_PER_THREAD; ++q) {
      const int x = xb + q;
      if (p0 + x >= b1) break;
      // `bad` = how many consecutive windows, starting with the current one, are ruled out by what was seen so far: an
      // invalid base at relative position t rules out windows 0..t, a record start at t >= 1 windows 0..t-1
      if (q == 0) {
        for (int t = 0; t < k; ++t) {
          const unsigned c = code[x + t];
          fwd = (fwd << 2) | (c & 3u);
          rcv |= (uint64_t)(3u - (c & 3u)) << (2 * t);
          const int b = (c & 4u) ? t + 1 : ((t > 0 && (c & 8u)) ? t : 0);
          bad = b > bad ? b : bad;
        }
      } else {
        const unsigned c = code[x + k - 1];
        fwd = ((fwd << 2) | (c & 3u)) & kmask;
        rcv = (rcv >> 2) | ((uint64_t)(3u - (c & 3u)) << (2 * (k - 1)));
        bad = bad > 0 ? bad - 1 : 0;
        const int b = (c & 4u) ? k : (((c & 8u) && k > 1) ? k - 1 : 0);
        bad = b > bad ? b : bad;
      }
      if (bad == 0) {
        f(fwd);
        if (rc) f(rcv);
      }
    }
  }
  __syncthreads();
}

// block-wide bitonic sort of n (key, count) pairs by key, in place; n_pad = power of two >= n, slots [n, n_pad) must be
// addressable and are filled with the all-ones key
__device__ __forceinline__ void rk_sort_pairs(uint64_t* keys, uint32_t* cnt, int n, int n_pad) {
  for (int i = n + threadIdx.x; i < n_pad; i += blockDim.x) { keys[i] = KEY_INVALID; cnt[i] = 0; }
  __syncthreads();
  for (int size = 2; size <= n_pad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (n_pad >> 1); t += blockDim.x) {
        const int lo = (t / stride) * 2 * stride + (t % stride);
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a > b) == up) {
          keys[lo] = b; keys[hi] = a;
          const uint32_t ca = cnt[lo]; cnt[lo] = cnt[hi]; cnt[hi] = ca;
        }
      }
      __syncthreads();
    }
  }
}

// sort the n staged (mer, count) pairs at (m, c) by mer, in place: in shared memory, or for a deep region inside its
// global table slice.  Both fit: a region's staged pairs are distinct soft-clip k-mers, fewer than its table's slots,
// and a shared table has at most smem_cap slots.  The table must no longer be needed.
__device__ __forceinline__ void rk_sort_staged(uint64_t* m, uint32_t* c, int n, uint64_t* s_keys, uint32_t* s_cnt, int smem_cap,
                                               const RkTable& T, bool in_smem, uint32_t cap) {
  if (n <= 1) return;
  int n_pad = 2;
  while (n_pad < n) n_pad <<= 1;
  if (n_pad <= smem_cap) {                   // sort in shared memory (the table is no longer needed there)
    __threadfence_block();
    for (int i = threadIdx.x; i < n; i += RK_THREADS) { s_keys[i] = __ldcg(m + i); s_cnt[i] = __ldcg(c + i); }
    __syncthreads();
    rk_sort_pairs(s_keys, s_cnt, n, n_pad);
    for (int i = threadIdx.x; i < n; i += RK_THREADS) { m[i] = s_keys[i]; c[i] = s_cnt[i]; }
  } else if (!in_smem && (uint32_t)n_pad <= cap) {   // a deep region: sort inside its global table slice
    for (int i = threadIdx.x; i < n; i += RK_THREADS) { T.keys[i] = __ldcg(m + i); T.cnt[i] = __ldcg(c + i); }
    __syncthreads();
    rk_sort_pairs(T.keys, T.cnt, n, n_pad);
    for (int i = threadIdx.x; i < n; i += RK_THREADS) { m[i] = T.keys[i]; c[i] = T.cnt[i]; }
  } else {
    // cannot happen (see above)
  }
}

__global__ void __launch_bounds__(RK_THREADS) region_kmer_kernel(RegionKmerParams P) {
  BK_DYN_SMEM(uint8_t, rk_smem);
  uint64_t* s_keys = reinterpret_cast<uint64_t*>(rk_smem);
  uint32_t* s_cnt = reinterpret_cast<uint32_t*>(s_keys + P.smem_cap);
  uint8_t* s_code = reinterpret_cast<uint8_t*>(s_cnt + P.smem_cap);
  __shared__ int64_t s_rfirst;
  __shared__ int s_n, s_nn, s_dead, s_distinct;
  const int k = P.k;
  for (int r = blockIdx.x; r < P.n_regions; r += gridDim.x) {
    const int64_t sc0 = P.sc.bases ? P.sc.reg_base[r] : 0;
    const int64_t n_sc = P.sc.bases ? P.sc.reg_base[r + 1] - sc0 : 0;
    const bool has_reads = P.reads.bases && P.reads.reg_base[r + 1] != P.reads.reg_base[r];
    // no candidates / no case k-mers (with the report, a region without reads still counts its candidates)
    if (n_sc == 0 || (!has_reads && !P.kmer_report)) {
      if (threadIdx.x == 0) {
        P.seg_counts[r] = 0;
        if (P.nm_counts) P.nm_counts[r] = 0;
        if (P.kmer_report)
          for (int f = 0; f < KR_FIELDS; ++f) P.kmer_report[(size_t)r * KR_FIELDS + f] = 0;
      }
      continue;
    }
    RkTable T;
    const uint32_t cap = P.tab_cap[r];
    const int64_t goff = P.gtab_off[r];
    const bool in_smem = goff < 0;
    T.keys = in_smem ? s_keys : P.gkeys + goff;
    T.cnt = in_smem ? s_cnt : P.gcnt + goff;
    T.mask = cap - 1;
    T.glob = !in_smem;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < cap; i += RK_THREADS) { T.keys[i] = KEY_INVALID; T.cnt[i] = 0; }
    if (threadIdx.x == 0) { s_n = 0; s_nn = 0; s_dead = 0; s_distinct = 0; }
    __syncthreads();
    // 1. candidates: the distinct soft-clip k-mers (sv_processor.py:620)
    rk_for_each_window(P.sc, r, k, false, s_code, &s_rfirst, [&](uint64_t key) {
      if (rk_insert(T, key)) atomicAdd(&s_distinct, 1);
    });
    if (has_reads) {
      // 2. case counts over every read record (sv_processor.py:618; reported count is case[mer], :630-631)
      rk_for_each_window(P.reads, r, k, false, s_code, &s_rfirst, [&](uint64_t key) {
        const int s = rk_find(T, key);
        if (s >= 0) atomicAdd(&T.cnt[s], 1u);
      });
      // 3. minus the reference (forward + reverse complement FASTA, sv_processor.py:613-615,622) and the normal sample (K4)
      auto kill = [&](uint64_t key) {
        const int s = rk_find(T, key);
        if (s >= 0 && !(T.cnt_at(s) & RK_DEAD)) atomicOr(&T.cnt[s], RK_DEAD);
      };
      if (P.ref_mers) {
        for (int64_t i = P.ref_koff[r] + threadIdx.x; i < P.ref_koff[r + 1]; i += RK_THREADS) kill(P.ref_mers[i]);
        __syncthreads();
      } else if (P.ref.bases) {
        rk_for_each_window(P.ref, r, k, true, s_code, &s_rfirst, kill);
      }
      // the normal pass: the one thread whose atomicOr set the dead bit of a k-mer of the reads counts it (and stages it)
      if (P.normal.bases) rk_for_each_window(P.normal, r, k, false, s_code, &s_rfirst, [&](uint64_t key) {
        const int s = rk_find(T, key);
        if (s < 0 || (T.cnt_at(s) & RK_DEAD)) return;
        const uint32_t old = atomicOr(&T.cnt[s], RK_DEAD);
        if (old == 0 || (old & RK_DEAD)) return;
        const int dst = atomicAdd(&s_nn, 1);
        if (P.nm_mer) { P.nm_mer[sc0 + dst] = key; P.nm_cnt[sc0 + dst] = old; }
      });
    }
    // 4. survivors -> staging (unsorted), then sorted in place; the killed k-mers of the reads are counted for the report
    uint64_t* out_m = P.st_mer + sc0;
    uint32_t* out_c = P.st_cnt + sc0;
    int n_dead = 0;
    for (uint32_t i = threadIdx.x; i < cap; i += RK_THREADS) {
      const uint32_t c = T.cnt_at(i);
      if (c != 0 && !(c & RK_DEAD)) {
        const int dst = atomicAdd(&s_n, 1);
        out_m[dst] = T.key_at(i); out_c[dst] = c;
      } else if (c & ~RK_DEAD) {
        ++n_dead;                                                      // in the reads, removed by the reference or normal
      }
    }
    if (n_dead) atomicAdd(&s_dead, n_dead);
    __syncthreads();
    const int n = s_n;
    const int nn = s_nn;
    if (threadIdx.x == 0) {
      P.seg_counts[r] = (uint32_t)n;
      if (P.nm_counts) P.nm_counts[r] = (uint32_t)nn;
      if (P.kmer_report) {
        int32_t* row = P.kmer_report + (size_t)r * KR_FIELDS;
        row[KR_SOFT_CLIP] = s_distinct;
        row[KR_NOT_IN_READS] = s_distinct - s_dead - n;                // the candidates with count 0
        row[KR_IN_REFERENCE] = s_dead - nn;
        row[KR_IN_NORMAL] = nn;
        row[KR_SAMPLE_ONLY] = n;
      }
    }
    rk_sort_staged(out_m, out_c, n, s_keys, s_cnt, P.smem_cap, T, in_smem, cap);
    if (P.nm_mer && nn > 1) {
      __syncthreads();
      rk_sort_staged(P.nm_mer + sc0, P.nm_cnt + sc0, nn, s_keys, s_cnt, P.smem_cap, T, in_smem, cap);
    }
    __syncthreads();
  }
}

// staging -> dense (mer, count) arrays at so_off (one block per region)
__global__ void __launch_bounds__(256) region_compact_kernel(const uint64_t* __restrict__ st_mer, const uint32_t* __restrict__ st_cnt,
                                                              const int64_t* __restrict__ sc_reg_base, const int64_t* __restrict__ so_off,
                                                              int n_regions, uint64_t* __restrict__ so_mer, uint32_t* __restrict__ so_cnt) {
  for (int r = blockIdx.x; r < n_regions; r += gridDim.x) {
    const int64_t src = sc_reg_base[r], dst = so_off[r];
    const int n = (int)(so_off[r + 1] - dst);
    for (int i = threadIdx.x; i < n; i += blockDim.x) { so_mer[dst + i] = st_mer[src + i]; so_cnt[dst + i] = st_cnt[src + i]; }
  }
}

}  // namespace bk
