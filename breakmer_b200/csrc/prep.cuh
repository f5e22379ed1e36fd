// Kernels that turn the raw batch into the tables the assembler consumes:
//
//   read grouping   `fq_recs[seq].append(read)` (utils.py:239-244, Q28): identical
//                   read sequences of a region form one unique read; order =
//                   first occurrence; multiplicity = group size.  Hash every
//                   record, sort by hash (radix_sort.cuh), resolve runs of equal
//                   hash by exact byte comparison.
//   work order      regions ordered by a static cost estimate (unique reads x sample-only mers), most expensive
//                   first, by one single-block counting sort on the device.  (Seed order -- kmers.get_all_kmer_values,
//                   sv_assembly.py:280-285, Q7 -- and the homopolymer filter, :277, Q5, are evaluated inside the
//                   assembler: assemble.cuh next_seed / bind_region.)
//   inverted index  k-mer -> [(unique read, first position)] in read order; what
//                   find_reads/read_search (sv_assembly.py:102-122) recompute with
//                   a regex scan over every read for every k-mer.
#pragma once
#include "common.cuh"

namespace bk {

// ---------------------------------------------------------------------------------
// read grouping
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}

// one warp per record; key = 64-bit hash of (region, length, bytes), value = record index
__global__ void __launch_bounds__(128) read_hash_kernel(const uint8_t* __restrict__ bases, const int64_t* __restrict__ off,
                                                         const int32_t* __restrict__ rec_seg, int64_t n_rec,
                                                         uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int l = threadIdx.x & 31;
  if (r >= n_rec) return;
  const int64_t a = off[r];
  const int n = (int)(off[r + 1] - a);
  uint64_t h = 0x9e3779b97f4a7c15ull * (uint64_t)(l + 1);
  for (int x = l; x < n; x += 32) h = mix64(h ^ ((uint64_t)bases[a + x] + ((uint64_t)x << 8)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const uint64_t other = __shfl_down_sync(0xffffffffu, h, o);
    h = mix64(h * 0x100000001b3ull + other);
  }
  if (l == 0) {
    h = mix64(h ^ ((uint64_t)(uint32_t)rec_seg[r] << 32) ^ (uint64_t)n);
    keys[r] = h;
    vals[r] = (uint32_t)r;
  }
}

// thread per sorted position: leader = smallest record index of the run with the
// same region, length and bytes (exact; a hash collision only lengthens the scan)
__global__ void __launch_bounds__(128) group_leader_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                            int64_t n_rec, const uint8_t* __restrict__ bases,
                                                            const int64_t* __restrict__ off, const int32_t* __restrict__ rec_seg,
                                                            int32_t* __restrict__ leader_of, uint32_t* __restrict__ mult_by_rec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rec) return;
  const uint64_t key = keys[i];
  const uint32_t rec = vals[i];
  const int64_t a = off[rec];
  const int n = (int)(off[rec + 1] - a);
  const int seg = rec_seg[rec];
  int64_t j = i;
  while (j > 0 && (uint32_t)keys[j - 1] == (uint32_t)key) --j;     // the sort only orders the low 32 hash bits
  uint32_t leader = rec;
  for (int64_t t = j; t < i; ++t) {                   // stable sort: record indices ascend within the run
    const uint32_t cand = vals[t];
    const int64_t b = off[cand];
    if (rec_seg[cand] != seg || (int)(off[cand + 1] - b) != n) continue;
    bool same = true;
    for (int x = 0; x < n && same; ++x) same = bases[a + x] == bases[b + x];
    if (same) { leader = cand; break; }
  }
  leader_of[rec] = (int32_t)leader;
  atomicAdd(&mult_by_rec[leader], 1u);
}

__global__ void __launch_bounds__(256) leader_flag_kernel(const int32_t* __restrict__ leader_of, int64_t n_rec,
                                                           uint32_t* __restrict__ flag) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_rec) flag[r] = (leader_of[r] == (int32_t)r) ? 1u : 0u;
}

// leaders -> unique read table; u_index = exclusive scan of the leader flags
__global__ void __launch_bounds__(256) unique_scatter_kernel(const int32_t* __restrict__ leader_of,
                                                              const uint32_t* __restrict__ u_index, int64_t n_rec,
                                                              const uint32_t* __restrict__ mult_by_rec,
                                                              const uint8_t* __restrict__ flags, const int64_t* __restrict__ off,
                                                              int32_t* __restrict__ u_rec, uint32_t* __restrict__ u_mult,
                                                              uint8_t* __restrict__ u_io, int32_t* __restrict__ u_len) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rec || leader_of[r] != (int32_t)r) return;
  const uint32_t u = u_index[r];
  u_rec[u] = (int32_t)r;
  u_len[u] = (int32_t)(off[r + 1] - off[r]);
  u_mult[u] = mult_by_rec[r];
  u_io[u] = flags ? (flags[r] & 1u) : 0u;
}

// u_off[region] = u_index[first record of the region]; u_off[n_regions] = total
__global__ void __launch_bounds__(256) region_uoff_kernel(const int64_t* __restrict__ read_reg_off, int n_regions,
                                                           const uint32_t* __restrict__ u_index, int64_t n_rec,
                                                           const uint32_t* __restrict__ total, int64_t* __restrict__ u_off) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_regions) return;
  if (r == n_regions) { u_off[r] = *total; return; }
  const int64_t first = read_reg_off[r];
  u_off[r] = first < n_rec ? (int64_t)u_index[first] : (int64_t)*total;
}

// ---------------------------------------------------------------------------------
// sample-only table post-processing
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) widen_scan_kernel(const uint32_t* __restrict__ excl, const uint32_t* __restrict__ total,
                                                          int n, int64_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = excl[i];
  if (i == n) out[i] = *total;
}

// Work order of the assembler: regions by descending cost class.  cost = unique reads x sample-only mers (the DP work of a
// region grows with both); class = floor(8 * log2(cost + 1)) quantises it to 1/8 octave, which is all the longest-first
// heuristic needs.  One block: histogram, scan, scatter (order inside a class is arbitrary; results never depend on it).
// routed (or null): regions with a read above 4,095 bases in the "long_regions" mode; they come after all others (a
// second set of classes), so that assemble_kernel, bounded to the others, never binds one.
constexpr int WO_CLASSES = 512;
__global__ void __launch_bounds__(1024) work_order_kernel(const int64_t* __restrict__ so_off, const int64_t* __restrict__ u_off,
                                                          int n_regions, const uint8_t* __restrict__ routed,
                                                          int32_t* __restrict__ order) {
  __shared__ unsigned hist[2 * WO_CLASSES];
  __shared__ unsigned start[2 * WO_CLASSES];
  const int n_cls = routed ? 2 * WO_CLASSES : WO_CLASSES;
  for (int c = threadIdx.x; c < n_cls; c += blockDim.x) hist[c] = 0;
  __syncthreads();
  auto cls = [&](int r) {
    const float cost = (float)(so_off[r + 1] - so_off[r]) * (float)(u_off[r + 1] - u_off[r]) + 1.0f;
    int c = (int)(8.0f * __log2f(cost));
    c = c < 0 ? 0 : (c > WO_CLASSES - 1 ? WO_CLASSES - 1 : c);
    return WO_CLASSES - 1 - c + (routed && routed[r] ? WO_CLASSES : 0);   // ascending class = descending cost
  };
  for (int r = threadIdx.x; r < n_regions; r += blockDim.x) atomicAdd(&hist[cls(r)], 1u);
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (int c = 0; c < n_cls; ++c) { start[c] = run; run += hist[c]; }
  }
  __syncthreads();
  for (int r = threadIdx.x; r < n_regions; r += blockDim.x) order[atomicAdd(&start[cls(r)], 1u)] = r;
}

// ---------------------------------------------------------------------------------
// inverted index
// ---------------------------------------------------------------------------------
constexpr int IDX_WARPS = 8;     // one read per warp; shared memory is sized by the longest read of the batch

__device__ __forceinline__ bool window_code_dev(const uint8_t* seq, int x, int k, uint64_t& code) {
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

// one warp per unique read: every window whose mer is a sample-only mer of the
// region and that is the FIRST occurrence of that mer in the read emits
//   key  = [ global mer index | local read index : u_bits ], value = position   (k-mer -> reads)
//   key2 = [ global read index | local mer index : s_bits ], value = position   (read -> k-mers)
__global__ void __launch_bounds__(32 * IDX_WARPS) index_emit_kernel(
    const uint8_t* __restrict__ rbases, const int64_t* __restrict__ roff, const int64_t* __restrict__ u_off,
    const int32_t* __restrict__ u_rec, int n_regions, const uint32_t* __restrict__ n_uniq_dev, const int64_t* __restrict__ so_off,
    const uint64_t* __restrict__ so_mer, int k, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
    uint64_t* __restrict__ keys2, uint32_t* __restrict__ vals2, int u_bits, int s_bits, int ws_stride,
    int32_t* __restrict__ ws_global, uint32_t* __restrict__ n_out, uint32_t cap) {
  extern __shared__ int32_t ws_all[];          // IDX_WARPS x ws_stride : local mer index of every window of the warp's read
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  int32_t* ws = ws_all + (size_t)w * ws_stride;
  const int64_t u = (int64_t)blockIdx.x * IDX_WARPS + w;
  if (u >= (int64_t)*n_uniq_dev) return;           // the grid covers the record count, an upper bound of the unique reads
  int lo = 0, hi = n_regions;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (u_off[mid] <= u) lo = mid; else hi = mid;
  }
  const int region = lo;
  const int64_t gm0 = so_off[region];
  const int S = (int)(so_off[region + 1] - gm0);
  const uint64_t* mer = so_mer + gm0;
  const int rec = u_rec[u];
  const uint8_t* seq = rbases + roff[rec];
  const int len = (int)(roff[rec + 1] - roff[rec]);
  if (ws_global) ws = ws_global + roff[rec];         // reads above the shared table's reach: one slot per base of the read
  const int nwin = len - k + 1;                        // find_reads sees the last window too (Q8)
  const uint64_t ulocal = (uint64_t)(u - u_off[region]);
  if (S == 0) return;
  for (int t = 0; t < nwin; t += 32) {
    const int x = t + l;
    int s = -1;
    if (x < nwin) {
      uint64_t code;
      if (window_code_dev(seq, x, k, code)) {
        int a = 0, b = S;
        while (a < b) {
          const int mid = (a + b) >> 1;
          if (mer[mid] < code) a = mid + 1; else b = mid;
        }
        if (a < S && mer[a] == code) s = a;
      }
      ws[x] = s;
    }
    __syncwarp();
    bool first = s >= 0;
    if (first)
      for (int y = 0; y < x; ++y)
        if (ws[y] == s) { first = false; break; }
    const unsigned mk = __ballot_sync(0xffffffffu, first);
    if (mk) {
      uint32_t base = 0;
      if (l == 0) base = atomicAdd(n_out, (uint32_t)__popc(mk));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (first) {
        const uint32_t dst = base + __popc(mk & ((1u << l) - 1u));
        if (dst < cap) {                           // cannot overflow: at most one entry per window, cap = read bases
          keys[dst] = ((uint64_t)(gm0 + s) << u_bits) | ulocal;
          keys2[dst] = ((uint64_t)u << s_bits) | (uint64_t)s;
          vals[dst] = (uint32_t)x;
          vals2[dst] = (uint32_t)x;
        }
      }
    }
  }
}

// thread per (group + 1): post_off[g] = lower bound of g << low_bits in the sorted keys
// (n_post and n_groups live on the device; the grid covers an upper bound of n_groups + 1)
__global__ void __launch_bounds__(256) post_off_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ n_post_dev,
                                                        const uint32_t* __restrict__ n_groups_dev, int low_bits,
                                                        int64_t* __restrict__ post_off) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_post = (int64_t)*n_post_dev;
  if (g > (int64_t)*n_groups_dev) return;
  const uint64_t target = (uint64_t)g << low_bits;
  int64_t a = 0, b = n_post;
  while (a < b) {
    const int64_t mid = (a + b) >> 1;
    if (keys[mid] < target) a = mid + 1; else b = mid;
  }
  post_off[g] = a;
}

__global__ void __launch_bounds__(256) post_split_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                          const uint32_t* __restrict__ n_post_dev, int low_bits,
                                                          int32_t* __restrict__ post_read, int32_t* __restrict__ post_pos) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)*n_post_dev) return;
  post_read[i] = (int32_t)(keys[i] & ((1ull << low_bits) - 1ull));
  post_pos[i] = (int32_t)vals[i];
}

}  // namespace bk
