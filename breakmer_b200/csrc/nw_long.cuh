// `olc.nw` for pairs with a sequence above NW_MAX_LEN (4095) bases -- olc.py:40-107 has no length limit, the packed-cell
// warp kernels of nw.cuh have (14-bit score / 12-bit origin fields).  Rare path of bk_nw_batch: one CTA per (pair,
// direction) sweeps the table by anti-diagonals in 32-bit scores.  Cell (i, j) (row i = base i of seq2, column j = base
// j of seq1) lies on diagonal d = i + j and needs (i-1, j-1) of diagonal d-2 and (i-1, j), (i, j-1) of diagonal d-1:
// three rolling diagonals indexed by row, O(m + n) memory, one __syncthreads per diagonal.
//
// What the reference's traceback (olc.py:90-105) would return is carried FORWARD with the score: every cell holds the
// (i, j) at which a walk started from it stops (the first position with i == 0 or j == 0), taken over from the
// predecessor the pointer priority diag(3) > up(2) > left(1) of olc.py:62-74 picks.  So the five integers of the tuple
// need no pointer table; only when the alignment STRINGS are asked for (direction A of bk_nw_batch with want_aln) is
// the (n+1)(m+1)-byte pointer table written and walked back by one thread as olc.py does.
#pragma once
#include "nw_sweep.cuh"

namespace bk {

struct NwLongParams {
  const uint8_t* seqs;
  const int64_t* seq_off;
  const int32_t* pair_a;
  const int32_t* pair_b;
  const int64_t* long_idx;    // n_long pair indices (the pairs nw_batch_kernel skips)
  int32_t* out;               // n_pairs * 10, as NwBatchParams::out
  int32_t* diag;              // per CTA 9 * diag_stride: 3 rolling diagonals x {score, stop row, stop column}
  int64_t diag_stride;        // >= longest sequence of the long pairs + 1
  int want_aln;
  uint8_t* ptr_scratch;       // want_aln: (n+1)(m+1) bytes per long pair (direction A only)
  const int64_t* ptr_off;     // n_long
  uint8_t* aln1;
  uint8_t* aln2;
  const int64_t* aln_off;     // n_pairs (the caller's)
  int32_t* aln_len;           // n_pairs
};

// grid = 2 * n_long: CTA 2q = nw(seq1, seq2) of long pair q (fields 0-4 of its output row), CTA 2q+1 = nw(seq2, seq1)
__global__ void __launch_bounds__(NWL_THREADS) nw_long_kernel(NwLongParams p) {
  const int tid = threadIdx.x;
  const int64_t q = blockIdx.x >> 1;
  const int dir = blockIdx.x & 1;
  const int64_t pi = p.long_idx[q];
  const int ia = dir ? p.pair_b[pi] : p.pair_a[pi];
  const int ib = dir ? p.pair_a[pi] : p.pair_b[pi];
  const uint8_t* s1 = p.seqs + p.seq_off[ia];                       // columns (seq1 of this direction)
  const uint8_t* s2 = p.seqs + p.seq_off[ib];                       // rows
  const int m = (int)(p.seq_off[ia + 1] - p.seq_off[ia]);
  const int n = (int)(p.seq_off[ib + 1] - p.seq_off[ib]);
  int32_t* base = p.diag + (size_t)blockIdx.x * 9 * p.diag_stride;
  const bool want_ptr = p.want_aln && dir == 0;
  uint8_t* pm = want_ptr ? p.ptr_scratch + p.ptr_off[q] : nullptr;
  const size_t width = (size_t)m + 1;
  const NwlEnd e = nwl_sweep(s1, m, s2, n, base, (size_t)p.diag_stride, pm);
  if (e.owner) {
    int32_t* o = p.out + pi * 10 + dir * 5;
    o[0] = m; o[1] = e.oj; o[2] = e.i; o[3] = e.oi; o[4] = e.v;
  }
  if (want_ptr && tid == 0) {                                        // olc.py:86-105; stored end-first, the host flips
    int i = e.i, j = m, len = 0;
    uint8_t* a1 = p.aln1 + p.aln_off[pi];
    uint8_t* a2 = p.aln2 + p.aln_off[pi];
    for (;;) {
      const int t = i == 0 ? 2 : pm[(size_t)i * width + j];
      if (t == 3)      { a1[len] = s1[j - 1]; a2[len] = s2[i - 1]; --i; --j; }
      else if (t == 2) { a1[len] = s1[j - 1]; a2[len] = '-'; --j; }
      else             { a1[len] = '-'; a2[len] = s2[i - 1]; --i; }
      ++len;
      if (i == 0 || j == 0) break;
    }
    p.aln_len[pi] = len;
  }
}

}  // namespace bk
