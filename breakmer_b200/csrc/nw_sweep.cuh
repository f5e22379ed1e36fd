// The anti-diagonal sweep of `olc.nw` in 32-bit scores by one CTA (the method is described in nw_long.cuh), shared by
// nw_long_kernel (bk_nw_batch's pairs above 4,095 bases) and assemble_long_kernel (assemble.cuh).
#pragma once
#include "common.cuh"

namespace bk {

constexpr int NWL_THREADS = 256;

// End cell of one direction's sweep.  Every thread of the CTA gets v (score) and i (row); `owner` is set in exactly one
// thread, and only that thread's oi / oj (where the traceback stops) are meaningful.
struct NwlEnd {
  int v, i, oi, oj;
  bool owner;
};

// nw(s1, s2) of olc.py:40-107 (columns = s1 of length m, rows = s2 of length n, m, n >= 1) by the whole CTA of
// NWL_THREADS threads: the anti-diagonal sweep with the stop position carried forward.  diag: 9 * stride ints (stride >=
// n + 1); pm: the (n+1)(m+1)-byte pointer table, or null when the alignment strings are not wanted.  Every thread of the
// block must call it (one __syncthreads per diagonal).
__device__ __forceinline__ NwlEnd nwl_sweep(const uint8_t* s1, int m, const uint8_t* s2, int n, int32_t* base, size_t stride,
                                            uint8_t* pm) {
  __shared__ int red_v[NWL_THREADS];
  __shared__ int red_i[NWL_THREADS];
  const int tid = threadIdx.x;
  const size_t width = (size_t)m + 1;                                // buffer b, field f (score, stop row, stop column) at (3b + f) * stride

  // end cell of olc.py:79-83 over the last column (row 0 scores 0); per thread in ascending rows with >=
  int best_v = tid == 0 ? 0 : -2147483647 - 1, best_i = 0, best_oi = 0, best_oj = 0;
  int cur = 0;                                                       // buffer of diagonal d; (cur+2)%3 = d-1, (cur+1)%3 = d-2
  for (int d = 2; d <= m + n; ++d) {
    const int32_t* s_1 = base + (size_t)(3 * ((cur + 2) % 3)) * stride;     // diagonal d-1
    const int32_t* i_1 = s_1 + stride;
    const int32_t* j_1 = i_1 + stride;
    const int32_t* s_2 = base + (size_t)(3 * ((cur + 1) % 3)) * stride;     // diagonal d-2
    const int32_t* i_2 = s_2 + stride;
    const int32_t* j_2 = i_2 + stride;
    int32_t* s_0 = base + (size_t)(3 * cur) * stride;                       // diagonal d
    int32_t* i_0 = s_0 + stride;
    int32_t* j_0 = i_0 + stride;
    const int ilo = d - m > 1 ? d - m : 1;
    const int ihi = d - 1 < n ? d - 1 : n;
    for (int i = ilo + tid; i <= ihi; i += NWL_THREADS) {
      const int j = d - i;
      const bool top = i == 1, lft = j == 1;                         // the neighbours in row 0 / column 0 score 0
      const int dg = ((top || lft) ? 0 : s_2[i - 1]) + (s1[j - 1] == s2[i - 1] ? 1 : -2);   // olc.py:18-20, 63
      const int up = (lft ? 0 : s_1[i]) - 2;                         // score[i][j-1]: consumes seq1 (olc.py:64)
      const int lf = (top ? 0 : s_1[i - 1]) - 2;                     // score[i-1][j]: consumes seq2 (olc.py:65)
      int best = lf > up ? lf : up;
      best = dg > best ? dg : best;
      int si, sj;
      uint8_t t;
      if (best == dg)      { t = 3; if (top || lft) { si = i - 1; sj = j - 1; } else { si = i_2[i - 1]; sj = j_2[i - 1]; } }
      else if (best == up) { t = 2; if (lft)        { si = i;     sj = 0;     } else { si = i_1[i];     sj = j_1[i];     } }
      else                 { t = 1; if (top)        { si = 0;     sj = j;     } else { si = i_1[i - 1]; sj = j_1[i - 1]; } }
      s_0[i] = best;
      i_0[i] = si;
      j_0[i] = sj;
      if (pm) pm[(size_t)i * width + j] = t;
      if (j == m && best >= best_v) { best_v = best; best_i = i; best_oi = si; best_oj = sj; }
    }
    __syncthreads();
    cur = (cur + 1) % 3;
  }
  // the largest row among the maxima wins (>= scan in ascending rows)
  red_v[tid] = best_v;
  red_i[tid] = best_i;
  __syncthreads();
  for (int s = NWL_THREADS / 2; s > 0; s >>= 1) {
    if (tid < s) {
      const int v = red_v[tid + s], i2 = red_i[tid + s];
      if (v > red_v[tid] || (v == red_v[tid] && i2 > red_i[tid])) { red_v[tid] = v; red_i[tid] = i2; }
    }
    __syncthreads();
  }
  NwlEnd e;
  e.v = red_v[0];
  e.i = red_i[0];
  __syncthreads();                                                   // red_* are free again for the next sweep
  e.owner = best_v == e.v && best_i == e.i && (e.i > 0 || tid == 0);  // exactly one thread owns the end cell
  if (e.i == 0) { best_oi = 0; best_oj = m - 1; }                    // pointer[0][m] = 2 (olc.py:58-59): one step along row 0
  e.oi = best_oi;
  e.oj = best_oj;
  return e;
}

}  // namespace bk
