// assemble_long_kernel: the state machine of assemble.cuh with AsmCapLong, and its launcher.  Included into api.cu
// only: the assemble_kernel<W> units (asm_w*.cu) must not see it, as it shares their out-of-line helpers and would change
// how they compile.
#pragma once
#include "assemble.cuh"

namespace bk {

// mutable per-mer and per-read state of one region, cleared by the kernel itself (a region's result does not depend on
// what an earlier launch left in these arrays)
BK_DEV void clear_region_state(const AsmParams& P, int region) {
  const int64_t m0 = P.so_off[region], m1 = P.so_off[region + 1];
  for (int64_t s = m0 + lane(); s < m1; s += WARP) { P.m_used[s] = 0; P.m_checked[s] = 0; P.m_taken[s] = 0; P.m_first[s] = 0; }
  const int64_t u0 = P.u_off[region], u1 = P.u_off[region + 1];
  for (int64_t u = u0 + lane(); u < u1; u += WARP) {
    P.r_used[u] = 0; P.r_deleted[u] = 0; P.r_queued[u] = 0; P.r_buf[u] = 0; P.r_inreads[u] = 0;
  }
  syncwarp();
}

// One CTA of NWL_THREADS threads per region slot, regions from the queue route_long_kernel built (P.work_order, *L.n_queue
// long).  Warp 0 runs the state machine without speculation (width 1); all warps join the anti-diagonal sweep of a pair
// beyond the warp DP's 4,095 bases (long_round_dp).
__global__ void __launch_bounds__(NWL_THREADS, 1) assemble_long_kernel(AsmParams P, AsmLongScratch L) {
  __shared__ int32_t s_hash[MER_HASH_SIZE];
  __shared__ SpecShared sp;
  const int64_t slot = blockIdx.x;
  uint8_t* s_read = L.reads + slot * P.read_cap;
  uint8_t* s_contig = L.contig + slot * AsmCapLong::CAP;
  int32_t* diag = L.diag + slot * 9 * (AsmCapLong::CAP + 1);
  if (threadIdx.x >= WARP) {
    for (;;) {
      __syncthreads();                                 // command published
      if (sp.n < 0) return;
      long_pair_dp(&sp, s_read, s_contig, diag);
      __syncthreads();                                 // results published
    }
  }
  RegionCtxT<AsmCapLong> c;
  const int n_work = *L.n_queue;
  for (;;) {
    int w = 0;
    if (lane() == 0) w = atomicAdd(P.work_counter, 1);
    w = shfl(w, 0);
    if (w >= n_work) break;
    const int region = P.work_order[w];
    clear_region_state(P, region);
    bind_region(c, P, region, slot, s_read, s_contig, nullptr, s_hash, &sp, 1);
    c.nwl_diag = diag;
    assemble_region(c);
    if (lane() == 0) {
      P.region_status[region] = c.status; P.region_ncontigs[region] = c.n_out;
      P.region_cells[region] = c.n_cells;
      atomicAdd(&P.stats[0], c.n_align);
      atomicAdd(&P.stats[1], c.n_cells);
    }
    report_end(P.region_report, region, c.n_align);
    syncwarp();
  }
  if (lane() == 0) sp.n = -1;                          // dismiss the other warps
  __syncthreads();
}

// The long modes: after assemble_kernel, build assemble_long_kernel's queue on the device.  order[n_short, n_regions) are
// the regions routed at upload (a read above 4,095 bases, or every region with n_short = 0 for bk_compare_kmers_long;
// assemble_kernel never saw them), most expensive first; then, in work order, every region of order[0, n_short) that
// assemble_kernel stopped (status not ST_OK).  *ctg_snapshot = the contig cursor at this point: the descriptors below it
// are assemble_kernel's, and those of a rerouted region are dropped from the result.  The report's RR_FIRST_REASON of
// every queued region is set here, before assemble_long_kernel rebinds it: routed_reason for those routed at upload
// (the report starts zeroed, so 0 leaves it as is), the reason assemble_kernel stopped the others for (their status).  One block.
constexpr int ROUTE_THREADS = 256;
__global__ void __launch_bounds__(ROUTE_THREADS) route_long_kernel(const int32_t* __restrict__ order, int n_short, int n_regions,
                                                                   const int32_t* __restrict__ region_status,
                                                                   const unsigned long long* __restrict__ out_cursor,
                                                                   int32_t* __restrict__ queue, int* __restrict__ n_queue,
                                                                   unsigned long long* __restrict__ ctg_snapshot,
                                                                   int32_t* __restrict__ report, int routed_reason) {
  __shared__ int s_warp[ROUTE_THREADS / WARP];
  const int n_long = n_regions - n_short;
  const int t = threadIdx.x, wi = t / WARP;
  if (t == 0) *ctg_snapshot = out_cursor[4];
  for (int i = t; i < n_long; i += ROUTE_THREADS) {
    const int r = order[n_short + i];
    queue[i] = r;
    if (routed_reason) report[(size_t)r * RR_FIELDS + RR_FIRST_REASON] = routed_reason;
  }
  int base = n_long;
  for (int i0 = 0; i0 < n_short; i0 += ROUTE_THREADS) {       // ordered compaction, one block-wide chunk at a time
    const int i = i0 + t;
    const bool take = i < n_short && region_status[order[i]] != ST_OK;
    const unsigned mk = ballot(take);
    if (lane() == 0) s_warp[wi] = popc(mk);
    __syncthreads();
    int before = 0, total = 0;
    for (int v = 0; v < ROUTE_THREADS / WARP; ++v) {
      before += v < wi ? s_warp[v] : 0;
      total += s_warp[v];
    }
    if (take) {
      const int r = order[i];
      queue[base + before + popc(mk & ((1u << lane()) - 1u))] = r;
      report[(size_t)r * RR_FIELDS + RR_FIRST_REASON] = region_status[r];
    }
    base += total;
    __syncthreads();                                 // s_warp is rewritten by the next chunk
  }
  if (t == 0) *n_queue = base;
}

inline cudaError_t launch_assemble_long(const AsmParams& A, const AsmLongScratch& L, int grid, cudaStream_t st) {
  assemble_long_kernel<<<grid, NWL_THREADS, 0, st>>>(A, L);
  return cudaGetLastError();
}
}  // namespace bk
