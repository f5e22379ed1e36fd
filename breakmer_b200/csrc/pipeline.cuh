// Batched whole-path pipeline: state shared by submit and wait (the orchestration itself is pipeline_impl.cuh).
#pragma once

#include <numeric>
#include <vector>

#include "assemble.cuh"
#include "assemble_launch.cuh"
#include "host_util.cuh"
#include "prep.cuh"

namespace bk {

struct RecordSet {          // one of: reads, soft clips, normal reads (device copies)
  const uint8_t* bases = nullptr;
  int64_t n_bases = 0;
  const int64_t* off = nullptr;       // n_rec + 1 (all records, empties included)
  int64_t n_rec = 0;
  const int32_t* seg = nullptr;       // region of every record
  // compacted view without empty records (k-mer emit needs distinct starts)
  const int64_t* koff = nullptr;
  const int32_t* kseg = nullptr;
  int64_t kn_rec = 0;
  // host copies of the region boundaries (bases, compacted records): the k-mer stage may run in region chunks
  std::vector<int64_t> reg_base, reg_krec;
  const int64_t* d_reg_base = nullptr;   // device copies (region_kmers.cuh)
  const int64_t* d_reg_krec = nullptr;
  int64_t max_reg_bases = 0;          // largest region (bases)
};

struct Pipeline {
  int n_regions = 0, k = 0, rc_thresh = 0, have_mers = 0;
  bool use_ref_cache = false;
  RecordSet ref, reads, sc, normal;
  const uint8_t* read_flags = nullptr;
  const int64_t* read_reg_off = nullptr;  // device
  const int32_t* read_len = nullptr;      // device, per region
  const uint64_t* in_mers = nullptr;      // have_mers
  const uint32_t* in_counts = nullptr;
  const int64_t* in_mers_off = nullptr;   // device
  int64_t n_in_mers = 0;
  int max_read_len = 0;
  int64_t total_read_bytes = 0;
  int64_t h2d_bytes = 0;
  // upper bounds known from the input offsets (they size arrays and sort keys; results never depend on them)
  int64_t max_reg_records = 0;            // most read records in one region  >= its unique reads
  int64_t max_reg_mers = 0;               // most soft-clip bases (or given mers) in one region >= its sample-only mers
  // hash-table placement of the k-mer stage (region_kmers.cuh): per region table slots, and the offset of its slice of
  // the global table when it does not fit shared memory
  const uint32_t* d_tab_cap = nullptr;
  const int64_t* d_gtab_off = nullptr;
  int rk_smem_cap = 1024;
  int64_t rk_gtab_slots = 0;
  // regions left out of the device pass because a read exceeds the DP's length limit (their status is
  // BK_ERR_CAPACITY, every other region of the batch is processed): reads of those regions are not uploaded
  std::vector<uint8_t> region_skipped;    // empty = none
  std::vector<int64_t> rec_shift;         // per region: records dropped in earlier regions (result indices are shifted back)
  std::vector<char> filt_bases;           // the filtered host copies (alive until the upload copies are done)
  std::vector<int64_t> filt_off, filt_reg_off;
  std::vector<uint8_t> filt_flags;
  // the "long_regions" mode (bk_set_option), fixed at upload: regions with reads up to ASM_LONG_MAX_LEN bases are kept,
  // and those with a read above NW_MAX_LEN go to assemble_long_kernel only
  bool long_regions = false;
  int n_routed = 0;                       // regions with a read above NW_MAX_LEN
  const uint8_t* d_routed = nullptr;      // device, per region (null when n_routed == 0)
  int max_short_read_len = 0;             // longest read of the other regions (sizes assemble_kernel's read buffers)
};

// everything submit() leaves behind for wait()
struct PendingBatch {
  bool active = false;
  const Pipeline* p = nullptr;
  Pipeline local;                          // non-resident submits own their Pipeline
  AsmParams A;
  int spec_w = 4, ctas_per_sm = 3, grid = 1, dyn_smem = 0;
  bool long_path = false;                  // bk_compare_kmers_long: assemble_long_kernel with its scratch L
  AsmLongScratch L{};
  // the "long_regions" mode: assemble_kernel on the first n_short regions of the work order, route_long_kernel, then
  // assemble_long_kernel (grid long_grid) on the device queue with A_long = A plus the long scratch
  bool route = false;
  int n_short = 0, long_grid = 0;
  AsmParams A_long;                        // only its scratch fields (read_cap, w_*) are kept; the rest comes from A
  int32_t* queue = nullptr;
  int* n_queue = nullptr;
  int* long_counter = nullptr;
  unsigned long long* ctg_snapshot = nullptr;
  const int32_t* h_queue = nullptr;        // pinned copies
  const int* h_n_queue = nullptr;
  const unsigned long long* h_snapshot = nullptr;
  uint8_t* zero_lo = nullptr;
  size_t zero_bytes = 0;
  unsigned long long cap_seq = 0;
  int64_t n_keys = 0, n_sorted = 0;
  // device
  const uint64_t* so_mer = nullptr; const uint32_t* so_cnt = nullptr;
  const int64_t* so_off = nullptr; const int64_t* u_off = nullptr;
  const int32_t* u_rec = nullptr; const uint32_t* u_mult = nullptr;
  const uint32_t* d_counts = nullptr;      // [0] unique reads, [1] sample-only k-mers, [2] postings
  // pinned host
  const uint32_t* h_counts = nullptr;
  const unsigned long long* h_cursor = nullptr;
  const unsigned long long* h_stats = nullptr;
  int32_t* h_status = nullptr;
  unsigned long long* h_cells = nullptr;
  const int64_t* h_so_off = nullptr; const int64_t* h_u_off = nullptr;
};

}  // namespace bk

