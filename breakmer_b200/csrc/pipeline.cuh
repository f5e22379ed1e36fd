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

// Which regions the assembly of a call takes, and with which kernel
enum LongMode {
  LONG_OFF,     // reads up to NW_MAX_LEN bases, assemble_kernel only (the default)
  LONG_ROUTE,   // reads up to ASM_LONG_MAX_LEN bases: assemble_kernel, then assemble_long_kernel (the "long_regions" option)
  LONG_ALL,     // reads up to ASM_LONG_MAX_LEN bases, every region to assemble_long_kernel (bk_compare_kmers_long)
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
  // the long assembler's mode, fixed at upload.  assemble_kernel takes the first n_short regions of the work order; in
  // the long modes, assemble_long_kernel takes the others and those assemble_kernel stopped
  LongMode long_mode = LONG_OFF;
  bool keep_rejected = false;             // the "rejected_contigs" option, fixed at upload like long_mode
  int n_short = 0;                        // LONG_OFF: all; LONG_ROUTE: those without a read above NW_MAX_LEN; LONG_ALL: 0
  const uint8_t* d_routed = nullptr;      // device, per region: a read above NW_MAX_LEN (LONG_ROUTE; null when none)
  int max_short_read_len = 0;             // longest read of the other regions (sizes assemble_kernel's read buffers)
};

// assemble_long_kernel's grid, scratch, queue and work counter in the long modes (long_assembly_scratch, long_params)
struct LongAssembly {
  int grid = 0, read_cap = 0;
  uint8_t* w_cseq = nullptr; int32_t* w_cnt = nullptr; int32_t* w_K = nullptr; int32_t* w_NK = nullptr;
  uint64_t* w_wcode = nullptr; int32_t* w_diff = nullptr; int2* w_edge = nullptr; uint2* w_lastcol = nullptr;
  uint8_t* w_tab = nullptr;
  int32_t* queue = nullptr;
  int* counter = nullptr;
  AsmLongScratch L{};
};

// everything submit() leaves behind for wait()
struct PendingBatch {
  bool active = false;
  const Pipeline* p = nullptr;
  Pipeline local;                          // non-resident submits own their Pipeline
  AsmParams A;                             // assemble_kernel's; assemble_long_kernel's is long_params(A, LA)
  int spec_w = 4, ctas_per_sm = 3, grid = 1, dyn_smem = 0;
  // the long modes: after assemble_kernel (if n_short > 0), route_long_kernel, then assemble_long_kernel on the queue
  bool route = false;
  LongAssembly LA;
  int* n_queue = nullptr;
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
  // the per-region report of the batch's result (bk_region_report): readable while the device arena is the one the
  // result was made in (result_epoch == h->dev.resets())
  bool has_result = false;
  size_t result_epoch = 0;
  std::vector<uint8_t> report_skipped;     // Pipeline::region_skipped of the batch
  std::vector<int32_t> h_reason;           // the device's region_status: 0 or the RR_* reason
  std::vector<int32_t> long_queue;         // the regions assemble_long_kernel ran (the long modes)
  std::vector<int32_t> h_report;           // host copy, made on request
  // the rejected contigs of the result (bk_rejected_contigs; keep_rejected: the batch was uploaded with the option on):
  // per region offsets into them and their reasons, growth order; their payload is at n_contigs + j of the ctg_* tables
  bool keep_rejected = false;
  std::vector<int64_t> rej_reg_off;
  std::vector<int32_t> rej_reason;
};

}  // namespace bk

